"""Deterministic mode, host side (no GPU): the flag's precedence, seeded priors, the `seed`
plumbing of CellTraining and `python -m cellcomm_b200`, and which `ops` calls the engine makes
with the mode off (exactly the atomic-path calls) and on (every reduction carries the
workspace).  The kernels themselves are checked in test_deterministic_gpu.py."""
import numpy as np
import pytest
import torch

import ops_emulator
from cellcomm_b200 import engine as eng

REDUCTIONS = ("colsum", "bias_grad", "bn_stats", "bn_bwd_stats", "mse_fwd_bwd")


class RecordingOps:
    """ops_emulator plus a call log; the reductions also accept (and log) `ws=`, which the
    emulator's exact sums do not need."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        fn = getattr(ops_emulator, name)
        if not callable(fn) or name in ("alloc2d", "pad_ld", "launch_count"):
            return fn

        def call(*args, **kwargs):
            ws = kwargs.pop("ws", None) if name in REDUCTIONS else None
            self.calls.append((name, ws))
            return fn(*args, **kwargs)
        return call

    @staticmethod
    def reduce_ws_floats(rows, cols):
        return 8 + 2 * int(rows) * int(cols)


@pytest.fixture
def rec(monkeypatch):
    r = RecordingOps()
    monkeypatch.setattr(eng, "ops", r)
    return r


def _step(e, Z, G, B, seed):
    g = torch.Generator().manual_seed(seed)
    x = ops_emulator.alloc2d(B, G)
    x.copy_(torch.poisson(torch.rand(B, G, generator=g) * 3, generator=g))
    e.set_latents(torch.rand(B, Z, generator=g), torch.rand(B, Z, generator=g), B)
    return [float(v) for v in e.train_step(x)]


@pytest.mark.parametrize("fused", [True, False])
def test_engine_calls_with_the_mode_off_and_on(rec, fused):
    runs = {}
    for det in (False, True):
        rec.calls.clear()
        e = eng.BiGanEngine("cont", 3, 200, max_batch=16, device="cpu", seed=4, deterministic=det)
        e.set_fused_optimizer(fused)
        losses = _step(e, 3, 200, 16, 9)
        runs[det] = (list(rec.calls), losses, e)
    off, on = runs[False][0], runs[True][0]
    # off: no call carries a workspace (what the engine called before the mode existed)
    assert all(ws is None for _, ws in off)
    assert not hasattr(runs[False][2], "reduce_ws")
    # on: the same calls in the same order, and every reduction carries the one workspace
    assert [n for n, _ in off] == [n for n, _ in on]
    ws = runs[True][2].reduce_ws
    assert ws.dtype == torch.float32 and bool((ws == 0).all())
    red = [(n, w) for n, w in on if n in REDUCTIONS]
    assert {n for n, _ in red} >= {"bias_grad", "bn_stats", "bn_bwd_stats", "mse_fwd_bwd"}
    assert all(w is ws for _, w in red)
    assert all(w is None for n, w in on if n not in REDUCTIONS)
    assert runs[False][1] == runs[True][1]          # the emulator's sums ignore the workspace


def test_workspace_grows_with_the_batch(rec):
    e = eng.BiGanEngine("cont", 3, 200, max_batch=4, device="cpu", seed=1, deterministic=True)
    widest = max(max(n.g.widths) for n in e.nets.values())
    assert e.reduce_ws.numel() == rec.reduce_ws_floats(4, widest)
    e.reserve(32)
    assert e.reduce_ws.numel() == rec.reduce_ws_floats(32, widest)
    assert all(n.reduce_kw["ws"] is e.reduce_ws for n in e.nets.values())


@pytest.mark.parametrize("kwarg,env,expected", [
    (None, None, False), (None, "0", False), (None, "1", True),
    (True, "0", True), (False, "1", False), (True, None, True)])
def test_flag_precedence(rec, monkeypatch, kwarg, env, expected):
    from cellcomm_b200.bigan_cont import ContinuousCellBiGan
    if env is None:
        monkeypatch.delenv("CELLCOMM_B200_DETERMINISTIC", raising=False)
    else:
        monkeypatch.setenv("CELLCOMM_B200_DETERMINISTIC", env)
    net = ContinuousCellBiGan(3, 40, device="cpu", seed=0, deterministic=kwarg)
    assert net.deterministic is expected
    assert net._engine.deterministic is expected


def test_seed_makes_the_priors_repeatable(rec):
    from cellcomm_b200.bigan_cont import ContinuousCellBiGan
    from cellcomm_b200.bigan_classify import ClassifyCellBiGan
    a = ContinuousCellBiGan(3, 40, device="cpu", seed=5)
    b = ContinuousCellBiGan(3, 40, device="cpu", seed=5)
    c = ContinuousCellBiGan(3, 40, device="cpu", seed=6)
    pa, pb = a.random_uniform_vector(64), b.random_uniform_vector(64)
    assert np.array_equal(pa, pb)
    assert np.array_equal(a.random_encoding_vector(8), b.random_encoding_vector(8))
    assert not np.array_equal(pa, c.random_uniform_vector(64))
    k1 = ClassifyCellBiGan(4, 40, device="cpu", seed=5)
    k2 = ClassifyCellBiGan(4, 40, device="cpu", seed=5)
    assert np.array_equal(k1.random_uniform_vector(64), k2.random_uniform_vector(64))
    u = ContinuousCellBiGan(3, 40, device="cpu")
    v = ContinuousCellBiGan(3, 40, device="cpu")
    assert not np.array_equal(u.random_uniform_vector(64), v.random_uniform_vector(64))


def test_cell_training_forwards_seed_only_when_given(monkeypatch):
    from cellcomm_b200 import bigan_cont
    from cellcomm_b200.cell_type_training import CellTraining
    made = []

    class Net:
        def __init__(self, *args, **kwargs):
            made.append((args, kwargs))
    monkeypatch.setattr(bigan_cont, "ContinuousCellBiGan", Net)
    data = np.zeros((5, 7))
    CellTraining(data, 3, 2)
    CellTraining(data, 3, 2, 4, seed=11)
    assert made == [((2,), {"gene_size": 7}), ((2,), {"gene_size": 7, "seed": 11})]


@pytest.mark.parametrize("value,expected", [(None, None), ("", None), ("7", 7), (" 42 ", 42),
                                            ("-3", -3)])
def test_cellcomm_seed_parsing(monkeypatch, value, expected):
    from cellcomm_b200 import __main__ as entry
    if value is None:
        monkeypatch.delenv("CELLCOMM_SEED", raising=False)
    else:
        monkeypatch.setenv("CELLCOMM_SEED", value)
    assert entry.env_seed() == expected


def test_cellcomm_seed_rejects_garbage(monkeypatch):
    from cellcomm_b200 import __main__ as entry
    monkeypatch.setenv("CELLCOMM_SEED", "seven")
    with pytest.raises(ValueError):
        entry.env_seed()


@pytest.mark.parametrize("seed", [None, 7])
def test_run_training_seeds_the_sampler_and_the_network(monkeypatch, seed):
    from cellcomm_b200 import __main__ as entry
    made = []

    class Trainer:
        def __init__(self, cells, **kwargs):
            made.append(kwargs)

        def run(self, iterations, interceptors):
            made.append(np.random.randint(0, 1 << 30))
    if seed is None:
        monkeypatch.delenv("CELLCOMM_SEED", raising=False)
    else:
        monkeypatch.setenv("CELLCOMM_SEED", str(seed))
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.setattr(entry, "load_matrix", lambda path, verbose=False: "cells")
    monkeypatch.setattr(entry, "CellTraining", Trainer)
    monkeypatch.setattr(entry, "create_interceptors", lambda *a: None)
    entry.run_training(16)
    assert made[0] == {"batch_size": 16, "encoding_size": 3, "seed": seed}
    if seed is not None:
        np.random.seed(seed)
        assert made[1] == np.random.randint(0, 1 << 30)
