"""Cell scores on the GPU: cc_recon_sqerr against fp64 numpy, score_cells against its
definition (encoding_prediction, G.predict, D.predict), no side effects on training, device
memory bounded by one tile, the `score` command and the validation.csv interceptor of the entry
point."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _ops():
    from cellcomm_b200 import ops
    return ops


def _csr(dense):
    from cellcomm_b200.cell_type_training import CellMatrix
    return CellMatrix.from_dense(dense)


def _pred_tile(host, ld, pad=float("nan")):
    """[rows, cols] view of a [rows, ld] device buffer whose padding columns hold `pad`"""
    rows, cols = host.shape
    buf = torch.full((max(rows, 1), ld), pad, dtype=torch.float32, device="cuda")
    buf[:rows, :cols] = torch.from_numpy(host)
    return buf[:rows, :cols]


def _sqerr(pred, mat, row0=0, scale=1.0):
    ops = _ops()
    rowptr, colidx, values = mat.device_csr("cuda")
    out = torch.full((pred.shape[0],), -1.0, dtype=torch.float32, device="cuda")
    ops.recon_sqerr(pred, rowptr, colidx, values, row0, out, scale=scale)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _want(pred, dense, scale=1.0):
    return scale * np.sum(np.square(pred.astype(np.float64) - dense.astype(np.float64)), axis=1)


def _close(got, want, rel=1e-5):
    assert got.dtype == np.float32
    np.testing.assert_allclose(got, want, rtol=rel, atol=0)


def _counts(rows, cols, seed, density=0.1):
    rng = np.random.default_rng(seed)
    x = np.where(rng.random((rows, cols)) < density, rng.geometric(0.3, (rows, cols)), 0)
    return x.astype(np.float64)


@pytest.mark.parametrize("cols", [5, 63, 65, 1000, 33694])
@pytest.mark.parametrize("ld", ["pad64", "odd"])
def test_recon_sqerr_matches_fp64(cols, ld):
    """vector path (ld a multiple of 4) and scalar path (odd ld); NaN in the padding columns
    would poison any sum that read them"""
    rows = 37
    x = _counts(rows, cols, cols)
    x[3] = 0.0                                   # an empty row
    x[4] = np.arange(1, cols + 1)                # a fully dense row
    pred = np.random.default_rng(cols + 1).normal(0.0, 2.0, (rows, cols)).astype(np.float32)
    pred[5] = x[5]                               # a perfect reconstruction
    ldx = (cols + 63) // 64 * 64 if ld == "pad64" else (cols + 1 if (cols + 1) % 4 else cols + 2)
    got = _sqerr(_pred_tile(pred, ldx), _csr(x), scale=1.0 / cols)
    _close(got, _want(pred, x, 1.0 / cols))
    assert got[5] == 0.0


def test_recon_sqerr_explicit_zeros_count_once():
    from cellcomm_b200.cell_type_training import CellMatrix
    # row 0: an explicit zero at column 1 next to a stored 5 at column 3; row 1: only zeros
    m = CellMatrix(np.array([0, 2, 4]), np.array([1, 3, 0, 2]), np.array([0.0, 5.0, 0.0, 0.0]),
                   np.array([1, 2]), np.arange(1, 5))
    pred = np.array([[1.0, 2.0, 3.0, 4.0], [0.5, 0.0, -1.5, 2.0]], np.float32)
    got = _sqerr(_pred_tile(pred, 64), m)
    _close(got, _want(pred, m.to_numpy()))
    np.testing.assert_array_equal(got, [1 + 4 + 9 + 1, 0.25 + 2.25 + 4])


def test_recon_sqerr_row0_into_a_larger_csr():
    x = _counts(500, 777, 3)
    mat = _csr(x)
    pred = np.random.default_rng(4).normal(0, 1, (120, 777)).astype(np.float32)
    got = _sqerr(_pred_tile(pred, 832), mat, row0=313)
    _close(got, _want(pred, x[313:433]))
    with pytest.raises(ValueError, match="outside"):
        _sqerr(_pred_tile(pred, 832), mat, row0=381)


def test_recon_sqerr_no_cancellation():
    """x = 4,000 and p = 4,000.25 on most genes: the squares are 0.0625 each; the expanded form
    sum p^2 - 2 sum p x + sum x^2 loses them all in fp32"""
    cols = 33694
    x = np.zeros((4, cols))
    x[:, : 30000] = 4000.0
    pred = x.astype(np.float32) + np.float32(0.25)
    got = _sqerr(_pred_tile(pred, 33728), _csr(x), scale=1.0 / cols)
    want = _want(pred, x, 1.0 / cols)
    _close(got, want)
    p32, x32 = pred.astype(np.float32), x.astype(np.float32)
    expanded = ((p32 * p32).sum(1, dtype=np.float32) - 2 * (p32 * x32).sum(1, dtype=np.float32)
                + (x32 * x32).sum(1, dtype=np.float32)) / cols
    assert np.all(np.abs(expanded - want) > 0.1 * want)      # visibly wrong


def test_recon_sqerr_repeated_launches_same_bits():
    x = _counts(300, 33694, 9, density=0.06)
    pred = _pred_tile(np.random.default_rng(2).normal(0, 3, (300, 33694)).astype(np.float32),
                      33728)
    mat = _csr(x)
    first = _sqerr(pred, mat)
    for _ in range(3):
        assert _sqerr(pred, mat).tobytes() == first.tobytes()


def test_recon_sqerr_rejects_too_many_columns():
    from cellcomm_b200 import _lib
    cols = (1 << 18) + 1
    pred = torch.zeros((1, cols), dtype=torch.float32, device="cuda")
    mat = _csr(np.zeros((1, 1)))
    with pytest.raises(_lib.CCError, match="bitmap"):
        _ops().recon_sqerr(pred, *mat.device_csr("cuda"), 0,
                           torch.zeros(1, dtype=torch.float32, device="cuda"))


# ------------------------------------------------------------------ the public API
def _net(variant, G, seed=3, **kw):
    if variant == "cont":
        from cellcomm_b200.bigan_cont import ContinuousCellBiGan as N
    else:
        from cellcomm_b200.bigan_classify import ClassifyCellBiGan as N
    return N(3, G, seed=seed, **kw)


def _cells(n, G, seed, per_row=60):
    """n cells built as a CSR (no dense intermediate): per_row stored genes per cell, one in
    each of per_row equal column bands, counts 1 + geometric; 1 % of the cells empty and 5 %
    with a count of 3,000 (above the 256 that bf16 holds exactly)"""
    from cellcomm_b200.cell_type_training import CellMatrix
    rng = np.random.default_rng(seed)
    k = min(per_row, G)
    band = G // k
    cols = (np.arange(k) * band + rng.integers(0, band, (n, k))).astype(np.int32)
    vals = rng.geometric(0.3, (n, k)).astype(np.float64)
    vals[rng.random(n) < 0.05, 0] = 3000.0
    counts = np.where(rng.random(n) < 0.01, 0, k)
    keep = np.arange(k)[None, :] < counts[:, None]
    rowptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(counts, out=rowptr[1:])
    return CellMatrix(rowptr, cols[keep], vals[keep], np.arange(1, n + 1), np.arange(1, G + 1))


@pytest.mark.parametrize("variant", ["cont", "classify"])
@pytest.mark.parametrize("G,n", [(5, 7), (33694, 5000)])
def test_score_cells_matches_the_definition(variant, G, n):
    net = _net(variant, G)
    mat = _cells(n, G, G)
    r = np.random.default_rng(1).random((n, 3), dtype=np.float32)
    s = net.score_cells(mat, r)
    assert s.encodings.shape == (n, 3) and s.mse.shape == (n,) and s.d_real.shape == (n,)
    assert all(a.dtype == np.float32 for a in s)
    z = net.encoding_prediction(mat)
    assert s.encodings.tobytes() == z.tobytes()
    d = net._discriminator.predict((z, mat)).reshape(-1)
    assert s.d_real.tobytes() == d.tobytes()
    assert np.all((s.d_real >= 0) & (s.d_real <= 1))
    pred = net._generator.predict((z, r)).astype(np.float64)
    want = np.mean(np.square(pred - mat.to_numpy()), axis=1)
    np.testing.assert_allclose(s.mse, want, rtol=1e-5, atol=0)


def test_score_cells_wraps_other_inputs_and_draws_like_generate_cells():
    from cellcomm_b200.cell_type_training import CellBatch
    net = _net("cont", 700)
    mat = _cells(300, 700, 2)
    state = net._prior_rng.bit_generator.state
    numpy_state = np.random.get_state()
    s = net.score_cells(mat)                                      # random_in=None
    after = net._prior_rng.bit_generator.state
    g = np.random.default_rng()
    g.bit_generator.state = state
    r = g.random((300, 3), dtype=np.float32)
    assert after == g.bit_generator.state
    again = net.score_cells(mat, r)
    assert net._prior_rng.bit_generator.state == after             # random_in given: no draw
    assert np.random.get_state()[1].tobytes() == numpy_state[1].tobytes()
    for a, b in zip(s, again):
        assert a.tobytes() == b.tobytes()
    dense = net.score_cells(mat.to_numpy(np.float32), r)
    batch = net.score_cells(CellBatch(mat, np.arange(300)), r)
    for a, b, c in zip(again, dense, batch):
        assert a.tobytes() == b.tobytes() == c.tobytes()


def _engine_state(net):
    e = net._engine
    e.join()
    torch.cuda.synchronize()
    out = {"rng": e.rng_counter.clone(), "loss": e.loss_buf.clone()}
    for k, n in e.nets.items():
        out[k + ".p32"], out[k + ".p16"] = n.p32.clone(), n.p16.clone()
        out[k + ".ms"], out[k + ".mom"] = n.ms.clone(), n.mom.clone()
        for i, L in enumerate(L for L in n.layers if L["kind"] == "bn"):
            out[f"{k}.bn{i}.mean"] = L["moving_mean"].clone()
            out[f"{k}.bn{i}.var"] = L["moving_var"].clone()
    return out


def test_scoring_between_steps_has_no_side_effects():
    from cellcomm_b200.cell_type_training import CellBatch
    G, N, B = 800, 400, 64
    data = _cells(N, G, 4, per_row=80)
    rng = np.random.default_rng(4)
    pos = [rng.permutation(N)[:B] for _ in range(2)]
    held = _cells(5000, G, 5)                     # two tiles: the engine's buffers grow
    r = np.random.default_rng(6).random((5000, 3), dtype=np.float32)

    def run(score):
        net = _net("cont", G, seed=21, deterministic=True)
        losses = [[float(v) for v in net.trainings_step(CellBatch(data, pos[0]))]]
        before = _engine_state(net)
        if score:
            np_state, prior = np.random.get_state(), net._prior_rng.bit_generator.state
            net.score_cells(held, r)
            after = _engine_state(net)
            assert all(torch.equal(before[k], after[k]) for k in before)
            assert np.random.get_state()[1].tobytes() == np_state[1].tobytes()
            assert net._prior_rng.bit_generator.state == prior
        losses.append([float(v) for v in net.trainings_step(CellBatch(data, pos[1]))])
        return losses, _engine_state(net)

    la, sa = run(True)
    lb, sb = run(False)
    assert la == lb
    bad = [k for k in sa if not torch.equal(sa[k], sb[k])]
    assert not bad, bad


def test_device_memory_is_bounded_by_one_tile():
    G, n = 33694, 100_000
    net = _net("cont", G, seed=8)
    warm = _cells(4097, G, 1)
    net.score_cells(warm, np.zeros((4097, 3), np.float32))        # the nets' 4096-row buffers
    mat = _cells(n, G, 2)
    rowptr, colidx, values = mat.device_csr("cuda")
    r = np.random.default_rng(3).random((n, 3), dtype=np.float32)
    enc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    mse = torch.empty(n, dtype=torch.float32, device="cuda")
    d = torch.empty(n, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    net._engine.score_stream(rowptr, colidx, values, 0, n, r, enc, mse, d)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    tiles = 4096 * 33728 * (4 + 2)                # the fp32 generator tile + the bf16 cell tile
    assert grown <= tiles + n * 3 * 4 + (16 << 20), grown
    assert grown < n * G * 4 // 8
    assert torch.isfinite(mse).all() and torch.isfinite(d).all()


# ------------------------------------------------------------------ the score command
def _expressive(net, seed=0):
    gen = net._engine.G
    w = gen.get_weights()
    w[-1] = w[-1] + np.random.default_rng(seed).uniform(-1.0, 3.0, w[-1].shape).astype(np.float32)
    gen.set_weights(w)
    return net


def test_score_command_is_repeatable_and_aligns_genes(tmp_path):
    from cellcomm_b200.__main__ import main
    from cellcomm_b200.cell_type_training import CellMatrix
    G, n = 2000, 300
    net = _expressive(_net("cont", G, seed=12))
    ckpt = str(tmp_path / "net.npz")
    net.save_checkpoint(ckpt)
    genes = np.arange(G) * 2 + 7
    src = CellMatrix.from_dense(np.ones((3, G)), columns=genes)
    src_path = src.to_mtx(str(tmp_path / "source.mtx"))
    # the scored matrix: 1,500 of the source's genes and 300 the source does not have
    rng = np.random.default_rng(5)
    own = np.union1d(rng.choice(genes, 1500, replace=False), genes[-1] + 2 * np.arange(1, 301))
    x = _counts(n, len(own), 8, density=0.2)
    x[:, 0] += 1.0                                   # every row and column survives the file
    x[0, :] += 1.0
    cells = CellMatrix.from_dense(x, index=np.arange(n) * 3 + 11, columns=own)
    cells_path = cells.to_mtx(str(tmp_path / "cells.mtx"))
    outs = [str(tmp_path / f"s{i}.csv") for i in range(2)]
    state = np.random.get_state()
    for out in outs:
        main(["", "score", ckpt, src_path, cells_path, out])
    np.random.set_state(state)
    text = open(outs[0], "rb").read()
    assert text == open(outs[1], "rb").read()
    lines = text.decode().splitlines()
    assert lines[0] == "barcode,mse,d-real,z0,z1,z2" and len(lines) == n + 1
    got = np.array([[float(v) for v in line.split(",")] for line in lines[1:]])
    np.testing.assert_array_equal(got[:, 0], cells.index)
    # = scoring the dense reindexed equivalent with the checkpoint's own noise draw
    ref = _net("cont", G, seed=99)
    ref.load_checkpoint(ckpt)
    aligned = np.zeros((n, G))
    where = np.searchsorted(genes, own)
    ok = (where < G) & (genes[np.minimum(where, G - 1)] == own)
    aligned[:, where[ok]] = x[:, ok]
    want = ref.score_cells(aligned)
    assert got[:, 1].astype(np.float32).tobytes() == want.mse.tobytes()
    assert got[:, 2].astype(np.float32).tobytes() == want.d_real.tobytes()
    assert got[:, 3:].astype(np.float32).tobytes() == want.encodings.tobytes()
    assert sorted(os.listdir(tmp_path)) == ["cells.mtx", "net.npz", "s0.csv", "s1.csv",
                                            "source.mtx"]


# ------------------------------------------------------------------ the entry point
def _entry_point_data(tmp):
    sys.path.insert(0, HERE)
    from test_entry_point_gpu import SOURCE, _write_data_dir
    _write_data_dir(tmp)
    held = os.path.join(tmp, "held_out.mtx")
    rng = np.random.default_rng(17)
    with open(held, "w") as f:                        # genes 1..750: 50 the source lacks
        rows = [(g, b, int(rng.integers(1, 9))) for b in range(1, 41)
                for g in sorted(rng.choice(np.arange(1, 751), 60, replace=False))]
        f.write(f"%%MatrixMarket matrix coordinate integer general\n%\n750 40 {len(rows)}\n")
        f.writelines(f"{g} {b} {v}\n" for g, b, v in rows)
    return SOURCE, held


def _run(cmd, tmp, held):
    env = dict(os.environ, CELLCOMM_DATA_DIR=tmp, CELLCOMM_ITERATIONS="3",
               CELLCOMM_BATCH_SIZE="16", CELLCOMM_VALIDATION_MATRIX=held,
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "src"), ROOT]))
    out = subprocess.run(cmd, cwd=tmp, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-3000:])
    runs = os.listdir(os.path.join(tmp, "logs"))
    assert len(runs) == 1
    lines = open(os.path.join(tmp, "logs", runs[0], "validation.csv")).read().splitlines()
    assert lines[0] == "iteration,mse,d-real,real-pct"
    assert [line.split(",")[0] for line in lines[1:]] == ["0", "1", "2"]
    vals = np.array([[float(v) for v in line.split(",")[1:]] for line in lines[1:]])
    assert np.isfinite(vals).all() and np.all(vals[:, 0] > 0)
    assert np.all((vals[:, 1] >= 0) & (vals[:, 1] <= 1)) and np.all((vals[:, 2] >= 0) & (vals[:, 2] <= 1))


def test_entry_point_writes_validation_rows(tmp_path):
    tmp = str(tmp_path)
    _, held = _entry_point_data(tmp)
    _run([sys.executable, os.path.join(ROOT, "src")], tmp, held)


def test_entry_point_validation_under_torchrun_two_gpus(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    tmp = str(tmp_path)
    _, held = _entry_point_data(tmp)
    port = 29500 + (os.getpid() % 200)
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
          "--master-addr", "127.0.0.1", "--master-port", str(port), "-m", "cellcomm_b200"],
         tmp, held)
