"""Comparing generated cells with real ones on the GPU: cc_col_moments against fp64 numpy, the
streamed gene_statistics / generated_gene_statistics against their definitions, compare_cells'
grouping, no side effects on training, device memory bounded by one tile, and the `compare`
command."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ops():
    from cellcomm_b200 import ops
    return ops


def _tile(host, ld, pad=float("nan")):
    """[rows, cols] view of a [rows, ld] device buffer whose padding columns hold `pad`"""
    rows, cols = host.shape
    buf = torch.full((max(rows, 1), ld), pad, dtype=torch.float32, device="cuda")
    buf[:rows, :cols] = torch.from_numpy(np.ascontiguousarray(host, dtype=np.float32))
    return buf[:rows, :cols]


def _ld(cols, kind):
    return (cols + 63) // 64 * 64 if kind == "pad64" else (cols + 1 if (cols + 1) % 4 else cols + 2)


def _acc(cols):
    return (torch.zeros(cols, dtype=torch.float64, device="cuda"),
            torch.zeros(cols, dtype=torch.float64, device="cuda"),
            torch.zeros(cols, dtype=torch.int64, device="cuda"))


def _ws(rows, cols):
    n = _ops().col_moments_ws_bytes(rows, cols)
    return torch.zeros(n, dtype=torch.uint8, device="cuda") if n else None


def _moments(x, round=False, acc=None, ws="auto"):
    acc = acc or _acc(x.shape[1])
    _ops().col_moments(x, *acc, round=round, ws=_ws(*x.shape) if ws == "auto" else ws)
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy() for t in acc)


def _want(x, round=False):
    v = x.astype(np.float64)
    if round:
        v = np.rint(v)
    return v.sum(0), (v * v).sum(0), np.count_nonzero(v, axis=0).astype(np.int64)


def _counts(rows, cols, seed, density=0.1):
    rng = np.random.default_rng(seed)
    x = np.where(rng.random((rows, cols)) < density, rng.geometric(0.3, (rows, cols)), 0)
    return x.astype(np.float32)


@pytest.mark.parametrize("cols", [5, 63, 65, 1000, 33694])
@pytest.mark.parametrize("rows", [0, 1, 37, 4096])
@pytest.mark.parametrize("ld", ["pad64", "odd"])
def test_col_moments_matches_fp64(cols, rows, ld):
    """vector path (ld a multiple of 4) and scalar path (odd ld); NaN in the padding columns
    would poison any sum that read them.  Integer data: exact; random floats: rtol 1e-12."""
    x = _counts(rows, cols, cols + rows)
    if rows:
        x[0, :] = np.arange(cols) % 7                     # a dense row with zeros in it
    got = _moments(_tile(x, _ld(cols, ld)))
    want = _want(x)
    for g, w in zip(got, want):
        assert g.tobytes() == w.tobytes()
    f = np.where(x > 0, np.random.default_rng(rows).random(x.shape) * 50, 0).astype(np.float32)
    got = _moments(_tile(f, _ld(cols, ld)))
    want = _want(f)
    np.testing.assert_allclose(got[0], want[0], rtol=1e-12, atol=0)
    np.testing.assert_allclose(got[1], want[1], rtol=1e-12, atol=0)
    np.testing.assert_array_equal(got[2], want[2])


@pytest.mark.parametrize("ld", ["pad64", "odd"])
def test_col_moments_round_half_even(ld):
    vals = np.array([0.5, 1.5, 2.5, -1.5, -0.4, -0.5, 0.49999997, 3.7], np.float32)
    x = np.resize(vals, (600, 9))                          # several slabs, shifted columns
    s1, s2, nz = _moments(_tile(x, _ld(9, ld)), round=True)
    w1, w2, wn = _want(x, round=True)
    assert s1.tobytes() == w1.tobytes() and s2.tobytes() == w2.tobytes()
    np.testing.assert_array_equal(nz, wn)
    # per value: rint(0.5) = 0, 1.5 -> 2, 2.5 -> 2, -1.5 -> -2, -0.4 -> -0.0 (not detected)
    one = _tile(np.array([[0.5, 1.5, 2.5, -1.5, -0.4]], np.float32), _ld(5, ld))
    s1, s2, nz = _moments(one, round=True)
    np.testing.assert_array_equal(s1, [0.0, 2.0, 2.0, -2.0, 0.0])
    np.testing.assert_array_equal(nz, [0, 1, 1, 1, 0])
    s1, _, nz = _moments(one, round=False)
    np.testing.assert_array_equal(nz, [1, 1, 1, 1, 1])
    np.testing.assert_array_equal(s1, np.float64(np.float32([0.5, 1.5, 2.5, -1.5, -0.4])))


def test_col_moments_chained_halves_equal_one_launch():
    x = _counts(4096, 33694, 5, density=0.3)
    t = _tile(x, 33728)
    whole = _moments(t)
    acc = _acc(33694)
    ws = _ws(4096, 33694)                                 # one workspace serves both halves
    _ops().col_moments(t[:1500], *acc, ws=ws)
    halves = _moments(t[1500:], acc=acc, ws=ws)
    for a, b in zip(whole, halves):
        assert a.tobytes() == b.tobytes()


def test_col_moments_repeated_launches_same_bits():
    f = np.random.default_rng(2).normal(3.0, 2.0, (4096, 20000)).astype(np.float32)
    t = _tile(f, 20032)
    first = _moments(t)
    for _ in range(3):
        again = _moments(t)
        assert all(a.tobytes() == b.tobytes() for a, b in zip(first, again))


def test_col_moments_rejects_a_small_workspace():
    from cellcomm_b200 import _lib
    t = _tile(np.ones((4096, 1000), np.float32), 1024)
    need = _ops().col_moments_ws_bytes(4096, 1000)
    assert need > 0 and _ops().col_moments_ws_bytes(256, 1000) == 0
    for ws in (None, torch.zeros(need - 1, dtype=torch.uint8, device="cuda")):
        acc = _acc(1000)
        with pytest.raises(_lib.CCError, match="workspace"):
            _ops().col_moments(t, *acc, ws=ws)
        torch.cuda.synchronize()
        assert all(int(a.abs().sum()) == 0 for a in acc)   # nothing was added


# ------------------------------------------------------------------ the public API
def _net(variant, G, seed=3, **kw):
    if variant == "cont":
        from cellcomm_b200.bigan_cont import ContinuousCellBiGan as N
    else:
        from cellcomm_b200.bigan_classify import ClassifyCellBiGan as N
    return N(3, G, seed=seed, **kw)


def _expressive(net, seed=0):
    """raise the generator's output biases so generated cells are far from empty"""
    gen = net._engine.G
    w = gen.get_weights()
    w[-1] = w[-1] + np.random.default_rng(seed).uniform(-1.0, 3.0, w[-1].shape).astype(np.float32)
    gen.set_weights(w)
    return net


def _cells(n, G, seed, per_row=60):
    """n cells built as a CSR: per_row stored genes per cell, counts 1 + geometric, 1 % of the
    cells empty and 5 % with a count of 3,000"""
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


def _same(a, b):
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and x.shape == y.shape
        assert x.tobytes() == y.tobytes()


@pytest.mark.parametrize("variant", ["cont", "classify"])
def test_gene_statistics_streams_the_definition(variant):
    from cellcomm_b200.bigan_basic import BasicBiGan
    G, n = 33694, 5000
    net = _net(variant, G)
    mat = _cells(n, G, 7)
    labels = np.random.default_rng(1).choice([0, 2, 4], n, p=[0.2, 0.7, 0.1])
    labels[123] = 3                                       # a group of one; group 1 is empty
    got = net.gene_statistics(mat, labels, 5)
    _same(got, BasicBiGan.gene_statistics(net, mat, labels, 5))
    np.testing.assert_array_equal(got.cells, np.bincount(labels, minlength=5))
    assert np.isnan(got.mean[1]).all() and np.isnan(got.var[3]).all()
    assert not np.isnan(got.mean[2]).any()
    # a dense array is wrapped with CellMatrix.from_dense
    small = _cells(300, G, 8)
    _same(net.gene_statistics(small.to_numpy(np.float32)), net.gene_statistics(small))


@pytest.mark.parametrize("variant", ["cont", "classify"])
def test_generated_gene_statistics_streams_the_definition(variant):
    """three generator tiles; group 1 ends on a tile edge, group 2 is empty, group 3 crosses
    a tile edge, groups 0 and 4 lie inside one tile"""
    from cellcomm_b200.bigan_basic import BasicBiGan
    G = 33694
    net = _expressive(_net(variant, G, seed=5))
    bounds = [0, 1000, 4096, 4096, 8500, 8692]
    n = bounds[-1]
    labels = np.repeat(np.arange(5), np.diff(bounds))
    enc = np.random.default_rng(2).random((n, 3), dtype=np.float32)
    r = np.random.default_rng(3).random((n, 3), dtype=np.float32)
    got = net.generated_gene_statistics(enc, r, labels, 5)
    cells = net.generate_cells(enc, r)
    assert np.count_nonzero(cells) > n * 1000              # far from empty
    _same(got, BasicBiGan.gene_statistics(net, cells, labels, 5))
    del cells
    _same(got, net.gene_statistics(net.generate_cell_matrix(enc, r), labels, 5))
    with pytest.raises(ValueError, match="sorted by group"):
        net.generated_gene_statistics(enc, r, labels[::-1], 5)


@pytest.mark.parametrize("variant", ["cont", "classify"])
def test_compare_cells_groups_and_counts(variant):
    G, n = 2000, 3000
    net = _expressive(_net(variant, G, seed=9))
    mat = _cells(n, G, 4)
    state = net._prior_rng.bit_generator.state
    c = net.compare_cells(mat)
    if variant == "classify":
        labels = np.argmax(net.encoding_prediction(mat), -1)
        K = 3
    else:
        labels, K = np.zeros(n, np.int64), 1
    _same(c.real, net.gene_statistics(mat, labels, K))
    np.testing.assert_array_equal(c.generated.cells, c.real.cells)
    assert c.real.cells.sum() == n
    # the same draws again give the same generated statistics
    net._prior_rng.bit_generator.state = state
    if variant == "classify":
        enc = np.repeat(np.eye(3, dtype=np.float32), c.real.cells, axis=0)
    else:
        enc = net.random_encoding_vector(n)
    noise = net.random_uniform_vector(n)
    _same(c.generated, net.generated_gene_statistics(enc, noise, np.repeat(np.arange(K),
                                                                            c.real.cells), K))


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


def test_statistics_between_steps_have_no_side_effects():
    from cellcomm_b200.cell_type_training import CellBatch
    G, N, B = 800, 400, 64
    data = _cells(N, G, 4, per_row=80)
    rng = np.random.default_rng(4)
    pos = [rng.permutation(N)[:B] for _ in range(2)]
    enc = np.random.default_rng(5).random((5000, 3), dtype=np.float32)   # two tiles
    r = np.random.default_rng(6).random((5000, 3), dtype=np.float32)
    labels = np.repeat([0, 1], [3000, 2000])

    def run(compare):
        net = _net("cont", G, seed=21, deterministic=True)
        losses = [[float(v) for v in net.trainings_step(CellBatch(data, pos[0]))]]
        before = _engine_state(net)
        if compare:
            np_state, prior = np.random.get_state(), net._prior_rng.bit_generator.state
            net.generated_gene_statistics(enc, r, labels)
            net.gene_statistics(data, np.arange(N) % 3)
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
    G, n, K = 33694, 100_000, 3
    net = _net("cont", G, seed=8)
    warm = np.zeros((4097, 3), np.float32)
    net.generated_gene_statistics(warm, warm)              # the nets' 4096-row buffers
    enc = np.random.default_rng(2).random((n, 3), dtype=np.float32)
    r = np.random.default_rng(3).random((n, 3), dtype=np.float32)
    bounds = [0, 30_000, 30_001, n]
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    sums = net._engine.moments_stream(bounds, z32=enc, r32=r)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    tile = 4096 * 33728 * 4
    accumulators = 3 * K * G * 8
    ws = _ops().col_moments_ws_bytes(4096, G)
    latents = 2 * n * 3 * 4
    assert grown <= tile + accumulators + ws + latents + (16 << 20), grown
    assert grown < n * G * 4 // 8
    sizes = torch.tensor(np.diff(bounds), device="cuda")[:, None]
    assert bool((sums[2] <= sizes).all()) and bool((sums[0] >= 0).all())


# ------------------------------------------------------------------ the compare command
def test_compare_command_is_repeatable_and_matches_compare_cells(tmp_path):
    from cellcomm_b200.__main__ import main
    from cellcomm_b200.bigan_basic import comparison_summary
    from cellcomm_b200.cell_type_training import CellMatrix
    G, n = 2000, 700
    net = _expressive(_net("classify", G, seed=12))
    ckpt = str(tmp_path / "net.npz")
    net.save_checkpoint(ckpt)
    genes = np.arange(G) * 2 + 7
    src = CellMatrix.from_dense(np.ones((3, G)), columns=genes)
    src_path = src.to_mtx(str(tmp_path / "source.mtx"))
    rng = np.random.default_rng(5)
    own = np.union1d(rng.choice(genes, 1500, replace=False), genes[-1] + 2 * np.arange(1, 301))
    x = np.where(rng.random((n, len(own))) < 0.2, rng.geometric(0.3, (n, len(own))), 0)
    x = x.astype(np.float64)
    x[:, 0] += 1.0                                       # every row and column survives the file
    x[0, :] += 1.0
    cells = CellMatrix.from_dense(x, index=np.arange(n) * 3 + 11, columns=own)
    cells_path = cells.to_mtx(str(tmp_path / "cells.mtx"))
    outs = [str(tmp_path / f"out{i}") for i in range(2)]
    state = np.random.get_state()
    for out in outs:
        main(["", "compare", ckpt, src_path, cells_path, out])
    np.random.set_state(state)
    for name in ("genes.csv", "groups.csv"):
        assert open(os.path.join(outs[0], name), "rb").read() == \
            open(os.path.join(outs[1], name), "rb").read()
    assert sorted(os.listdir(outs[0])) == ["genes.csv", "groups.csv"]
    # = compare_cells of the aligned cells on the restored checkpoint
    ref = _net("classify", G, seed=99)
    ref.load_checkpoint(ckpt)
    want = ref.compare_cells(cells.reindex_columns(genes))
    lines = open(os.path.join(outs[0], "genes.csv")).read().splitlines()
    assert len(lines) == 1 + 3 * G
    got = np.array([[float(v) for v in line.split(",")] for line in lines[1:]])
    np.testing.assert_array_equal(got[:, 0], np.repeat(np.arange(3), G))
    np.testing.assert_array_equal(got[:, 1], np.tile(genes, 3))
    for j, a in enumerate((want.real.mean, want.real.var, want.real.detected,
                           want.generated.mean, want.generated.var, want.generated.detected)):
        assert got[:, 2 + j].tobytes() == a.reshape(-1).tobytes()
    rows = open(os.path.join(outs[0], "groups.csv")).read().splitlines()[1:]
    for line, row in zip(rows, comparison_summary(want)):
        f = line.split(",")
        assert [int(v) for v in f[:3]] == [row.group, row.real_cells, row.generated_cells]
        assert np.array([float(v) for v in f[3:]]).tobytes() == \
            np.array(row[3:], dtype=np.float64).tobytes()
    assert sum(int(line.split(",")[1]) for line in rows) == n
