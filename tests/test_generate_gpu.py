"""Generated cells as a sparse matrix on the GPU: the round + compaction kernels against
scipy, generate_cell_matrix against generate_cells (bit for bit), no side effects on training,
device memory bounded by one tile, the .mtx round trip and the `generate` command."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

EDGE = [0.5, 1.5, 2.5, 0.49999997, -0.4, -0.5, -0.7, -0.0]
TILE_BYTES_33694 = 4096 * 33728 * 4           # fp32 generator tile, ld padded to 64


def _ops():
    from cellcomm_b200 import ops
    return ops


def _tile(host, ld, pad=7.0):
    """[rows, cols] view of a [rows, ld] device buffer whose padding columns hold `pad`"""
    rows, cols = host.shape
    buf = torch.full((max(rows, 1), ld), pad, dtype=torch.float32, device="cuda")
    buf[:rows, :cols] = torch.from_numpy(host)
    return buf[:rows, :cols]


def _compact(x, base=0):
    """count + fill -> host (rowptr, colidx, values)"""
    ops = _ops()
    rows = x.shape[0]
    rowptr = torch.full((rows + 1,), -1, dtype=torch.int64, device="cuda")
    rowptr[0] = base
    ops.round_csr_count(x, rowptr)
    nnz = int(rowptr[-1]) - base
    colidx = torch.full((nnz,), -1, dtype=torch.int32, device="cuda")
    values = torch.full((nnz,), 99.0, dtype=torch.float32, device="cuda")
    ops.round_csr_fill(x, rowptr, colidx, values)
    torch.cuda.synchronize()
    return rowptr.cpu().numpy(), colidx.cpu().numpy(), values.cpu().numpy()


def _check(host, got, base=0):
    want = sp.csr_matrix(np.rint(host))
    want.eliminate_zeros()
    rowptr, colidx, values = got
    np.testing.assert_array_equal(rowptr, base + want.indptr.astype(np.int64))
    np.testing.assert_array_equal(colidx, want.indices)
    assert values.dtype == np.float32
    assert values.tobytes() == want.data.astype(np.float32).tobytes()


def _random(rows, cols, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(0.0, 1.5, (rows, cols)).astype(np.float32)
    x[rng.random((rows, cols)) < 0.3] = 0.0
    return x


def test_round_half_even_edges():
    x = np.array([EDGE, [-v for v in EDGE]], dtype=np.float32)
    got = _compact(_tile(x, 64))
    _check(x, got)
    np.testing.assert_array_equal(got[0], [0, 3, 6])
    np.testing.assert_array_equal(got[1], [1, 2, 6, 1, 2, 6])
    np.testing.assert_array_equal(got[2], [2, 2, -1, -2, -2, 1])


@pytest.mark.parametrize("cols", [1, 3, 5, 127, 129, 33694])
@pytest.mark.parametrize("ld", ["pad64", "odd"])
def test_kernels_match_scipy(cols, ld):
    """vector path (ld padded to 64) and scalar path (odd ld): padding columns hold 7.0, which
    would round to a non-zero if it were read as an entry"""
    rows = 37
    x = _random(rows, cols, cols)
    x[3] = 0.0                                   # an all-zero row
    x[4] = 3.0                                   # an all-non-zero row
    x[5, : len(EDGE[:cols])] = EDGE[:cols]
    if ld == "pad64":
        ldx = (cols + 63) // 64 * 64
    else:
        ldx = cols + 1 if (cols + 1) % 4 else cols + 2
    _check(x, _compact(_tile(x, ldx)))


def test_zero_rows_and_zero_cols():
    ops = _ops()
    rowptr = torch.full((1,), 5, dtype=torch.int64, device="cuda")
    x = torch.zeros((0, 100), dtype=torch.float32, device="cuda")
    ops.round_csr_count(x, rowptr)
    ops.round_csr_fill(x, rowptr, torch.zeros(0, dtype=torch.int32, device="cuda"),
                       torch.zeros(0, dtype=torch.float32, device="cuda"))
    assert int(rowptr[0]) == 5
    host = np.zeros((4, 0), np.float32)
    _check(host, _compact(_tile(host, 64), base=3), base=3)


def test_base_offset_and_chained_tiles():
    a, b = _random(50, 1000, 1), _random(70, 1000, 2)
    _check(a, _compact(_tile(a, 1024), base=123456789012), base=123456789012)
    # two tiles through one device rowptr: the second call's base is the first one's end
    ops = _ops()
    rowptr = torch.zeros(121, dtype=torch.int64, device="cuda")
    xa, xb = _tile(a, 1024), _tile(b, 1024)
    ops.round_csr_count(xa, rowptr[:51])
    ops.round_csr_count(xb, rowptr[50:])
    na, nb = int(rowptr[50]), int(rowptr[120] - rowptr[50])
    ca, va = (torch.empty(na, dtype=t, device="cuda") for t in (torch.int32, torch.float32))
    cb, vb = (torch.empty(nb, dtype=t, device="cuda") for t in (torch.int32, torch.float32))
    ops.round_csr_fill(xa, rowptr[:51], ca, va)
    ops.round_csr_fill(xb, rowptr[50:], cb, vb)
    both = np.concatenate([a, b])
    _check(both, (rowptr.cpu().numpy(), torch.cat([ca, cb]).cpu().numpy(),
                  torch.cat([va, vb]).cpu().numpy()))


def test_repeated_launch_same_bytes():
    x = _tile(_random(300, 33694, 5), 33728)
    first = _compact(x)
    for _ in range(2):
        again = _compact(x)
        for u, v in zip(first, again):
            assert u.tobytes() == v.tobytes()


# ------------------------------------------------------------------ the public API
def _net(variant, G, seed=3, **kw):
    if variant == "cont":
        from cellcomm_b200.bigan_cont import ContinuousCellBiGan as N
    else:
        from cellcomm_b200.bigan_classify import ClassifyCellBiGan as N
    return N(3, G, seed=seed, **kw)


def _expressive(net, seed=0):
    """An untrained generator rounds almost everything to 0: shift its output bias by a seeded
    uniform [-1, 3) so that the rounded cells hold zeros, small counts and .5 ties."""
    gen = net._engine.G
    w = gen.get_weights()
    w[-1] = w[-1] + np.random.default_rng(seed).uniform(-1.0, 3.0, w[-1].shape).astype(np.float32)
    gen.set_weights(w)
    return net


def _priors(net, n, seed):
    rng = np.random.default_rng(seed)
    if net.VARIANT == "cont":
        z = rng.random((n, 3), dtype=np.float32)
    else:
        z = np.eye(3, dtype=np.float32)[rng.integers(0, 3, n)]
    return z, rng.random((n, 3), dtype=np.float32)


@pytest.mark.parametrize("variant", ["cont", "classify"])
@pytest.mark.parametrize("G,n", [(300, 1000), (33694, 2 * 4096 + 123)])
def test_generate_cell_matrix_equals_generate_cells(variant, G, n):
    net = _expressive(_net(variant, G))
    z, r = _priors(net, n, G)
    dense = net.generate_cells(z, r)
    m = net.generate_cell_matrix(z, r)
    assert m.shape == (n, G)
    np.testing.assert_array_equal(m.index, np.arange(1, n + 1))
    np.testing.assert_array_equal(m.columns, np.arange(1, G + 1))
    got = m.to_numpy(np.float32)
    assert np.array_equal(got, dense)
    assert m.nnz == np.count_nonzero(dense)
    assert 0.2 * n * G < m.nnz < 0.95 * n * G
    # strictly ascending columns inside every row (the CSR every consumer expects)
    inside = np.ones(max(m.nnz - 1, 0), bool)
    starts = m.rowptr[1:-1]
    inside[starts[(starts > 0) & (starts < m.nnz)] - 1] = False
    assert np.all(np.diff(m.colidx.astype(np.int64))[inside] > 0)


@pytest.mark.parametrize("variant", ["cont", "classify"])
def test_random_in_none_draws_like_generate_cells(variant):
    net = _expressive(_net(variant, 500))
    z, _ = _priors(net, 700, 1)
    state = net._prior_rng.bit_generator.state
    dense = net.generate_cells(z)
    net._prior_rng.bit_generator.state = state
    cols = np.arange(500, dtype=np.int64) * 2 + 11
    m = net.generate_cell_matrix(z, columns=cols)
    assert net._prior_rng.bit_generator.state == _advance(state, 700)
    assert np.array_equal(m.to_numpy(np.float32), dense)
    np.testing.assert_array_equal(m.columns, cols)
    with pytest.raises(ValueError, match="ascending gene ids"):
        net.generate_cell_matrix(z, columns=cols[::-1])


def _advance(state, n):
    g = np.random.default_rng()
    g.bit_generator.state = state
    g.random((n, 3), dtype=np.float32)
    return g.bit_generator.state


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


def test_generation_between_steps_has_no_side_effects():
    from cellcomm_b200.cell_type_training import CellBatch, CellMatrix
    G, N, B = 800, 400, 64
    rng = np.random.default_rng(4)
    data = CellMatrix.from_dense(((rng.random((N, G)) < 0.1) * rng.poisson(2.0, (N, G)))
                                 .astype(np.float64))
    pos = [rng.permutation(N)[:B] for _ in range(2)]

    def run(generate):
        net = _net("cont", G, seed=21, deterministic=True)
        losses = [[float(v) for v in net.trainings_step(CellBatch(data, pos[0]))]]
        before = _engine_state(net)
        if generate:
            z, r = _priors(net, 5000, 9)          # two tiles: the engine's buffers grow
            net.generate_cell_matrix(z, r)
            after = _engine_state(net)
            assert all(torch.equal(before[k], after[k]) for k in before)
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
    eng = net._engine
    z, r = _priors(net, 4097, 2)
    net.generate_cell_matrix(z, r)                 # warm up: the generator's 4096-row buffers
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    z, r = _priors(net, n, 3)
    seen = {"rows": 0, "nnz": 0}

    def consume(row0, rowptr, colidx, values):
        assert row0 == seen["rows"] and rowptr[0] == 0
        assert len(colidx) == len(values) == rowptr[-1]
        seen["rows"] += len(rowptr) - 1
        seen["nnz"] += int(rowptr[-1])

    eng.generate_csr(z, r, consume=consume)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    worst_entries = 4096 * G * 8
    assert seen["rows"] == n and seen["nnz"] > 0
    assert grown <= TILE_BYTES_33694 + worst_entries + (16 << 20), grown
    assert grown < n * G * 4 // 8


def test_mtx_round_trip_and_encoding(tmp_path):
    from cellcomm_b200.cell_type_training import CellMatrix, load_matrix
    G, n = 256, 600
    net = _expressive(_net("cont", G, seed=6))
    z, r = _priors(net, n, 5)
    m = net.generate_cell_matrix(z, r, columns=np.arange(G) * 3 + 100)
    back = load_matrix(m.to_mtx(str(tmp_path / "gen.mtx")))
    dense = m.to_numpy()
    rows, cols = dense.any(1), dense.any(0)
    want = CellMatrix.from_dense(dense[rows][:, cols], index=m.index[rows],
                                 columns=m.columns[cols])
    for name in ("rowptr", "colidx", "index", "columns"):
        np.testing.assert_array_equal(getattr(back, name), getattr(want, name), err_msg=name)
    assert back.values64.tobytes() == want.values64.tobytes()
    if cols.all():
        enc = net.encoding_prediction(back)
        assert enc.shape == (len(back), 3) and np.isfinite(enc).all()
        assert np.array_equal(enc, net.encoding_prediction(want))


def test_generate_command_is_repeatable(tmp_path):
    from cellcomm_b200.__main__ import main
    from cellcomm_b200.cell_type_training import CellMatrix, load_matrix
    G, n = 2000, 300
    net = _expressive(_net("cont", G, seed=12))
    ckpt = str(tmp_path / "net.npz")
    net.save_checkpoint(ckpt)
    src = CellMatrix.from_dense(np.ones((3, G)), columns=np.arange(G) + 7)
    src_path = src.to_mtx(str(tmp_path / "source.mtx"))
    outs = [str(tmp_path / f"gen{i}.mtx") for i in range(2)]
    state = np.random.get_state()
    for out in outs:
        main(["", "generate", ckpt, src_path, str(n), out])
    np.random.set_state(state)
    assert open(outs[0], "rb").read() == open(outs[1], "rb").read()
    back = load_matrix(outs[0])
    assert len(back) == n
    assert set(back.columns) <= set(src.columns)
    assert sorted(os.listdir(tmp_path)) == ["gen0.mtx", "gen1.mtx", "net.npz", "source.mtx"]
