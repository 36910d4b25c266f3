"""The two-sample test on the GPU: cc_log1p_features bit for bit against the numpy definition,
cc_mmd_sums against fp64 numpy on the same fp32 Gram matrix, the streamed two_sample_test
against the base-class definition, calibration, no side effects between training steps, the
device-memory bound and the `twosample` command."""
import os

import numpy as np
import pytest
import torch

from cellcomm_b200.bigan_basic import (BasicBiGan, MMD_SCALES, kernel_sums, log1p_features,
                                       pack_labellings, permutation_p_value, mmd_from_sums,
                                       two_sample_labellings)

pytestmark = pytest.mark.gpu


def _ops():
    from cellcomm_b200 import ops
    return ops


def _tile(host, ld, pad=float("nan")):
    rows, cols = host.shape
    buf = torch.full((max(rows, 1), ld), pad, dtype=torch.float32, device="cuda")
    buf[:rows, :cols] = torch.from_numpy(np.ascontiguousarray(host, dtype=np.float32))
    return buf[:rows, :cols]


def _features(x, ld, round):
    ops = _ops()
    rows, cols = x.shape
    t = _tile(x, ld)
    fld = (cols + 63) // 64 * 64
    fbuf = torch.full((max(rows, 1), fld), 1.0, dtype=torch.bfloat16, device="cuda")
    f = fbuf[:rows, :cols]
    lib = torch.full((rows,), -1.0, dtype=torch.float64, device="cuda")
    det = torch.full((rows,), -1, dtype=torch.int32, device="cuda")
    ops.log1p_features(t, f, lib, det, round=round)
    torch.cuda.synchronize()
    return fbuf[:rows].view(torch.int16).cpu().numpy(), lib.cpu().numpy(), det.cpu().numpy()


@pytest.mark.parametrize("cols", [5, 63, 64, 1000, 33694])
@pytest.mark.parametrize("rows", [0, 1, 37, 300])
@pytest.mark.parametrize("ld", ["pad", "odd"])
@pytest.mark.parametrize("round", [False, True])
def test_log1p_features_bit_exact(cols, rows, ld, round):
    rng = np.random.default_rng(cols * 7 + rows)
    x = np.where(rng.random((rows, cols)) < 0.2, rng.geometric(0.2, (rows, cols)), 0)
    x = x.astype(np.float32)
    if rows:
        x[0, : min(cols, 6)] = [-0.0, 0.5, 2.5, 300.0, 1e5, 255.0][: min(cols, 6)]
        if rows > 1:
            x[1] = rng.random(cols).astype(np.float32) * 1000     # non-integers, fp64 log1p
    ldx = (cols + 63) // 64 * 64 if ld == "pad" else cols + (1 if (cols + 1) % 4 else 2)
    f, lib, det = _features(x, ldx, round)
    v = np.rint(x) if round else x
    want = log1p_features(v.astype(np.float64))
    fld = (cols + 63) // 64 * 64
    exp = np.zeros((rows, fld), np.float32)
    exp[:, :cols] = want
    exp_bits = (exp.view(np.uint32) >> 16).astype(np.uint16).view(np.int16)
    assert f.tobytes() == exp_bits.tobytes()
    np.testing.assert_array_equal(lib, v.astype(np.float64).sum(1))
    np.testing.assert_array_equal(det, np.count_nonzero(v, axis=1))


def _gram_case(N, K, seed):
    rng = np.random.default_rng(seed)
    F = rng.normal(size=(N, K)).astype(np.float32)
    G32 = (F.astype(np.float64) @ F.T.astype(np.float64)).astype(np.float32)
    G32 = (G32 + G32.T) / 2
    ld = (N + 63) // 64 * 64
    buf = torch.full((N, ld), float("nan"), dtype=torch.float32, device="cuda")
    buf[:, :N] = torch.from_numpy(G32)
    return G32, buf[:, :N]


def _d2_fp32(G32):
    g = np.diag(G32)
    return np.maximum((g[:, None] + g[None, :]).astype(np.float32) - np.float32(2) * G32,
                      np.float32(0))


def _device_sums(gram, inv, masks):
    ops = _ops()
    L = len(masks)
    out = torch.empty((L, len(inv), 3), dtype=torch.float64, device="cuda")
    ws = torch.empty(max(1, ops.mmd_sums_ws_bytes(gram.shape[0], len(inv), L)),
                     dtype=torch.uint8, device="cuda")
    ops.mmd_sums(gram, inv, torch.from_numpy(pack_labellings(masks).view(np.int32)).cuda(), out,
                 ws=ws)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("N", [2, 129, 1000, 4096])
def test_mmd_sums_matches_fp64(N):
    G32, gram = _gram_case(N, 16, N)
    d2 = _d2_fp32(G32)
    med = float(np.sort(d2[np.triu_indices(N, 1)])[(N * (N - 1) // 2 - 1) // 2])
    inv = [np.float32(1.0 / (s * med)) for s in (0.5, 1.0, 2.0, 3.0)][: 3 if N > 2 else 4]
    n = N // 2
    masks = two_sample_labellings(n, 7, 1, 0)
    if N % 2:
        masks = np.concatenate([masks, np.zeros((len(masks), 1), bool)], 1)
    got = _device_sums(gram, inv, masks)
    want = kernel_sums(d2.astype(np.float64), masks, [1.0 / float(g) for g in inv])
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-300)
    again = _device_sums(gram, inv, masks)
    assert got.tobytes() == again.tobytes()


def test_mmd_sums_rejects_a_small_workspace():
    from cellcomm_b200 import _lib
    ops = _ops()
    G32, gram = _gram_case(300, 8, 3)
    masks = torch.from_numpy(pack_labellings(two_sample_labellings(150, 3, 0, 0)).view(np.int32))
    need = ops.mmd_sums_ws_bytes(300, 2, 4)
    out = torch.zeros((4, 2, 3), dtype=torch.float64, device="cuda")
    for ws in (None, torch.zeros(need - 8, dtype=torch.uint8, device="cuda")):
        with pytest.raises(_lib.CCError, match="workspace"):
            ops.mmd_sums(gram, [1.0, 2.0], masks.cuda(), out, ws=ws)


# ------------------------------------------------------------------ the public API
def _net(variant, G, seed=3, **kw):
    if variant == "cont":
        from cellcomm_b200.bigan_cont import ContinuousCellBiGan as N
    else:
        from cellcomm_b200.bigan_classify import ClassifyCellBiGan as N
    return N(3, G, seed=seed, **kw)


def _expressive(net, seed=0):
    gen = net._engine.G
    w = gen.get_weights()
    w[-1] = w[-1] + np.random.default_rng(seed).uniform(-1.0, 3.0, w[-1].shape).astype(np.float32)
    gen.set_weights(w)
    return net


def _cells(n, G, seed, per_row=60, scale=1):
    from cellcomm_b200.cell_type_training import CellMatrix
    rng = np.random.default_rng(seed)
    k = min(per_row, G)
    band = G // k
    cols = (np.arange(k) * band + rng.integers(0, band, (n, k))).astype(np.int32)
    vals = rng.geometric(0.3, (n, k)).astype(np.float64) * scale
    rowptr = np.arange(n + 1, dtype=np.int64) * k
    return CellMatrix(rowptr, cols.reshape(-1), vals.reshape(-1), np.arange(1, n + 1),
                      np.arange(1, G + 1))


@pytest.mark.parametrize("variant", ["cont", "classify"])
def test_two_sample_test_streams_the_definition(variant):
    """33,694 genes; a generator tile of 1,024 rows here (PREDICT_TILE is what generate_cells
    and the stream both tile by), so generation crosses tiles while the host definition stays
    affordable"""
    G, n, P = 33694, 1500, 40
    net = _expressive(_net(variant, G, seed=5))
    net.PREDICT_TILE = 1024
    mat = _cells(n, G, 7)
    state = net._prior_rng.bit_generator.state
    np_state = np.random.get_state()
    got = net.two_sample_test(mat, max_cells=1400, permutations=P, seed=3)
    net._prior_rng.bit_generator.state = state
    np.random.set_state(np_state)
    want = BasicBiGan.two_sample_test(net, mat, max_cells=1400, permutations=P, seed=3)
    np.testing.assert_array_equal(got.real_cells, want.real_cells)
    np.testing.assert_array_equal(got.generated_cells, want.generated_cells)
    assert got.generated_cells.sum() > 1024
    np.testing.assert_allclose(got.sqdist_median, want.sqdist_median, rtol=1e-4)
    live = want.real_cells >= 2
    nn = want.real_cells[live].astype(np.float64)
    assert np.isnan(got.mmd2[~live]).all()
    # tolerance relative to XX / (n (n - 1)) + YY / (n (n - 1)) ~ 2 * mean kernel value <= 2
    np.testing.assert_allclose(got.mmd2[live], want.mmd2[live], atol=2e-4, rtol=0)
    assert np.all(np.abs(got.p_value[live] - want.p_value[live]) <= 3.0 / (P + 1))
    np.testing.assert_array_equal(got.library_size_ks, want.library_size_ks)
    np.testing.assert_array_equal(got.genes_detected_ks, want.genes_detected_ks)
    assert nn.size


def _real_vs_real(net, a, b, P, seed):
    eng = net._engine
    csr = a.device_csr(eng.device)
    fa = eng.features_stream(csr=csr, order=np.arange(len(a)))[0]
    fb = eng.features_stream(csr=b.device_csr(eng.device), order=np.arange(len(b)))[0]
    n = len(a)
    _, sums = eng.mmd_sums(fa, fb, MMD_SCALES, pack_labellings(two_sample_labellings(n, P, seed,
                                                                                      0)))
    return permutation_p_value(mmd_from_sums(n, sums[..., 0], sums[..., 1], sums[..., 2]))


def test_calibration():
    from cellcomm_b200.cell_type_training import CellMatrix
    G, P = 2000, 200
    net = _net("cont", G, seed=4)
    mat = _cells(1200, G, 9, per_row=40)
    dense = mat.to_numpy()
    low = 0
    for h in range(10):
        perm = np.random.default_rng([h, 77]).permutation(len(dense))
        a = CellMatrix.from_dense(dense[perm[:600]])
        b = CellMatrix.from_dense(dense[perm[600:]])
        low += int(np.sum(_real_vs_real(net, a, b, P, h) < 0.05))
    assert low <= 3, low
    a = CellMatrix.from_dense(dense[:400])
    b = CellMatrix.from_dense(dense[:400] * 2)
    np.testing.assert_array_equal(_real_vs_real(net, a, b, P, 0), [1.0 / (P + 1)] * 3)


def _engine_state(net):
    e = net._engine
    e.join()
    torch.cuda.synchronize()
    out = {"rng": e.rng_counter.clone(), "loss": e.loss_buf.clone()}
    for k, n in e.nets.items():
        out[k + ".p32"], out[k + ".p16"] = n.p32.clone(), n.p16.clone()
        out[k + ".ms"], out[k + ".mom"] = n.ms.clone(), n.mom.clone()
    return out


def test_two_sample_test_between_steps_has_no_side_effects():
    from cellcomm_b200.cell_type_training import CellBatch
    G, N, B = 800, 400, 64
    data = _cells(N, G, 4, per_row=80)
    pos = [np.random.default_rng(4).permutation(N)[:B] for _ in range(2)]

    def run(test):
        net = _net("cont", G, seed=21, deterministic=True)
        losses = [[float(v) for v in net.trainings_step(CellBatch(data, pos[0]))]]
        if test:
            before = _engine_state(net)
            # the test draws its priors from the host streams, as compare_cells does: put them
            # back so the next step draws what it would have drawn
            np_state, prior = np.random.get_state(), net._prior_rng.bit_generator.state
            net.two_sample_test(data, permutations=20)
            np.random.set_state(np_state)
            net._prior_rng.bit_generator.state = prior
            after = _engine_state(net)
            assert all(torch.equal(before[k], after[k]) for k in before)
        losses.append([float(v) for v in net.trainings_step(CellBatch(data, pos[1]))])
        return losses, _engine_state(net)

    la, sa = run(True)
    lb, sb = run(False)
    assert la == lb
    assert all(torch.equal(sa[k], sb[k]) for k in sa)


def test_device_memory_is_bounded():
    G, n = 33694, 4096
    net = _net("cont", G, seed=8)
    mat = _cells(n, G, 3)
    net.two_sample_test(_cells(10, G, 1), permutations=2)         # the nets' buffers
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    net.two_sample_test(mat, permutations=100)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    ld = 33728
    tile = 4096 * ld * 4
    feats = 2 * n * ld * 2
    gram = (2 * n) * (2 * n) * 4
    csr = mat.nnz * 16 + (n + 1) * 8
    assert grown <= tile + feats + 2 * gram + csr + (64 << 20), grown


def test_twosample_command_is_repeatable(tmp_path):
    from cellcomm_b200.__main__ import main
    from cellcomm_b200.cell_type_training import CellMatrix
    G, n = 2000, 700
    net = _expressive(_net("classify", G, seed=12))
    ckpt = str(tmp_path / "net.npz")
    net.save_checkpoint(ckpt)
    genes = np.arange(G) * 2 + 7
    src = CellMatrix.from_dense(np.ones((3, G)), columns=genes)
    src_path = src.to_mtx(str(tmp_path / "source.mtx"))
    rng = np.random.default_rng(5)
    x = np.where(rng.random((n, G)) < 0.05, rng.geometric(0.3, (n, G)), 0).astype(np.float64)
    x[:, 0] += 1.0
    x[0, :] += 1.0
    cells = CellMatrix.from_dense(x, index=np.arange(n) + 1, columns=genes)
    cells_path = cells.to_mtx(str(tmp_path / "cells.mtx"))
    outs = [str(tmp_path / f"t{i}.csv") for i in range(2)]
    for out in outs:
        main(["", "twosample", ckpt, src_path, cells_path, out])
    assert open(outs[0], "rb").read() == open(outs[1], "rb").read()
    ref = _net("classify", G, seed=99)
    ref.load_checkpoint(ckpt)
    want = ref.two_sample_test(cells.reindex_columns(genes))
    lines = open(outs[0]).read().splitlines()
    assert len(lines) == 1 + 3
    for k, line in enumerate(lines[1:]):
        f = line.split(",")
        assert [int(v) for v in f[:3]] == [k, want.real_cells[k], want.generated_cells[k]]
        vals = [want.sqdist_median[k]]
        for b in range(3):
            vals += [want.mmd2[k, b], want.p_value[k, b]]
        vals += [want.library_size_ks[k], want.genes_detected_ks[k]]
        assert np.array([float(v) for v in f[3:]]).tobytes() == np.array(vals).tobytes()
