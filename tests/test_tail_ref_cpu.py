"""The host references of tests/tail_ref.py checked on their own, without a GPU: Philox against
the Random123 known-answer vectors and a scalar port, the RNG counter layout, the bf16 helpers
against torch, and the fp64 formulas against torch autograd."""
import numpy as np
import pytest
import torch

import tail_ref as R

M32 = 0xFFFFFFFF

# Random123 kat_vectors, philox4x32_10: (counter, key) -> output
PHILOX_KAT = [
    ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    ([M32] * 4, [M32, M32], [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
     [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
]


def _words_to_halves(ctr, key):
    lo = ctr[0] | (ctr[1] << 32)
    hi = ctr[2] | (ctr[3] << 32)
    return key[0] | (key[1] << 32), hi, lo


@pytest.mark.parametrize("ctr,key,want", PHILOX_KAT)
def test_philox_known_answers(ctr, key, want):
    assert R.philox_scalar(ctr, key) == want
    seed, hi, lo = _words_to_halves(ctr, key)
    got = R.philox_block(seed, np.uint64(hi), np.uint64(lo))
    assert [int(v) for v in got] == want


def test_philox_vectorised_matches_scalar():
    rng = np.random.default_rng(5)
    n = 300
    seeds = [int(v) for v in rng.integers(0, 2 ** 64, n, dtype=np.uint64)]
    seeds[:4] = [0, M32, 1 << 32, (1 << 64) - 1]          # high key word alone / all ones
    his = rng.integers(0, 2 ** 64, n, dtype=np.uint64)
    los = rng.integers(0, 2 ** 64, n, dtype=np.uint64)
    for i in range(n):
        got = R.philox_block(seeds[i], his[i], los[i])
        h, l = int(his[i]), int(los[i])
        want = R.philox_scalar([l & M32, l >> 32, h & M32, h >> 32],
                               [seeds[i] & M32, seeds[i] >> 32])
        assert [int(v) for v in got] == want, i
    # broadcasting one key over a vector of counters
    got = R.philox_block(seeds[7], his[3], los[:50])
    for j in range(50):
        l, h = int(los[j]), int(his[3])
        assert [int(v) for v in got[j]] == R.philox_scalar(
            [l & M32, l >> 32, h & M32, h >> 32], [seeds[7] & M32, seeds[7] >> 32])


@pytest.mark.parametrize("seed,step,sid", [(0, 0, 0), (123, 7, 5), ((0xDEADBEEF << 32) | 17, 3, 1000),
                                           (99, (1 << 33) + 5, (1 << 24) - 1),
                                           ((1 << 64) - 1, (1 << 40) - 1, 0)])
@pytest.mark.parametrize("rows,cols", [(1, 1), (3, 9), (2, 4), (4, 6), (2, 15)])
def test_rng_layout_matches_scalar(seed, step, sid, rows, cols):
    """rng_uniform(r, c) is lane c % 4 of block r * ceil(cols / 4) + c // 4 with counter hi
    (sid << 40) ^ step: checked element by element with the scalar Philox."""
    u = R.rng_uniform(seed, step, sid, rows, cols)
    assert u.shape == (rows, cols) and u.dtype == np.float32
    bpr = (cols + 3) // 4
    hi = ((sid << 40) ^ step) & ((1 << 64) - 1)
    for r in range(rows):
        for c in range(cols):
            blk = r * bpr + c // 4
            o = R.philox_scalar([blk & M32, blk >> 32, hi & M32, hi >> 32],
                                [seed & M32, seed >> 32])[c % 4]
            assert u[r, c] == np.float32((o >> 8) / 2 ** 24)


def test_rng_stream_id_limits():
    """The documented limits of the counter layout: stream ids alias modulo 2^24, and ids below
    2^24 give distinct streams."""
    a = R.rng_uniform(1, 2, 5, 2, 8)
    assert np.array_equal(a, R.rng_uniform(1, 2, 5 + (1 << 24), 2, 8))
    assert not np.array_equal(a, R.rng_uniform(1, 2, 6, 2, 8))
    assert not np.array_equal(R.rng_uniform(1, 2, 0, 2, 8), R.rng_uniform(1, 2, (1 << 24) - 1, 2, 8))
    # a step of 2^40 lands on stream id 1's counters
    assert np.array_equal(R.rng_uniform(1, 1 << 40, 0, 2, 8), R.rng_uniform(1, 0, 1, 2, 8))


def test_uniform_range_and_bf16_edge():
    u = R.rng_uniform(9, 0, 1, 512, 1024)
    assert u.min() >= 0 and u.max() < 1
    assert abs(float(u.mean()) - 0.5) < 5e-3
    # bf16 rounding of u >= 1 - 2^-9 reaches exactly 1.0 (the top of the bf16 [0.5, 1) binade
    # has spacing 2^-8): cc_uniform's bf16 copy is in [0, 1], not [0, 1)
    top = np.float32(1 - 2.0 ** -24)
    assert R.bf16_round(np.array([top], np.float32))[0] == 1.0
    assert (R.bf16_round(u) == 1.0).any()


def _bf16_torch(x32):
    return torch.from_numpy(x32).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def test_bf16_helpers_match_torch():
    rng = np.random.default_rng(1)
    x = np.concatenate([
        rng.standard_normal(100000).astype(np.float32) * 10.0 ** rng.integers(-30, 30, 100000),
        rng.integers(0, 2 ** 32, 100000, dtype=np.uint64).astype(np.uint32).view(np.float32),  # noqa
        np.array([0.0, -0.0, np.inf, -np.inf, 1.0, 1 + 2 ** -8, 1 + 3 * 2 ** -8, 1 + 2 ** -9,
                  1 + 3 * 2 ** -9, 3.3895314e38, 3.4028235e38, 1e-45, -1e-45, 2 ** -126,
                  2 ** -133 * 3], np.float32)])
    x = x[~np.isnan(x)]
    assert np.array_equal(R.bf16_bits(x), _bf16_torch(x))
    assert np.array_equal(R.bf16_round(x).view(np.uint32),
                          torch.from_numpy(x).to(torch.bfloat16).float().numpy().view(np.uint32))
    nan = np.array([np.nan], np.float32)
    assert np.isnan(R.bf16_round(nan)[0])


def test_split_matches_torch():
    rng = np.random.default_rng(2)
    x = (rng.standard_normal(200000) * 10.0 ** rng.integers(-20, 20, 200000)).astype(np.float32)
    hi, lo = R.split_ref(x)
    t = torch.from_numpy(x)
    th = t.to(torch.bfloat16)
    tl = (t - th.float()).to(torch.bfloat16)
    assert np.array_equal(hi.view(np.uint32), th.float().numpy().view(np.uint32))
    assert np.array_equal(lo.view(np.uint32), tl.float().numpy().view(np.uint32))
    # hi + lo keeps 16 significant bits
    err = np.abs(hi.astype(np.float64) + lo - x)
    assert np.all(err <= np.abs(x.astype(np.float64)) * 2.0 ** -16)


def test_ulp_helpers():
    assert R.ulp32(1.0) == 2.0 ** -23 and R.ulp32(1.5) == 2.0 ** -23 and R.ulp32(0.75) == 2.0 ** -24
    assert R.ulp16(1.0) == 2.0 ** -7 and R.ulp16(-3.0) == 2.0 ** -6
    assert R.ulp32(0.0) == 2.0 ** -149


def test_fp64_formulas_match_torch_autograd():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((37, 5)) * 2 + 30
    gamma, beta = rng.random(5) + 0.5, rng.standard_normal(5)
    dy = rng.standard_normal((37, 5)) + 0.3
    y, mean, rstd, var = R.bn_train64(x, gamma, beta, 1e-3)
    xt = torch.from_numpy(x).requires_grad_(True)
    gt, bt = torch.from_numpy(gamma).requires_grad_(True), torch.from_numpy(beta).requires_grad_(True)
    yt = torch.nn.functional.batch_norm(xt, None, None, gt, bt, training=True, eps=1e-3)
    yt.backward(torch.from_numpy(dy))
    assert np.allclose(y, yt.detach().numpy(), rtol=1e-12, atol=1e-12)
    assert np.allclose(var, x.var(0)) and np.allclose(mean, x.mean(0))
    dx, dg, db = R.bn_train_bwd64(dy, x, gamma, 1e-3)
    assert np.allclose(dx, xt.grad.numpy(), rtol=1e-10, atol=1e-12)
    assert np.allclose(dg, gt.grad.numpy(), rtol=1e-10) and np.allclose(db, bt.grad.numpy())
    # softmax and its backward
    z = rng.standard_normal((9, 7)) * 30
    zt = torch.from_numpy(z).requires_grad_(True)
    st = torch.softmax(zt, -1)
    g = rng.standard_normal((9, 7))
    st.backward(torch.from_numpy(g))
    s = R.softmax64(z)
    assert np.allclose(s, st.detach().numpy(), rtol=1e-12, atol=1e-300)
    assert np.allclose(R.softmax_bwd64(g, s), zt.grad.numpy(), rtol=1e-9, atol=1e-15)
    # losses
    lg = np.array([-100, -88, -20, -5, -1e-3, 1e-3, 5, 20, 88, 100.0])
    for t in (0.0, float(np.float32(0.95)), 1.0):
        ls = torch.nn.functional.logsigmoid
        want = -(t * ls(torch.from_numpy(lg)) + (1 - t) * ls(-torch.from_numpy(lg)))
        assert np.allclose(R.bce_logits64(lg, t), want.numpy(), rtol=1e-13, atol=1e-300)
    p = np.array([0.0, 1e-9, 0.5, 1 - 1e-9, 1.0])
    eps = np.float32(1e-7)              # Keras clips in fp32: [eps, 1 - eps] = [1e-7, 1 - 2^-23]
    q = np.clip(p, float(eps), float(np.float32(1) - eps))
    assert float(np.float32(1) - eps) == 1 - 2.0 ** -23
    assert np.allclose(R.bce_probs64(p, 0.95), -(0.95 * np.log(q) + 0.05 * np.log(1 - q)),
                       rtol=1e-6)
    pr, tg = rng.standard_normal((6, 4)), rng.standard_normal((6, 4))
    prt = torch.from_numpy(pr).requires_grad_(True)
    lt = torch.nn.functional.mse_loss(prt, torch.from_numpy(tg)) * 6 / 12   # n_total = 12
    lt.backward()
    loss, grad = R.mse64(pr, tg, 12)
    assert np.isclose(loss, lt.item(), rtol=1e-13) and np.allclose(grad, prt.grad.numpy())
    assert np.array_equal(R.onehot_argmax(np.array([[1.0, 3, 3], [-np.inf, -np.inf, -np.inf]])),
                          np.array([[0, 1, 0], [1, 0, 0]], np.float32))
    assert np.array_equal(R.round_half_even(np.array([0.5, 1.5, 2.5, -0.5, -2.5])),
                          np.array([0.0, 2, 2, -0.0, -2]))


def test_rmsprop64_matches_keras_recurrence():
    w, g = np.array([1.0, -2.0]), np.array([0.5, 0.0])
    ms, mom = np.zeros(2), np.zeros(2)
    w1, ms1, mom1 = R.rmsprop64(w, g, ms, mom, 0.0075, 0.85, 0.1, 1e-7)
    assert np.allclose(ms1, [0.15 * 0.25, 0.0])
    assert np.allclose(mom1, [0.0075 * 0.5 / np.sqrt(0.15 * 0.25 + 1e-7), 0.0])
    assert np.allclose(w1, w - mom1)


def test_colreduce_geometry():
    # one column block: slabs fill ~2 waves but keep >= 64 rows each
    assert R.colreduce_grid(4096, 1, 148) == (1, 64, 64)
    assert R.colreduce_grid(65, 129, 148) == (2, 2, 33)
    # 2 * SMs - 1 column blocks: one slab each would be too few for 2 waves, so two slabs;
    # from 2 * SMs blocks on, one slab
    assert R.colreduce_grid(4096, 128 * 295, 148)[1] == 2
    assert R.colreduce_grid(4096, 128 * 296, 148)[1] == 1
    assert R.colreduce_adds(2048, 1, 148) == 64 // 8 + 8 + 32
    assert R.fallback_cols(148) == 2424845
