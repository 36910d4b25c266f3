"""The GEMM host references of tests/gemm_ref.py, without a GPU: the exactness certificate,
the fp32 epilogue emulation on hand-worked cases, and the dispatch mirror's reach."""
import numpy as np
import pytest

import gemm_ref as G
import tail_ref as R

SMS = 148


@pytest.mark.parametrize("ks,shifts,emax", [
    ([1], None, 0),
    ([64], None, 20),
    ([257], None, 5),
    ([3369], None, 20),
    ([100, 100, 100], [(0, 0), (-8, 0), (0, -8)], 3),     # x_hi W + x_lo W + x_hi W_lo
    ([700, 700, 700], [(0, 0), (-9, 0), (0, -9)], 0),
    ([65, 1, 130, 7], None, 2),
])
def test_certificate_holds_in_every_order(ks, shifts, emax):
    """fp32 sums taken in sequential, reversed, shuffled, 64-blocked and split-then-summed
    orders all equal the exact fp64 product, segment by segment and summed over segments."""
    rng = np.random.default_rng(sum(ks))
    M, N = 5, 7
    ex = G.exact_operands(rng, M, N, ks, shifts, emax=emax)
    a = np.concatenate(ex.a, axis=1)
    b = np.concatenate(ex.b, axis=0)
    for i, s in enumerate(G.fp32_sum_orders(a, b, rng)):
        assert np.array_equal(s.astype(np.float64), ex.p64), f"order {i}"
    # the products are bf16 x bf16: exact in fp32
    assert np.array_equal(R.bf16_round(a), a) and np.array_equal(R.bf16_round(b), b)
    if sum(ks) >= 64:
        assert ex.full_width()[0, 0], "output (0, 0) must need all 24 bits"


def test_certificate_rejects_and_detects():
    rng = np.random.default_rng(1)
    with pytest.raises(AssertionError):
        G.exact_operands(rng, 2, 2, [300], mag=255)        # 300 * 255^2 > 2^24
    with pytest.raises(ValueError):
        G.max_mag(2 ** 25)
    # reduced-precision accumulation would fail: a bf16 or tf32 rounding of the full-width
    # output changes it
    ex = G.exact_operands(rng, 3, 3, [3369])
    v = ex.v32[0, 0]
    assert ex.full_width()[0, 0]
    assert R.bf16_round(np.float32(v)) != v
    tf32 = (np.array([v], np.float32).view(np.uint32) & ~np.uint32(0x1FFF)).view(np.float32)[0]
    assert tf32 != v
    # a dropped lo segment changes the result
    ex = G.exact_operands(rng, 4, 4, [50, 50], [(0, 0), (-8, 0)])
    hi_only = ex.a[0].astype(np.float64) @ ex.b[0].astype(np.float64)
    assert not np.array_equal(hi_only, ex.p64)


def test_fma32_single_rounding():
    # 1 + 2^-24 rounds to 1 as a product then sum, but fmaf keeps the tie-breaking bit
    a, b, c = np.float32(1 + 2 ** -12), np.float32(1 + 2 ** -12), np.float32(-1.0)
    assert G.fma32(a, b, c) == np.float32(2 ** -11 + 2 ** -24)
    assert (a * b + c) == np.float32(2 ** -11)              # two roundings lose 2^-24
    # ties of the fp32 result resolve to even, with the sticky bit from far below
    one = np.float32(1.0)
    assert G.fma32(one, np.float32(2 ** -24), one) == one                   # exact tie -> even
    assert G.fma32(np.float32(2 ** -24 + 2 ** -47), one, one) == np.float32(1 + 2 ** -23)
    assert G.fma32(np.float32(0.3), np.float32(10.0), np.float32(0.0)) == np.float32(0.3) * np.float32(10)
    rng = np.random.default_rng(2)
    x, y, z = (rng.standard_normal(10000).astype(np.float32) for _ in range(3))
    ref = [float(np.float32(float(np.longdouble(p) * q + r))) for p, q, r in zip(x[:50], y[:50], z[:50])]
    assert np.array_equal(G.fma32(x[:50], y[:50], z[:50]), np.array(ref, np.float32))
    got = G.fma32(x, y, z).astype(np.float64)
    exact = x.astype(np.float64) * y + z
    assert np.all(np.abs(got - exact) <= 0.5 * R.ulp32(got) + 1e-45)


def test_epilogue_hand_worked():
    v = np.array([[257.0, 259.0, -3.0, 0.0, 1.5]], np.float32)
    # out16: bf16 ties go to even (257 -> 256, 259 -> 260); -0.0 compares equal to 0
    x, _ = G.epilogue(v)
    assert G.store16(x).tolist() == [[256.0, 260.0, -3.0, 0.0, 1.5]]
    assert G.store16_lo(x).tolist() == [[1.0, -1.0, 0.0, 0.0, 0.0]]
    assert G.bf16_ties(x).tolist() == [[True, True, False, False, False]]
    # relu at zero and below; bias and alpha fused
    x, _ = G.epilogue(v, alpha=0.5, bias=np.array([0, 0, 1.5, -0.0, -0.75], np.float32), act=G.ACT_RELU)
    assert x.tolist() == [[128.5, 129.5, 0.0, 0.0, 0.0]]
    # act' relu: y > 0 only (y = 0 and y < 0 give 0)
    y = np.array([[1.0, 0.0, -2.0, 0.5, -0.0]], np.float32)
    x, _ = G.epilogue(v, dact=G.ACT_RELU, y=y)
    assert x.tolist() == [[257.0, 0.0, 0.0, 0.0, 0.0]]
    # act' sigmoid: y (1 - y) rounded, then the product rounded
    x, _ = G.epilogue(v, dact=G.ACT_SIGMOID, y=np.array([[0.5, 1.0, 0.0, 0.25, -1.0]], np.float32))
    assert x.tolist() == [[64.25, 0.0, -0.0, 0.0, -3.0]]
    # beta32: one fp32 add; beta16: fp32 add then one bf16 rounding
    prev = np.array([[2.0 ** 24, 1.0, 3.0, -0.0, 0.25]], np.float32)
    assert G.store32(v, prev).tolist() == [[2.0 ** 24 + 256, 260.0, 0.0, 0.0, 1.75]]
    prev16 = np.array([[1.0, 1.0, 0.5, 0.0, 0.0]], np.float32)
    assert G.store16(v, prev16).tolist() == [[258.0, 260.0, -2.5, 0.0, 1.5]]
    # sigmoid: held to a bound around the fp64 value of the exact pre-activation
    s, pre = G.epilogue(np.array([[0.0, 4.0]], np.float32), act=G.ACT_SIGMOID)
    assert s[0, 0] == 0.5 and pre.tolist() == [[0.0, 4.0]]
    tol = G.sigmoid_bound(s, pre, R.ulp32)
    assert np.all(tol > 0) and np.all(tol < 1e-6)


def test_store16_lo_matches_split_ref():
    rng = np.random.default_rng(3)
    x = (rng.standard_normal(20000) * 10.0 ** rng.uniform(-10, 10, 20000)).astype(np.float32)
    hi, lo = R.split_ref(x)
    assert np.array_equal(G.store16(x), hi) and np.array_equal(G.store16_lo(x), lo)


def test_kernel_name_parses_profiler_names():
    n = G.kernel_name("void cc::gemm_tcgen05_persistent_kernel<256, 4, false, true, true, 4, false, 2, "
                      "false>(cc::TmaMaps, cc::GemmParams, int, int)")
    assert n == G.persistent(256, 4, 0, 1, 1, 4, 0, 2, 0)
    assert G.kernel_name("void cc::gemm_tcgen05_kernel<128, 3, true, false>(cc::TmaMaps, cc::GemmParams)") \
        == G.onetile(128, 3, 1, 0)
    assert G.kernel_name("cc::splitk_finalize_kernel(cc::EpiParams, float const*, long long, long long, int)") \
        == "splitk_finalize_kernel"
    assert G.kernel_name("void cc::bias_act_kernel(float const*)") is None


def test_mirror_reaches_every_instantiation():
    insts = G.instantiations()
    assert len(insts) == 49
    seen = set()
    for c in G.coverage_cases():
        names, _ = G.dispatch(sms=SMS, **c)
        seen.update(names)
    assert seen == insts


def test_mirror_rules():
    # automatic split at batch 128 with a long reduction: min(2 SMs / tiles, k-blocks / 4) =
    # 131 wanted, 5 k-blocks each -> 106 k-ranges
    names, splits = G.dispatch(128, 512, [33694], 0, 1, sms=SMS, workspace_elems=1 << 24)
    assert splits == 106 and len(names) == 2
    # the workspace caps the split count; too small a workspace means no split
    _, s = G.dispatch(128, 300, [4000], 0, 1, sms=SMS, force_splits=7, workspace_elems=3 * 128 * 512)
    assert s == 3
    names, s = G.dispatch(128, 300, [4000], 0, 1, sms=SMS, force_splits=7, workspace_elems=128 * 512 + 1)
    assert s == 1 and len(names) == 1
    # no empty split: 10 k-blocks in 7 splits are 5 ranges of 2
    _, s = G.dispatch(128, 300, [640], 0, 1, sms=SMS, force_splits=7, workspace_elems=1 << 24)
    assert s == 5
    # a fused optimiser never splits, and takes a cluster only for a long batch reduction
    names, s = G.dispatch(300, 300, [512], 1, 1, sms=SMS, rms="reg", workspace_elems=1 << 24)
    assert s == 1 and names[0].endswith(",1,0>")
    names, _ = G.dispatch(300, 300, [576], 1, 1, sms=SMS, rms="blocked")
    assert names[0].endswith(",2,1>")
