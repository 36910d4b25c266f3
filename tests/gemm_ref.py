"""Host references for the tcgen05 GEMM (csrc/gemm_sm100.cu); no GPU needed.

Three parts:
- Exactly summable operands.  a[i, k] = m[i, k] 2^(e_i + sa) and b[k, j] = n[k, j] 2^(f_j + sb)
  with integers |m|, |n| <= 255 (exact in bf16), an exponent per row of A and per column of B
  and a shift (sa, sb) per segment (-8 / -9 for the low-order term of a hi + lo pair).  Every
  product of output (i, j) is then a multiple of g = 2^(e_i + f_j + min_s(sa + sb)); when the
  magnitudes of all terms sum to less than 2^24 g, every partial sum is an fp32 number and fp32
  accumulation is exact in any order.  `exact_operands` checks that certificate and returns the
  exact product (integer-valued fp64 BLAS sums below 2^53 are exact).
- The fp32 epilogue in numpy, in the kernels' order of operations: v = fmaf(v, alpha, bias),
  act, v *= act'(y), then the stores, beta and the low-order term.  Every step is one IEEE
  operation on exact inputs, so it is bit exact; sigmoid (__expf) is the one step held to a
  bound instead.
- A mirror of gemm_impl's dispatch rules: which kernel instantiations a descriptor launches.
"""
import math
import re

import numpy as np

import tail_ref as R

BM, BK = 128, 64
F32_BITS = 24


# ------------------------------------------------------------------------ exact operands
class Exact:
    """Operands of one GEMM: a[s] logical [M, k_s] and b[s] logical [k_s, N] (float32 arrays
    holding bf16-exact values), the exact product p64 [M, N] and the product in granularity
    units (acc, integers) with its certificate sum(|terms|) (absacc)."""

    def __init__(self, a, b, p64, acc, absacc):
        self.a, self.b, self.p64, self.acc, self.absacc = a, b, p64, acc, absacc

    @property
    def v32(self):
        return self.p64.astype(np.float32)

    def full_width(self):
        """Outputs whose exact sum needs all 24 bits: |acc| >= 2^20 units and odd."""
        a = np.abs(self.acc)
        return (a >= 2.0 ** 20) & (np.fmod(a, 2.0) == 1.0)


def max_mag(k_eff):
    """Largest odd integer magnitude m <= 255 with k_eff * m^2 < 2^24."""
    m = min(255, int(math.isqrt((2 ** F32_BITS - 1) // max(1, k_eff))))
    if m % 2 == 0:
        m -= 1
    if m < 1:
        raise ValueError(f"no exactly summable magnitude for {k_eff} unit terms")
    return m


def exact_operands(rng, M, N, ks, shifts=None, emax=0, mag=None, big=True):
    """Exactly summable operands for sum_s A_s[M, k_s] B_s[k_s, N].

    shifts: per segment (sa, sb) exponent shifts, default (0, 0).  emax: the per-row / per-column
    exponents are drawn from [-emax, emax].  mag: integer magnitude bound (default: the largest
    the certificate allows for these k).  big: row 0 of A and column 0 of B are one-signed at
    full magnitude and acc[0, 0] is made odd, so that output needs all 24 bits when the
    certificate allows 2^20 units."""
    ks = list(ks)
    shifts = list(shifts) if shifts is not None else [(0, 0)] * len(ks)
    assert len(shifts) == len(ks)
    wmin = min(sa + sb for sa, sb in shifts)
    w = [2.0 ** (sa + sb - wmin) for sa, sb in shifts]
    k_eff = int(sum(k * wi for k, wi in zip(ks, w)))
    mag = max_mag(k_eff) if mag is None else int(mag)
    ea = rng.integers(-emax, emax + 1, M) if emax else np.zeros(M, np.int64)
    fb = rng.integers(-emax, emax + 1, N) if emax else np.zeros(N, np.int64)
    ms = [rng.integers(-mag, mag + 1, (M, k)).astype(np.float64) for k in ks]
    ns = [rng.integers(-mag, mag + 1, (k, N)).astype(np.float64) for k in ks]
    if big:
        for m_, n_ in zip(ms, ns):
            m_[0, :] = mag
            n_[:, 0] = mag
        fine = w.index(1.0)
        acc00 = sum(wi * float(m_[0] @ n_[:, 0]) for wi, m_, n_ in zip(w, ms, ns))
        if acc00 % 2 == 0 and mag % 2 == 1:
            ns[fine][0, 0] -= 1.0          # changes acc[0, 0] by m[0, 0] = mag (odd)
    absacc = sum(wi * (np.abs(m_) @ np.abs(n_)) for wi, m_, n_ in zip(w, ms, ns))
    if absacc.max() >= 2.0 ** F32_BITS:
        raise AssertionError(f"certificate fails: sum |terms| = {absacc.max()} units >= 2^24")
    acc = sum(wi * (m_ @ n_) for wi, m_, n_ in zip(w, ms, ns))
    scale = np.ldexp(1.0, (ea[:, None] + fb[None, :] + wmin).astype(np.int64))
    p64 = acc * scale
    a = [np.ldexp(m_, (ea + sa)[:, None]).astype(np.float32) for m_, (sa, _) in zip(ms, shifts)]
    b = [np.ldexp(n_, (fb + sb)[None, :]).astype(np.float32) for n_, (_, sb) in zip(ns, shifts)]
    for t in a + b:
        assert np.array_equal(R.bf16_round(t), t), "operand not exact in bf16"
    assert np.array_equal(p64.astype(np.float32).astype(np.float64), p64), "product not fp32"
    return Exact(a, b, p64, acc, absacc)


def fp32_sum_orders(a, b, rng):
    """sum_k a[:, k] b[k, :] accumulated in fp32 in five orders (sequential, reversed, shuffled,
    64-blocked, split into three ranges and the partials summed): a list of [M, N] float32."""
    prod = (a[:, :, None] * b[None, :, :]).astype(np.float32)      # exact: 8 x 8 bits
    K = prod.shape[1]

    def seq(order):
        s = np.zeros((prod.shape[0], prod.shape[2]), np.float32)
        for k in order:
            s = s + prod[:, k]
        return s

    out = [seq(range(K)), seq(range(K - 1, -1, -1)), seq(rng.permutation(K))]
    blocks = [seq(range(k0, min(K, k0 + 64))) for k0 in range(0, K, 64)]
    s = np.zeros_like(blocks[0])
    for blk in blocks:
        s = s + blk
    out.append(s)
    cuts = [0, K // 3, 2 * K // 3, K]
    s = np.zeros_like(blocks[0])
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        s = s + seq(range(lo, hi))
    out.append(s)
    return out


# --------------------------------------------------------------------------- fp32 epilogue
def fma32(a, b, c):
    """fmaf(a, b, c) with one rounding: a * b is exact in fp64; the fp64 sum is rounded to odd
    (TwoSum error decides the sticky bit), which then rounds correctly to fp32."""
    a, b, c = (np.asarray(t, np.float32).astype(np.float64) for t in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    odd = (np.ascontiguousarray(s).view(np.int64) & 1) == 1
    nudge = (err != 0) & ~odd
    s = np.where(nudge, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


ACT_NONE, ACT_SIGMOID, ACT_RELU = 0, 1, 2


def epilogue(v32, alpha=1.0, bias=None, act=0, dact=0, y=None):
    """The epilogue value before the stores: fmaf(v, alpha, bias), act, v *= act'(y).  Sigmoid
    is returned as its fp64 value of the exact pre-activation (the caller holds it to
    sigmoid_bound); everything else is exact fp32."""
    v32 = np.asarray(v32, np.float32)
    b = np.zeros(v32.shape[-1], np.float32) if bias is None else np.asarray(bias, np.float32)
    x = fma32(v32, np.float32(alpha), b[None, :])
    if act == ACT_RELU:
        x = np.maximum(x, np.float32(0))
    elif act == ACT_SIGMOID:
        assert dact == 0, "sigmoid is held to a bound: no act' after it"
        return R.sigmoid64(x.astype(np.float64)), x
    if dact:
        y = np.asarray(y, np.float32)
        if dact == ACT_SIGMOID:
            t = y * (np.float32(1) - y)
        else:
            t = np.where(y > 0, np.float32(1), np.float32(0)).astype(np.float32)
        x = (x * t).astype(np.float32)
    return x, x


def sigmoid_bound(ref64, pre32, ulp):
    """The bound test_bias_act holds 1 / (1 + __expf(-x)) to: __expf's error relative to
    exp(-x) = (1 - s) / s, two roundings, one ulp of the stored type."""
    e = 1.0 - ref64
    return (R.expf_rel_bound(pre32) * e + 3 * R.FP32_U) * ref64 + ulp(ref64) + 2.0 ** -125


def store32(x, prev=None):
    """out32 = v (+ out32 with beta32), one fp32 add."""
    x = np.asarray(x, np.float32)
    return x.copy() if prev is None else (np.asarray(prev, np.float32) + x).astype(np.float32)


def store16(x, prev16=None):
    """out16 = bf16(v (+ float(out16) with beta16)): the add in fp32, then round-to-nearest-even."""
    x = np.asarray(x, np.float32)
    if prev16 is not None:
        x = (np.asarray(prev16, np.float32) + x).astype(np.float32)
    return R.bf16_round(x)


def store16_lo(x):
    """out16_lo = bf16(v - float(bf16(v))) (the subtraction is exact in fp32)."""
    x = np.asarray(x, np.float32)
    return R.bf16_round((x - R.bf16_round(x)).astype(np.float32))


def bf16_ties(x):
    """fp32 values exactly halfway between two bf16 neighbours."""
    bits = np.ascontiguousarray(x, np.float32).view(np.uint32)
    return (bits & 0xFFFF) == 0x8000


# ------------------------------------------------------------------------ dispatch mirror
def instantiations():
    """Every kernel instantiation of the GEMM unit, as canonical names (see kernel_name)."""
    out = set()
    for bn, st in ((256, 4), (128, 6)):
        for a in (0, 1):
            for b in (0, 1):
                for math_ in (0, 1):
                    for cl in (1, 2):
                        out.add(persistent(bn, st, a, b, math_, 4, 0, cl, 0))
    for nf in (0, 1):
        for cl in (1, 2):
            out.add(persistent(256, 3, 1, 1, 0, 8, nf, cl, 0))
            out.add(persistent(256, 4, 1, 1, 0, 8, nf, cl, 1))
    for bn, st in ((256, 2), (128, 3)):
        for a in (0, 1):
            for b in (0, 1):
                out.add(onetile(bn, st, a, b))
    out.add("splitk_finalize_kernel")
    return out


def persistent(*args):
    return "persistent<" + ",".join(str(int(x)) for x in args) + ">"


def onetile(*args):
    return "onetile<" + ",".join(str(int(x)) for x in args) + ">"


_TEMPLATE = re.compile(r"(gemm_tcgen05_persistent_kernel|gemm_tcgen05_kernel)<([^>]*)>")


def kernel_name(demangled):
    """Canonical name of a profiler kernel name, or None if it is not a GEMM-unit kernel."""
    if "splitk_finalize_kernel" in demangled:
        return "splitk_finalize_kernel"
    m = _TEMPLATE.search(demangled)
    if not m:
        return None
    args = []
    for t in m.group(2).split(","):
        t = t.strip()
        t = re.sub(r"^\(\w+\)", "", t)
        args.append({"true": 1, "false": 0}.get(t, None) if t in ("true", "false") else int(t))
    return (persistent if m.group(1) == "gemm_tcgen05_persistent_kernel" else onetile)(*args)


def dispatch(M, N, ks, a_mn, b_mn, *, sms, workspace_elems=0, force_splits=0, force_bn=0,
             math_=False, rms=None, env_persistent_splitk=1, env_rms_nfast=-1):
    """gemm_impl's choices for a descriptor: (kernel names in launch order, splits).
    rms: None, "reg" (row-major state) or "blocked".  workspace_elems = 0: no workspace."""
    bn = force_bn or (256 if N > 128 else 128)
    kbl = [(k + BK - 1) // BK for k in ks]
    total = sum(kbl)
    mt, nt = (M + BM - 1) // BM, (N + bn - 1) // bn
    splits = 1
    if workspace_elems and rms is None:
        want = force_splits
        if want == 0:
            tiles = mt * nt
            if 2 * tiles <= sms and total >= 8:
                want = max(1, (2 * sms) // tiles)
                want = min(want, total // 4)
            else:
                want = 1
        want = min(want, total)
        want = min(want, workspace_elems // (mt * BM * nt * bn))
        if want >= 2:
            splits = want
    kbps = (total + splits - 1) // splits
    splits = (total + kbps - 1) // kbps
    if splits < 2:
        splits = 1
    persistent_ = splits == 1 or env_persistent_splitk != 0
    cluster = 2 if (persistent_ and mt >= 2 and (rms is None or total > 8)) else 1
    if persistent_:
        if bn == 256 and rms is not None and a_mn and b_mn and not math_:
            nfast = env_rms_nfast
            if nfast < 0:
                nfast = 1 if total * BK * N * 2 <= (48 << 20) else 0
            if rms == "blocked":
                return [persistent(256, 4, 1, 1, 0, 8, nfast, cluster, 1)], 1
            return [persistent(256, 3, 1, 1, 0, 8, nfast, cluster, 0)], 1
        st = 4 if bn == 256 else 6
        if splits >= 2:
            return [persistent(bn, st, a_mn, b_mn, 0, 4, 0, cluster, 0), "splitk_finalize_kernel"], splits
        return [persistent(bn, st, a_mn, b_mn, math_, 4, 0, cluster, 0)], 1
    st = 2 if bn == 256 else 3
    return [onetile(bn, st, a_mn, b_mn), "splitk_finalize_kernel"], splits


def coverage_cases():
    """One descriptor per instantiation that dispatch() reaches it with: dicts of dispatch()'s
    arguments (sms = 148-class machine; the choices below do not depend on the SM count
    because no case lets the automatic split decide)."""
    cases = []
    for bn in (128, 256):
        n = 100 if bn == 128 else 300
        for a in (0, 1):
            for b in (0, 1):
                for cl, m in ((1, 100), (2, 300)):
                    for math_ in (False, True):
                        cases.append(dict(M=m, N=n, ks=[200], a_mn=a, b_mn=b, math_=math_))
                    cases.append(dict(M=m, N=n, ks=[200], a_mn=a, b_mn=b, force_splits=2,
                                      workspace_elems=1 << 24, env_persistent_splitk=0))
    for rms in ("reg", "blocked"):
        for nf in (0, 1):
            for cl, (m, k) in ((1, (100, 200)), (2, (300, 600))):
                cases.append(dict(M=m, N=300, ks=[k], a_mn=1, b_mn=1, rms=rms, env_rms_nfast=nf))
    return cases
