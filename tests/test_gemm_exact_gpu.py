"""cc_gemm bit for bit: exactly summable operands (tests/gemm_ref.py) on every dispatch path,
operand orientation, edge shape and epilogue output.

The operands are bf16 integers times a power of two per row of A and per column of B, sized so
that every partial sum of an output fits fp32's 24-bit significand.  fp32 accumulation is then
exact in any order, however the kernel tiles, splits, clusters or orders the reduction, and the
epilogue is one IEEE operation after another on exact inputs: every output must equal the numpy
emulation bit for bit (zeros compared by value).  Sigmoid (__expf) is the one step held to a
bound, and the fused RMSprop update is held to fp64 within test_rmsprop's bounds.

Every operand and output is a view into a flat buffer pre-filled with a NaN sentinel, with
sentinel rows after the operand's last row: a read of operand padding turns outputs into NaN,
and everything outside each output view must still hold the sentinel afterwards.  Each call's
launch count is checked against the dispatch mirror, and one test sees every one of the 49
kernel instantiations run under the profiler."""
import ctypes as C

import numpy as np
import pytest
import torch

import gemm_ref as G
import tail_ref as R

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32
SENTINEL = {BF16: (torch.int16, 0x7FC1), F32: (torch.int32, 0x7FC0DEAD)}
LR, RHO, MOM, EPS = 0.0075, 0.85, 0.1, 1e-7


@pytest.fixture(scope="module")
def lib():
    from cellcomm_b200 import _lib
    return _lib


_SMS = []


def sms():
    if not _SMS:
        _SMS.append(torch.cuda.get_device_properties(0).multi_processor_count)
    return _SMS[0]


def rup(x, m):
    return (x + m - 1) // m * m


class Mat:
    """[rows, cols] view with leading dimension ld at element offset off inside a flat
    sentinel-filled device buffer with `extra` sentinel rows after the last one."""

    def __init__(self, rows, cols, dtype, ld=None, off=0, extra=0, data=None):
        self.rows, self.cols, self.dtype = rows, cols, dtype
        self.ld = ld if ld is not None else rup(cols, 8 if dtype == BF16 else 4)
        self.off = off
        n = off + (rows + extra) * self.ld + 16
        idt, self.pat = SENTINEL[dtype]
        self.raw = torch.full((n,), self.pat, dtype=idt, device="cuda")
        self.t = torch.as_strided(self.raw.view(dtype), (rows, cols), (self.ld, 1), off)
        if data is not None:
            self.set(data)

    def set(self, data):
        self.t.copy_(torch.from_numpy(np.ascontiguousarray(data, np.float32)).to(self.dtype))

    @property
    def ptr(self):
        return self.t.data_ptr()

    def get(self):
        return self.t.float().cpu().numpy()

    def bits(self):
        return self.t.contiguous().view(SENTINEL[self.dtype][0]).cpu().numpy()

    def check_sentinel(self, what, cols=None):
        """Everything outside the view (or outside its first `cols` columns) holds the sentinel."""
        raw = self.raw.cpu().numpy()
        inside = np.zeros(raw.shape[0], bool)
        idx = self.off + np.add.outer(np.arange(self.rows, dtype=np.int64) * self.ld,
                                      np.arange(self.cols if cols is None else cols, dtype=np.int64))
        inside[idx.ravel()] = True
        bad = np.count_nonzero(raw[~inside] != np.array(self.pat).astype(raw.dtype))
        assert bad == 0, f"{what}: {bad} elements outside the view were written"


def assert_exact(got, want, what):
    """Equal values (so -0.0 == +0.0; NaN never matches)."""
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    bad = ~(got == want)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {bad.sum()} of {bad.size} differ, first at {i}: "
                             f"got {got[i]!r}, want {want[i]!r}")


def assert_within(got, ref, tol, what):
    err = np.abs(np.asarray(got, np.float64) - ref)
    bad = ~(err <= tol)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {bad.sum()} of {bad.size} outside the bound, first at {i}: "
                             f"got {got[i]!r}, want {ref[i]!r}, err {err[i]:.3g} > "
                             f"{np.broadcast_to(tol, err.shape)[i]:.3g}")


def operands(ex, a_mn, b_mn, lay=(0, 0), extra=64):
    """Device operands of Exact `ex`: A stored [M, k] (a_mn = 0) or [k, M]; B stored [N, k]
    (b_mn = 0) or [k, N].  lay = (extra ld, base offset) in elements."""
    As, Bs = [], []
    for a, b in zip(ex.a, ex.b):
        sa = a.T if a_mn else a
        sb = b if b_mn else b.T
        As.append(Mat(sa.shape[0], sa.shape[1], BF16, rup(sa.shape[1], 8) + lay[0], lay[1], extra, sa))
        Bs.append(Mat(sb.shape[0], sb.shape[1], BF16, rup(sb.shape[1], 8) + lay[0], lay[1], extra, sb))
    return As, Bs


class Ws:
    def __init__(self, elems):
        self.t = torch.empty(max(1, elems), dtype=F32, device="cuda")
        self.elems = elems


_WS = []


def full_ws():
    if not _WS:
        _WS.append(Ws(296 * 128 * 256 * 2))
    return _WS[0]


def desc(lib, M, N, As, Bs, ks, a_mn, b_mn, *, alpha=1.0, bias=None, act=0, dact_y=None, dact=0,
         out32=None, beta32=0, out16=None, beta16=0, lo=None, ws=None, splits=0, bn=0):
    d = lib.GemmDesc()
    d.M, d.N, d.a_mn_major, d.b_mn_major, d.nseg = M, N, a_mn, b_mn, len(As)
    for s, (a, b, k) in enumerate(zip(As, Bs, ks)):
        d.a[s], d.lda[s], d.b[s], d.ldb[s], d.k[s] = a.ptr, a.ld, b.ptr, b.ld, k
    d.alpha, d.act = alpha, act
    d.bias = None if bias is None else bias.data_ptr()
    if dact_y is not None:
        d.dact_y, d.ld_dact, d.dact = dact_y.ptr, dact_y.ld, dact
    if out32 is not None:
        d.out32, d.ld32, d.beta32 = out32.ptr, out32.ld, beta32
    if out16 is not None:
        d.out16, d.ld16, d.beta16 = out16.ptr, out16.ld, beta16
    if lo is not None:
        d.out16_lo, d.ld16_lo = lo.ptr, lo.ld
    if ws is not None:
        d.workspace, d.workspace_elems = ws.t.data_ptr(), ws.elems
    d.force_splits, d.force_bn = splits, bn
    return d


def launch(lib, d, expect=None, what=""):
    """cc_gemm on the current stream; with `expect` (dispatch() kwargs) the launch count must
    match the mirror's."""
    from cellcomm_b200 import ops
    n0 = ops.launch_count()
    lib.check(lib.load().cc_gemm(C.byref(d), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    got = ops.launch_count() - n0
    if expect is not None:
        names, _ = G.dispatch(sms=sms(), **expect)
        assert got == len(names), f"{what}: {got} launches, the mirror says {names}"
    return got


# ============================================================ 1. orientation x edge shapes
ORIENT = [(0, 1), (0, 0), (1, 1), (1, 0)]
EDGE = [(1, 1, 1), (8, 63, 65), (63, 8, 64), (64, 65, 127), (65, 127, 128), (127, 128, 129),
        (128, 129, 8), (129, 257, 63), (257, 64, 257), (383, 300, 200), (383, 1, 3369),
        (1, 3369, 383)]
LAYS = [(0, 0), (8, 0), (0, 8), (8, 8)]


@pytest.mark.parametrize("a_mn,b_mn", ORIENT)
def test_orientation_edges(lib, a_mn, b_mn):
    """Every operand-major combination at M, N, K from 1 to 3369 (tile edges 63 / 64 / 65, 127 /
    128 / 129, 257; M = 383 is three row tiles, so the last CTA pair has an idle second CTA),
    operand ld of round_up(inner, 8) and + 8, bases 0 and 8 elements (a column slice), per-row
    and per-column exponents over +-20, and sentinel rows after every operand."""
    rng = np.random.default_rng(10 + 2 * a_mn + b_mn)
    for i, (M, N, K) in enumerate(EDGE):
        lay = LAYS[i % 4]
        what = f"({a_mn},{b_mn}) {M}x{N}x{K} lay {lay}"
        ex = G.exact_operands(rng, M, N, [K], emax=20)
        As, Bs = operands(ex, a_mn, b_mn, lay)
        o32 = Mat(M, N, F32, rup(N, 4) + 4 * (i % 2))
        o16 = Mat(M, N, BF16) if i % 3 == 0 else None
        launch(lib, desc(lib, M, N, As, Bs, [K], a_mn, b_mn, out32=o32, out16=o16),
               dict(M=M, N=N, ks=[K], a_mn=a_mn, b_mn=b_mn), what)
        assert_exact(o32.get(), ex.v32, what)
        o32.check_sentinel(what)
        if o16 is not None:
            assert_exact(o16.get(), G.store16(ex.v32), what + " out16")
            o16.check_sentinel(what + " out16")
        if K >= 64:
            assert ex.full_width()[0, 0]


# ======================================================================== 2. tile width / cluster
@pytest.mark.parametrize("bn_eff", [128, 160, 192, 224, 256])
def test_tile_width(lib, bn_eff, monkeypatch):
    """CC_GEMM_BN_EFF at every effective width, cluster 1 (one row tile) and 2, with bias, ReLU,
    out32 and out16."""
    monkeypatch.setenv("CC_GEMM_BN_EFF", str(bn_eff))
    rng = np.random.default_rng(bn_eff)
    for M, (a_mn, b_mn) in ((300, (0, 1)), (100, (1, 0)), (300, (0, 0)), (257, (1, 1))):
        N, K = 1000, 200
        what = f"bn_eff {bn_eff} M {M} ({a_mn},{b_mn})"
        ex = G.exact_operands(rng, M, N, [K], emax=3)
        As, Bs = operands(ex, a_mn, b_mn)
        bias = (rng.integers(-64, 64, N) * 2.0 ** -3).astype(np.float32)
        o32, o16 = Mat(M, N, F32), Mat(M, N, BF16)
        launch(lib, desc(lib, M, N, As, Bs, [K], a_mn, b_mn, bias=torch.from_numpy(bias).cuda(),
                         act=2, out32=o32, out16=o16),
               dict(M=M, N=N, ks=[K], a_mn=a_mn, b_mn=b_mn, math_=True), what)
        x, _ = G.epilogue(ex.v32, bias=bias, act=2)
        assert_exact(o32.get(), x, what)
        assert_exact(o16.get(), G.store16(x), what + " out16")
        o32.check_sentinel(what)
        o16.check_sentinel(what)


def test_tile_width_auto_and_forced_128(lib, monkeypatch):
    """The automatic width (N = 3369 at M = 2048) and bn = 128 forced at N = 300 with epilogue
    math and out16 + out16_lo."""
    rng = np.random.default_rng(7)
    M, N, K = 2048, 3369, 320
    ex = G.exact_operands(rng, M, N, [K], emax=6)
    As, Bs = operands(ex, 0, 1)
    for forced in ("0", "256"):
        monkeypatch.setenv("CC_GEMM_BN_EFF", forced)
        o32 = Mat(M, N, F32)
        launch(lib, desc(lib, M, N, As, Bs, [K], 0, 1, out32=o32),
               dict(M=M, N=N, ks=[K], a_mn=0, b_mn=1), f"bn_eff {forced}")
        assert_exact(o32.get(), ex.v32, f"bn_eff {forced}")
        o32.check_sentinel(f"bn_eff {forced}")
    monkeypatch.setenv("CC_GEMM_BN_EFF", "0")
    M, N, K = 300, 300, 200
    ex = G.exact_operands(rng, M, N, [K], mag=40)
    As, Bs = operands(ex, 0, 1)
    bias = (rng.integers(-1000, 1000, N) * 0.5).astype(np.float32)
    o32, o16, lo = Mat(M, N, F32), Mat(M, N, BF16), Mat(M, N, BF16)
    launch(lib, desc(lib, M, N, As, Bs, [K], 0, 1, bias=torch.from_numpy(bias).cuda(), act=2,
                     out32=o32, out16=o16, lo=lo, bn=128),
           dict(M=M, N=N, ks=[K], a_mn=0, b_mn=1, force_bn=128, math_=True), "bn 128")
    x, _ = G.epilogue(ex.v32, bias=bias, act=2)
    assert_exact(o32.get(), x, "bn 128 out32")
    assert_exact(o16.get(), G.store16(x), "bn 128 out16")
    assert_exact(lo.get(), G.store16_lo(x), "bn 128 lo")
    assert G.bf16_ties(x).any() and (G.store16_lo(x) != 0).any()
    for m in (o32, o16, lo):
        m.check_sentinel("bn 128")


# =============================================================================== 3. split-K
SPLITK = [
    (128, 300, (4000,), 2), (128, 300, (4000,), 3), (128, 300, (4000,), 7),
    (300, 100, (700, 1300), 6),                  # a segment boundary inside a k-range
    (257, 260, (128, 128, 128, 128), 4),         # every k-range starts on a segment boundary
    (130, 257, (64, 64, 640), 12),               # more k-ranges than a segment has k-blocks
    (130, 257, (320, 64, 640), 16),
]


@pytest.mark.parametrize("persistent", ["1", "0"])
@pytest.mark.parametrize("a_mn,b_mn", ORIENT)
def test_split_k(lib, persistent, a_mn, b_mn, monkeypatch):
    """Forced splits of 2, 3, 7 and more than one segment's k-blocks, up to 4 segments, in the
    persistent kernel (CC_GEMM_PERSISTENT_SPLITK=1) and the one-tile-per-CTA kernel (=0), with
    bias + ReLU applied by the finalize pass."""
    monkeypatch.setenv("CC_GEMM_PERSISTENT_SPLITK", persistent)
    rng = np.random.default_rng(30 + 4 * a_mn + 2 * b_mn + int(persistent))
    for M, N, ks, splits in SPLITK:
        what = f"{M}x{N} ks {ks} splits {splits} ({a_mn},{b_mn}) persistent {persistent}"
        ex = G.exact_operands(rng, M, N, ks, emax=4)
        As, Bs = operands(ex, a_mn, b_mn, LAYS[splits % 4])
        bias = (rng.integers(-64, 64, N) * 2.0 ** -2).astype(np.float32)
        o32, o16 = Mat(M, N, F32), Mat(M, N, BF16)
        n = launch(lib, desc(lib, M, N, As, Bs, list(ks), a_mn, b_mn, bias=torch.from_numpy(bias).cuda(),
                             act=2, out32=o32, out16=o16, ws=full_ws(), splits=splits),
                   dict(M=M, N=N, ks=list(ks), a_mn=a_mn, b_mn=b_mn, math_=True, force_splits=splits,
                        workspace_elems=full_ws().elems, env_persistent_splitk=int(persistent)), what)
        assert n == 2, what
        x, _ = G.epilogue(ex.v32, bias=bias, act=2)
        assert_exact(o32.get(), x, what)
        assert_exact(o16.get(), G.store16(x), what + " out16")
        o32.check_sentinel(what)
        o16.check_sentinel(what)


def test_split_k_auto_and_workspace_cap(lib):
    """The automatic split at M = 128, K = 33694 (full-width sums), a workspace that caps the
    split count, and one too small for any split."""
    rng = np.random.default_rng(40)
    M, N, K = 128, 512, 33694
    ex = G.exact_operands(rng, M, N, [K])
    assert ex.full_width()[0, 0]
    As, Bs = operands(ex, 0, 1)
    o32 = Mat(M, N, F32)
    n = launch(lib, desc(lib, M, N, As, Bs, [K], 0, 1, out32=o32, ws=full_ws()),
               dict(M=M, N=N, ks=[K], a_mn=0, b_mn=1, workspace_elems=full_ws().elems), "auto")
    assert n == 2
    assert_exact(o32.get(), ex.v32, "auto split")
    o32.check_sentinel("auto split")
    M, N, K = 200, 300, 4000
    ex = G.exact_operands(rng, M, N, [K], emax=2)
    As, Bs = operands(ex, 0, 0)
    tile = 256 * 512
    for elems, want in ((3 * tile + 5, 2), (2 * tile - 1, 1)):
        ws = Ws(elems)
        o32 = Mat(M, N, F32)
        n = launch(lib, desc(lib, M, N, As, Bs, [K], 0, 0, out32=o32, ws=ws, splits=7),
                   dict(M=M, N=N, ks=[K], a_mn=0, b_mn=0, force_splits=7, workspace_elems=elems),
                   f"ws {elems}")
        assert n == want
        _, s = G.dispatch(M, N, [K], 0, 0, sms=sms(), force_splits=7, workspace_elems=elems)
        assert s == (3 if want == 2 else 1)
        assert_exact(o32.get(), ex.v32, f"ws {elems}")
        o32.check_sentinel(f"ws {elems}")


# ================================================================ 4. hi + lo as the engine issues
HILO = [(0, 0), (-8, 0), (0, -8)]


def _lo_matters(ex, want_fn):
    """The expected result without the low-order segments differs from the full one."""
    hi = ex.a[0].astype(np.float64) @ ex.b[0].astype(np.float64)
    return not np.array_equal(want_fn(hi.astype(np.float32)), want_fn(ex.v32))


@pytest.mark.parametrize("M", [1, 130, 2048])
def test_hi_lo_forward(lib, M):
    """Net.forward on a split activation: x_hi W + x_lo W + x_hi W_lo (A K-major, B MN-major)
    into out32 with bias + ReLU, plus the output's own hi (out16) and lo (out16_lo) terms, from
    [:rows] views of buffers whose further rows hold other data."""
    rng = np.random.default_rng(50 + M)
    N, K = 300, 517
    ex = G.exact_operands(rng, M, N, [K] * 3, HILO, emax=2)
    As, Bs = operands(ex, 0, 1, extra=129)
    bias = (rng.integers(-99, 99, N) * 2.0 ** -1).astype(np.float32)
    o32, o16, lo = Mat(M, N, F32), Mat(M, N, BF16), Mat(M, N, BF16)
    ws = None if M == 130 else full_ws()       # 130: the persistent kernel unsplit
    launch(lib, desc(lib, M, N, As, Bs, [K] * 3, 0, 1, bias=torch.from_numpy(bias).cuda(), act=2,
                     out32=o32, out16=o16, lo=lo, ws=ws),
           dict(M=M, N=N, ks=[K] * 3, a_mn=0, b_mn=1, math_=True,
                workspace_elems=ws.elems if ws else 0), "fwd")
    x, _ = G.epilogue(ex.v32, bias=bias, act=2)
    assert_exact(o32.get(), x, "fwd out32")
    assert_exact(o16.get(), G.store16(x), "fwd out16")
    assert_exact(lo.get(), G.store16_lo(x), "fwd lo")
    assert _lo_matters(ex, lambda v: G.epilogue(v, bias=bias, act=2)[0])
    for m in (o32, o16, lo):
        m.check_sentinel("fwd")


@pytest.mark.parametrize("M", [64, 300])
def test_hi_lo_dgrad_beta32(lib, M):
    """dgrad into the fp32 gradient: dz_hi W^T + dz_lo W^T + dz_hi W_lo^T (both K-major) with
    beta32 onto existing values, then a second call with beta32 onto the first's result."""
    rng = np.random.default_rng(60 + M)
    N, K = 1000, 257                  # gradient [M, N] of an input width N; reduction over K
    o32 = Mat(M, N, F32)
    prev = (rng.integers(-2 ** 12, 2 ** 12, (M, N)) * 2.0 ** -6).astype(np.float32)
    o32.set(prev)
    want = prev
    for call in range(2):
        ex = G.exact_operands(rng, M, N, [K] * 3, HILO, emax=1)
        As, Bs = operands(ex, 0, 0, LAYS[call + 1])
        launch(lib, desc(lib, M, N, As, Bs, [K] * 3, 0, 0, out32=o32, beta32=1, ws=full_ws()),
               dict(M=M, N=N, ks=[K] * 3, a_mn=0, b_mn=0, workspace_elems=full_ws().elems), "dgrad")
        new = G.store32(ex.v32, want)
        assert _lo_matters(ex, lambda v: G.store32(v, want))
        want = new
        assert_exact(o32.get(), want, f"dgrad call {call}")
    o32.check_sentinel("dgrad")


@pytest.mark.parametrize("M,B", [(300, 1000), (100, 128)])
def test_hi_lo_wgrad(lib, M, B):
    """wgrad's three cross terms x_hi dz_hi + x_lo dz_hi + x_hi dz_lo (both MN-major)."""
    rng = np.random.default_rng(70 + M)
    N = 200
    ex = G.exact_operands(rng, M, N, [B] * 3, HILO, emax=3)
    As, Bs = operands(ex, 1, 1, extra=64)
    o32 = Mat(M, N, F32)
    launch(lib, desc(lib, M, N, As, Bs, [B] * 3, 1, 1, out32=o32, ws=full_ws()),
           dict(M=M, N=N, ks=[B] * 3, a_mn=1, b_mn=1, workspace_elems=full_ws().elems), "wgrad")
    assert_exact(o32.get(), ex.v32, "wgrad")
    assert _lo_matters(ex, lambda v: v)
    o32.check_sentinel("wgrad")


# ================================================================================ 5. epilogue
def out_geometry(cols, layout, dtype):
    pad = max(64, rup(cols, 64))
    if layout == "odd":
        return cols | 1, 0
    if layout == "ld4":
        ld = rup(cols, 4)
        return (ld + 4 if ld % 8 == 0 else ld), 0
    return pad, {"pad": 0, "off1": 1, "off3": 3}[layout]


# (alpha, bias: None / "al" / "off", act, act', outputs, output layout)
EPI = [
    (1.0, None, 0, 0, "32", "pad"),
    (1.0, "al", 2, 0, "32+16", "odd"),
    (0.5, None, 0, 0, "16", "ld4"),
    (0.3, None, 0, 1, "32", "off1"),
    (0.3, "off", 0, 0, "32+16", "off3"),
    (0.3, "al", 2, 2, "32+16", "ld4"),
    (1.0, "off", 2, 0, "16+lo", "pad"),
    (1.0, None, 0, 0, "16+lo", "off1"),
    (1.0, "al", 0, 0, "16+lo", "odd"),
    (1.0, None, 0, 2, "beta32", "odd"),
    (1.0, "al", 0, 1, "beta32", "off3"),
    (0.5, None, 0, 1, "beta16", "pad"),
    (0.5, "off", 0, 0, "beta16", "odd"),
    (1.0, "al", 1, 0, "32+16", "pad"),
    (1.0, "off", 1, 0, "32+16", "off1"),
    (0.5, None, 1, 0, "32", "odd"),
]
PATHS = [("persistent", "1", False), ("persistent split-K", "1", True), ("one-tile split-K", "0", True)]


@pytest.mark.parametrize("case", range(len(EPI)))
def test_epilogue(lib, case, monkeypatch):
    """Every epilogue step and output through the persistent unsplit kernel, persistent split-K
    (finalize pass) and one-tile split-K: all three equal the emulation, so each other."""
    alpha, bmode, act, dact, outs, layout = EPI[case]
    rng = np.random.default_rng(80 + case)
    M, N = ((131, 75), (257, 300))[case % 2]
    K = 330
    ex = G.exact_operands(rng, M, N, [K], [(-6, -6)], mag=31)
    As, Bs = operands(ex, 0, 1 - case % 2)
    bias = braw = None
    if bmode is not None:
        b = (rng.integers(-2 ** 10, 2 ** 10, N) * 2.0 ** -7).astype(np.float32)
        off = 1 if bmode == "off" else 0
        braw = torch.full((N + 8,), float("nan"), device="cuda")
        bias = braw[off:off + N]
        bias.copy_(torch.from_numpy(b))
    y = ydev = None
    if dact:
        choice = np.array([0.0, -0.0, 1.0, -0.5, -2.0, 0.25, 0.75, 0.5, 2.0 ** -9, 1 - 2.0 ** -8], np.float32)
        y = choice[rng.integers(0, len(choice), (M, N))]
        u = R.bf16_round(rng.random((M, N)).astype(np.float32))
        y = np.where(rng.random((M, N)) < 0.5, y, u).astype(np.float32)
        ydev = Mat(M, N, BF16, *out_geometry(N, layout, BF16), data=y)
    x, pre = G.epilogue(ex.v32, alpha=alpha, bias=None if bias is None else b, act=act, dact=dact, y=y)
    prev32 = (rng.integers(-2 ** 16, 2 ** 16, (M, N)) * 2.0 ** -8).astype(np.float32)
    prev16 = R.bf16_round((rng.integers(-255, 255, (M, N)) * 2.0 ** -3).astype(np.float32))
    if act != 1 and alpha != 0.3 and dact != 1:
        assert G.bf16_ties(x).any(), "the case must pin round-half-even"
    for name, mode, split in PATHS:
        monkeypatch.setenv("CC_GEMM_PERSISTENT_SPLITK", mode)
        what = f"case {case} {name}"
        ld, off = out_geometry(N, layout, F32)
        o32 = Mat(M, N, F32, ld, off) if outs in ("32", "32+16", "beta32") else None
        ld, off = out_geometry(N, layout, BF16)
        o16 = Mat(M, N, BF16, ld, off) if outs in ("16", "32+16", "16+lo", "beta16") else None
        lo = Mat(M, N, BF16, ld, off) if outs == "16+lo" else None
        if outs == "beta32":
            o32.set(prev32)
        if outs == "beta16":
            o16.set(prev16)
        ws = full_ws() if split else None
        math_ = alpha != 1.0 or bias is not None or act != 0 or dact != 0
        launch(lib, desc(lib, M, N, As, Bs, [K], 0, 1 - case % 2, alpha=alpha, bias=bias, act=act,
                         dact_y=ydev, dact=dact, out32=o32, beta32=int(outs == "beta32"), out16=o16,
                         beta16=int(outs == "beta16"), lo=lo, ws=ws, splits=3 if split else 0),
               dict(M=M, N=N, ks=[K], a_mn=0, b_mn=1 - case % 2, math_=math_,
                    workspace_elems=ws.elems if ws else 0, force_splits=3 if split else 0,
                    env_persistent_splitk=int(mode)), what)
        if act == 1:
            if o32 is not None:
                assert_within(o32.get(), x, G.sigmoid_bound(x, pre, R.ulp32), what + " out32")
            if o16 is not None:
                assert_within(o16.get(), x, G.sigmoid_bound(x, pre, R.ulp16), what + " out16")
        else:
            if o32 is not None:
                assert_exact(o32.get(), G.store32(x, prev32 if outs == "beta32" else None), what + " out32")
            if o16 is not None:
                assert_exact(o16.get(), G.store16(x, prev16 if outs == "beta16" else None), what + " out16")
            if lo is not None:
                assert_exact(lo.get(), G.store16_lo(x), what + " lo")
        for m in (o32, o16, lo):
            if m is not None:
                m.check_sentinel(what)
    if braw is not None:
        assert torch.isnan(braw[:1 if bmode == "off" else 0]).all() and torch.isnan(braw[N + (bmode == "off"):]).all()


# ========================================================================== 6. fused RMSprop
def _rms_check(got_w, got_s, got_m, w0, s0, m0, g, what):
    w, s, m = R.rmsprop64(w0.astype(np.float64), g.astype(np.float64), s0.astype(np.float64),
                          m0.astype(np.float64), *(float(np.float32(v)) for v in (LR, RHO, MOM, EPS)))
    lr, mo, eps = float(np.float32(LR)), float(np.float32(MOM)), float(np.float32(EPS))
    mom_abs = mo * np.abs(m0) + lr * np.abs(g) / np.sqrt(s + eps)
    assert_within(got_s, s, 1e-5 * s, what + " ms")
    assert_within(got_m, m, 1e-5 * mom_abs, what + " mom")
    assert_within(got_w, w, 1e-5 * np.abs(w) + 1e-5 * mom_abs, what + " w")


def _grad_operands(rng, M, N, B):
    """Gradient-sized exact operands: |g| from about 1e-5 to 1e-1 with exact zeros."""
    ex = G.exact_operands(rng, M, N, [B], [(-10, -10)], emax=3, mag=min(15, G.max_mag(B)))
    return ex


def _state(rng, M, N):
    w0 = (rng.standard_normal((M, N)) * 0.05).astype(np.float32)
    s0 = (rng.random((M, N)) * 1e-4).astype(np.float32)
    s0.reshape(-1)[::13] = 0.0
    m0 = (rng.standard_normal((M, N)) * 1e-3).astype(np.float32)
    return w0, s0, m0


@pytest.mark.parametrize("nfast", ["0", "1"])
def test_fused_rmsprop_register(lib, nfast, monkeypatch):
    """The row-major register path on both rasters: cluster 1 and 2, the vector state path
    (ld % 4 == 0) and the scalar one (ld % 4 == 2, ragged N), with and without the bf16 copy
    and the gradient output; p16 == bf16(p32) bit for bit; state padding untouched."""
    monkeypatch.setenv("CC_GEMM_RMS_NFAST", nfast)
    rng = np.random.default_rng(90 + int(nfast))
    for M, N, B, ldx, with16, grad in ((300, 300, 600, 0, True, True), (100, 301, 200, 1, True, False),
                                       (257, 1000, 96, 0, False, True), (300, 257, 640, 1, True, True)):
        what = f"rms {M}x{N} B {B} ld+{ldx} nfast {nfast}"
        ex = _grad_operands(rng, M, N, B)
        As, Bs = operands(ex, 1, 1)
        w0, s0, m0 = _state(rng, M, N)
        ld = rup(N, 64) + 2 * ldx if ldx else rup(N, 64)
        pw, ps, pm = (Mat(M, N, F32, ld, data=t) for t in (w0, s0, m0))
        p16 = Mat(M, N, BF16, ld) if with16 else None
        o32 = Mat(M, N, F32) if grad else None
        d = desc(lib, M, N, As, Bs, [B], 1, 1, out32=o32)
        d.rms_p32, d.rms_ms, d.rms_mom = pw.ptr, ps.ptr, pm.ptr
        d.rms_p16 = None if p16 is None else p16.ptr
        d.rms_ld = ld
        d.rms_lr, d.rms_rho, d.rms_momentum, d.rms_eps = LR, RHO, MOM, EPS
        launch(lib, d, dict(M=M, N=N, ks=[B], a_mn=1, b_mn=1, rms="reg", env_rms_nfast=int(nfast)), what)
        g = ex.v32
        assert np.abs(g).max() > 1e-3
        _rms_check(pw.get(), ps.get(), pm.get(), w0, s0, m0, g, what)
        if p16 is not None:
            assert np.array_equal(p16.bits().view(np.uint16), R.bf16_bits(pw.get())), what + " p16"
        if o32 is not None:
            assert_exact(o32.get(), g, what + " grad")
        for m in (pw, ps, pm, p16, o32):
            if m is not None:
                m.check_sentinel(what)


@pytest.mark.parametrize("nfast", ["0", "1"])
@pytest.mark.parametrize("row0", [0, 33, 64])
def test_fused_rmsprop_blocked(lib, row0, nfast, monkeypatch):
    """The blocked-state path at cluster 1 (batch 200) and cluster 2 (batch 640: more than 8
    k-blocks, two row tiles) with this GEMM's first layer row at 0, 33 and 64: the state equals
    fp64 RMSprop, p16 and lo are bf16(p32) and bf16(p32 - bf16(p32)) bit for bit, the bf16
    copies are written in whole 32-column chunks (bf16(0) between N and the chunk edge, the
    sentinel beyond), and the layer's other rows and padding state do not change."""
    from cellcomm_b200 import ops
    monkeypatch.setenv("CC_GEMM_RMS_NFAST", nfast)
    rng = np.random.default_rng(100 + row0 + int(nfast))
    for M, N, B in ((100, 300, 200), (300, 257, 640)):
        what = f"blocked {M}x{N} B {B} row0 {row0} nfast {nfast}"
        ex = _grad_operands(rng, M, N, B)
        As, Bs = operands(ex, 1, 1)
        Rr, ld = rup(row0 + M + 5, 32), rup(N, 64)
        w0, s0, m0 = (np.zeros((Rr, ld), np.float32) for _ in range(3))
        for full in (w0, s0, m0):
            st = _state(rng, Rr, N)
            full[:, :N] = st[0] if full is w0 else (np.abs(st[1]) if full is s0 else st[2])
        blk = [ops.state_rows_to_blocked(torch.from_numpy(t).cuda()).contiguous() for t in (w0, s0, m0)]
        p16, lo, o32 = Mat(M, N, BF16, ld), Mat(M, N, BF16, ld), Mat(M, N, F32, ld)
        d = desc(lib, M, N, As, Bs, [B], 1, 1, out32=o32)
        d.rms_p32, d.rms_ms, d.rms_mom = (t.data_ptr() for t in blk)
        d.rms_p16, d.rms_p16_lo, d.rms_ld, d.rms_blocked, d.rms_row0 = p16.ptr, lo.ptr, ld, 1, row0
        d.rms_lr, d.rms_rho, d.rms_momentum, d.rms_eps = LR, RHO, MOM, EPS
        launch(lib, d, dict(M=M, N=N, ks=[B], a_mn=1, b_mn=1, rms="blocked", env_rms_nfast=int(nfast)), what)
        got = [ops.state_blocked_to_rows(t, Rr, ld).cpu().numpy() for t in blk]
        g = ex.v32
        rs = slice(row0, row0 + M)
        _rms_check(got[0][rs, :N], got[1][rs, :N], got[2][rs, :N], w0[rs, :N], s0[rs, :N], m0[rs, :N], g, what)
        for t_got, t0, name in zip(got, (w0, s0, m0), "wsm"):
            keep = np.ones(t0.shape, bool)
            keep[rs, :N] = False
            assert np.array_equal(t_got[keep], t0[keep]), f"{what}: state {name} outside the block changed"
        edge = min(ld, rup(N, 32))
        wn = got[0][rs, :N]
        assert np.array_equal(p16.bits()[:, :N].view(np.uint16), R.bf16_bits(wn)), what + " p16"
        want_lo = R.bf16_bits((wn - R.bf16_round(wn)).astype(np.float32))
        assert np.array_equal(lo.bits()[:, :N].view(np.uint16), want_lo), what + " lo"
        assert_exact(o32.get(), g, what + " grad")
        for m in (p16, lo, o32):
            full = torch.as_strided(m.raw.view(m.dtype), (M, ld), (ld, 1), 0).float().cpu().numpy()
            assert np.all(full[:, N:edge] == 0), what + " chunk padding"
            m.check_sentinel(what, cols=edge)


# ============================================================================ 7. routed output
ROUTE = [(2, 0, "pad", "row"), (3, 4, "pad", "mid"), (4, 1028, "odd", "mid"), (3, 0, "odd", "row"),
         (2, 1028, "pad", "mid"), (4, 4, "odd", "row")]


@pytest.mark.parametrize("world,off0,ldm,boundary", ROUTE)
def test_routed_output(lib, world, off0, ldm, boundary):
    """The routed wgrad output on one device: element rel = route_off0 + r ld32 + c goes to
    route_base[min(rel / shard, world - 1)] + rel.  Each owner's slot holds exact bits, the
    sentinel everywhere else; ld32 % 4 == 0 takes the float4 path, ld32 % 4 != 0 the scalar one;
    shard boundaries fall inside a row or at a row start."""
    rng = np.random.default_rng(110 + world + off0)
    M, N, K = 300, 200, 192
    ld = rup(N, 64) if ldm == "pad" else N + 1
    total = off0 + M * ld
    base = rup(total // world, 8)
    if boundary == "row":   # shard - off0 is a multiple of ld and shard a multiple of 8
        shard = next(s for s in range(base - 8 * ld, base + 8 * ld)
                     if s > off0 and s % 8 == 0 and (s - off0) % ld == 0 and s * (world - 1) < total)
    else:
        shard = base + (8 if (base - off0) % ld == 0 else 0)
        assert (shard - off0) % ld != 0
    ex = G.exact_operands(rng, M, N, [K], emax=4)
    As, Bs = operands(ex, 1, 1)
    stage = [Mat(1, total + 64, F32) for _ in range(world)]
    local = torch.as_strided(stage[0].raw.view(F32), (M, N), (ld, 1), off0)
    d = desc(lib, M, N, As, Bs, [K], 1, 1)
    d.out32, d.ld32 = local.data_ptr(), ld
    d.route_world, d.route_shard, d.route_off0 = world, shard, off0
    for q in range(world):
        d.route_base[q] = stage[q].ptr
    launch(lib, d, dict(M=M, N=N, ks=[K], a_mn=1, b_mn=1), "route")
    rel = off0 + np.add.outer(np.arange(M) * ld, np.arange(N))
    owner = np.minimum(rel // shard, world - 1)
    assert len(np.unique(owner)) == world
    pat = np.uint32(SENTINEL[F32][1] & 0xFFFFFFFF)
    for q in range(world):
        raw = stage[q].raw.cpu().numpy().view(np.uint32)
        mine = owner == q
        assert_exact(raw[rel[mine]].view(np.float32), ex.v32[mine], f"owner {q}")
        written = np.zeros(raw.shape[0], bool)
        written[rel[mine]] = True
        assert np.all(raw[~written] == pat), f"owner {q}: written outside its share"


# ====================================================================== 8. rejected descriptors
def test_rejected_descriptors(lib):
    """Each invalid descriptor raises CCError before any launch and leaves every output at its
    sentinel."""
    from cellcomm_b200 import ops
    rng = np.random.default_rng(120)
    M, N, K = 130, 300, 200
    ex = G.exact_operands(rng, M, N, [K])
    As, Bs = operands(ex, 0, 1)
    Ak, Bk = operands(ex, 1, 1)
    o32, o16, lo = Mat(M, N, F32), Mat(M, N, BF16), Mat(M, N, BF16)
    misaligned = Mat(M, K + 1, BF16, rup(K + 1, 8) + 8, 0, 0, np.ones((M, K + 1), np.float32))
    stage = [Mat(1, M * 320 + 64, F32) for _ in range(2)]
    bias = torch.zeros(N, device="cuda")
    p32 = torch.zeros(rup(M, 32) * 320, device="cuda")

    def base(**kw):
        return desc(lib, M, N, As, Bs, [K], 0, 1, out32=o32, out16=o16, ws=full_ws(), **kw)

    cases = []
    d = base()
    d.a[0] = misaligned.ptr + 2
    cases.append(("operand base 2 bytes off", d))
    d = base()
    d.lda[0] = K + 4                       # 408 bytes: not a multiple of 16
    cases.append(("ld not a multiple of 8", d))
    d = base()
    d.k[0] = 0
    cases.append(("k = 0", d))
    d = base()
    d.nseg = 5
    cases.append(("5 segments", d))
    d = base(beta16=1, lo=lo)
    cases.append(("out16_lo with beta16", d))
    d = desc(lib, M, N, Ak, Bk, [K], 1, 1, bias=bias)
    d.rms_p32 = d.rms_ms = d.rms_mom = p32.data_ptr()
    d.rms_ld, d.rms_blocked = 320, 1
    cases.append(("rms_blocked with a bias", d))
    # the blocked path writes out32 / the bf16 copy in whole 32-column chunks: rows shorter than
    # round_up(N, 32) = 320 would spill into the next row
    for name, ld32, rms_ld in (("rms_blocked with ld32 < round_up(N, 32)", o32.ld, 320),
                               ("rms_blocked with rms_ld < N", None, 288)):
        d = desc(lib, M, N, Ak, Bk, [K], 1, 1, out32=o32 if ld32 else None)
        d.rms_p32 = d.rms_ms = d.rms_mom = p32.data_ptr()
        d.rms_ld, d.rms_blocked = rms_ld, 1
        cases.append((name, d))
    for name, beta, shift in (("route with beta32", 1, 0), ("route_base 4 bytes off", 0, 4)):
        d = desc(lib, M, N, Ak, Bk, [K], 1, 1, out32=o32, beta32=beta)
        d.route_world, d.route_shard, d.route_off0 = 2, 8 * 1000, 0
        d.route_base[0], d.route_base[1] = stage[0].ptr, stage[1].ptr + shift
        cases.append((name, d))
    for name, d in cases:
        n0 = ops.launch_count()
        with pytest.raises(lib.CCError):
            lib.check(lib.load().cc_gemm(C.byref(d), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert ops.launch_count() == n0, name
        for m in (o32, o16, lo):
            assert np.all(np.isnan(m.get())), f"{name}: an output was written"
            m.check_sentinel(name)
        for s in stage:
            assert np.all(np.isnan(s.get())), f"{name}: a route slot was written"


# ============================================================================== 9. coverage
def test_every_instantiation_runs(lib, monkeypatch):
    """One representative case of every dispatch-mirror entry under torch.profiler: the set of
    GEMM-unit kernels seen is all 49 instantiations, and each case's kernels are the mirror's."""
    from torch.profiler import ProfilerActivity, profile
    rng = np.random.default_rng(130)
    shared_ws = Ws(1 << 24)
    runs = []
    for c in G.coverage_cases():
        M, N, (K,) = c["M"], c["N"], c["ks"]
        a_mn, b_mn = c["a_mn"], c["b_mn"]
        ex = G.exact_operands(rng, M, N, [K], [(-10, -10)] if c.get("rms") else None, mag=7)
        As, Bs = operands(ex, a_mn, b_mn)
        o32 = Mat(M, N, F32, rup(N, 64) if c.get("rms") else None)   # blocked: whole 32-col chunks
        bias = torch.zeros(N, device="cuda") if c.get("math_") else None
        assert c.get("workspace_elems", 1 << 24) == 1 << 24
        ws = shared_ws if c.get("workspace_elems") else None
        d = desc(lib, M, N, As, Bs, [K], a_mn, b_mn, bias=bias, out32=o32, ws=ws,
                 splits=c.get("force_splits", 0))
        keep = [As, Bs, o32, bias, ws]
        if c.get("rms"):
            ld = rup(N, 64)
            rows = rup(M, 32)
            st = [torch.zeros(rows * ld, device="cuda") for _ in range(3)]
            p16 = Mat(M, N, BF16, ld)
            d.rms_p32, d.rms_ms, d.rms_mom = (t.data_ptr() for t in st)
            d.rms_p16, d.rms_ld = p16.ptr, ld
            d.rms_lr, d.rms_rho, d.rms_momentum, d.rms_eps = LR, RHO, MOM, EPS
            d.rms_blocked = int(c["rms"] == "blocked")
            keep += [st, p16]
        runs.append((c, d, keep, ex, o32))
    seen = set()
    for c, d, keep, ex, o32 in runs:
        monkeypatch.setenv("CC_GEMM_PERSISTENT_SPLITK", str(c.get("env_persistent_splitk", 1)))
        monkeypatch.setenv("CC_GEMM_RMS_NFAST", str(c.get("env_rms_nfast", -1)))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            launch(lib, d, c, str(c))
            torch.cuda.synchronize()
        names = {G.kernel_name(e.name) for e in prof.events()
                 if e.device_type == torch.autograd.DeviceType.CUDA}
        names.discard(None)
        want, _ = G.dispatch(sms=sms(), **c)
        assert names == set(want), f"{c}: ran {sorted(names)}, the mirror says {want}"
        assert_exact(o32.get(), ex.v32, str(c))
        seen |= names
    missing = G.instantiations() - seen
    assert not missing, f"never ran: {sorted(missing)}"
    assert len(seen) == 49
    print(f"{len(seen)} GEMM-unit instantiations ran")
