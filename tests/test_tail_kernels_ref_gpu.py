"""Every tail kernel (csrc/tail_kernels.cu) against an exact or fp64 host reference
(tests/tail_ref.py), on its vector, scalar, grid-stride, reduction and RNG paths.

Elementwise kernels run over a layout matrix: shapes from 1 x 1 to 2048 x 256, a 1 x N row
wide enough for for_each_chunk8's grid-stride walk, leading dimensions that take the 16-byte
vector path (pad_ld), the scalar path (odd ld, bases 1 and 3 elements off a flat buffer, as in
refresh_lo's clipped ranges) and fp32's float4 path without bf16's (ld % 8 == 4), and every
value of the entry point's dtype mask.  Every output lives in a buffer pre-filled with a
sentinel; what lies outside the view must still hold it afterwards.

Exact results are compared bit for bit.  Rounded ones are held to a bound derived beside the
check (fp32 unit roundoff u = 2^-24, ulp of the output dtype, __expf's documented error)."""
import numpy as np
import pytest
import torch

import tail_ref as R

pytestmark = pytest.mark.gpu

U = R.FP32_U
BF16, F32 = torch.bfloat16, torch.float32
SHAPES = [(1, 1), (1, 7), (3, 9), (5, 8), (77, 515), (130, 1001), (2048, 256)]
LAYOUTS = ["pad", "odd", "ld4", "off1", "off3"]
# sentinel bit patterns: NaNs with a payload no kernel writes
SENTINEL = {BF16: (torch.int16, 0x7FC1), F32: (torch.int32, 0x7FC0DEAD), torch.uint8: (torch.uint8, 0xA5)}


@pytest.fixture(scope="module")
def ops():
    from cellcomm_b200 import ops
    return ops


_SMS = []


def sms():
    if not _SMS:
        _SMS.append(torch.cuda.get_device_properties(0).multi_processor_count)
    return _SMS[0]


def shapes(layout):
    """The layout matrix's shapes; the 1 x N grid-stride row where its base offset differs."""
    out = list(SHAPES)
    if layout in ("pad", "off3"):
        out.append((1, R.fallback_cols(sms())))
    return out


def geometry(cols, layout):
    """(leading dimension, base offset in elements) of a layout."""
    pad = max(64, (cols + 63) // 64 * 64)
    if layout == "odd":
        return cols | 1, 0
    if layout == "ld4":
        ld = (cols + 3) // 4 * 4
        return (ld + 4 if ld % 8 == 0 else ld), 0
    return pad, {"pad": 0, "off1": 1, "off3": 3}[layout]


def dtypes(mask, n):
    return [F32 if (mask >> i) & 1 else BF16 for i in range(n)]


def stored(x32, dtype):
    """The fp32 value of x once stored in dtype."""
    return R.bf16_round(x32) if dtype == BF16 else np.asarray(x32, np.float32)


class Buf:
    """A [rows, cols] view with leading dimension / base offset of `layout` inside a flat device
    buffer pre-filled with a sentinel; `data` (fp32 or uint8 numpy) is stored into the view."""

    def __init__(self, rows, cols, dtype, layout="pad", data=None):
        self.ld, self.off = geometry(cols, layout)
        self.rows, self.cols, self.dtype = rows, cols, dtype
        n = self.off + (rows - 1) * self.ld + cols + 13
        idt, self.pat = SENTINEL[dtype]
        self.raw = torch.full((n,), self.pat, dtype=idt, device="cuda")
        flat = self.raw.view(dtype)
        self.t = torch.as_strided(flat, (rows, cols), (self.ld, 1), self.off)
        if data is not None:
            self.t.copy_(torch.from_numpy(np.ascontiguousarray(data)).to(dtype))

    def get(self):
        t = self.t.contiguous().cpu()
        return t.numpy() if self.dtype == torch.uint8 else t.float().numpy()

    def bits(self):
        t = self.t.contiguous().cpu()
        if self.dtype == BF16:
            return t.view(torch.int16).numpy().view(np.uint16)
        if self.dtype == F32:
            return t.view(torch.int32).numpy().view(np.uint32)
        return t.numpy()

    def check_sentinel(self, what=""):
        raw = self.raw.cpu().numpy()
        inside = np.zeros(raw.shape[0], bool)
        idx = self.off + np.add.outer(np.arange(self.rows, dtype=np.int64) * self.ld,
                                      np.arange(self.cols, dtype=np.int64))
        inside[idx.ravel()] = True
        bad = np.count_nonzero(raw[~inside] != np.array(self.pat).astype(raw.dtype))
        assert bad == 0, f"{what}: {bad} elements outside the view were written"


def want_bits(ref32, dtype):
    ref32 = np.ascontiguousarray(ref32, np.float32)
    return R.bf16_bits(ref32) if dtype == BF16 else ref32.view(np.uint32)


def assert_bits(buf, ref32, what):
    got, want = buf.bits(), want_bits(ref32, buf.dtype)
    bad = got != want
    if bad.any():
        i = np.argwhere(bad)[0]
        g = buf.get()[tuple(i)]
        raise AssertionError(f"{what}: {bad.sum()} of {bad.size} differ, first at {tuple(i)}: "
                             f"got {g!r}, want {np.float32(ref32[tuple(i)])!r}")
    buf.check_sentinel(what)


def assert_within(got, ref, tol, what):
    err = np.abs(np.asarray(got, np.float64) - ref)
    bad = ~(err <= tol)
    if bad.any():
        i = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {bad.sum()} of {bad.size} outside the bound, first at "
                             f"{tuple(i)}: got {got[tuple(i)]!r}, want {ref[tuple(i)]!r}, "
                             f"err {err[tuple(i)]:.3g} > {np.broadcast_to(tol, err.shape)[tuple(i)]:.3g}")


def ulp_of(dtype):
    return R.ulp16 if dtype == BF16 else R.ulp32


def randn(rng, rows, cols, scale=1.0, offset=0.0):
    return (rng.standard_normal((rows, cols), dtype=np.float32) * np.float32(scale)
            + np.float32(offset))


# =========================================================================== elementwise
@pytest.mark.parametrize("xmask", [0, 1])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_split_bf16(ops, layout, xmask):
    rng = np.random.default_rng(11)
    (xd,) = dtypes(xmask, 1)
    for rows, cols in shapes(layout):
        x = randn(rng, rows, cols) * np.float32(10.0) ** rng.integers(-8, 8, (rows, cols)).astype(np.float32)
        xb = Buf(rows, cols, xd, layout, x)
        hi, lo = Buf(rows, cols, BF16, layout), Buf(rows, cols, BF16, layout)
        ops.split_bf16(xb.t, hi.t, lo.t)
        h, l = R.split_ref(stored(x, xd))
        assert_bits(hi, h, f"hi {rows}x{cols}")
        assert_bits(lo, l, f"lo {rows}x{cols}")
        xb.check_sentinel("x")


@pytest.mark.parametrize("mask", range(4))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_copy2d_and_casts(ops, layout, mask):
    rng = np.random.default_rng(12)
    sd, dd = dtypes(mask, 2)
    for rows, cols in shapes(layout):
        x = stored(randn(rng, rows, cols, 3.0), sd)
        src = Buf(rows, cols, sd, layout, x)
        # the plain cast: bit-exact
        dst = Buf(rows, cols, dd, layout)
        ops.copy2d(src.t, dst.t)
        assert_bits(dst, x, f"cast {rows}x{cols}")
        # scale only: one fp32 product, bit-exact
        ops.copy2d(src.t, dst.t, scale=0.3)
        assert_bits(dst, x * np.float32(0.3), f"scale {rows}x{cols}")
        # scale + accumulate: one product and one sum in fp32, then the store: within 1 ulp of
        # the output dtype, plus the product's rounding where the compiler does not contract
        # the two into an FMA
        d0 = stored(randn(rng, rows, cols), dd)
        acc = Buf(rows, cols, dd, layout, d0)
        ops.copy2d(src.t, acc.t, beta=1, scale=1.7)
        prod = x.astype(np.float64) * np.float64(np.float32(1.7))
        exact = prod + d0
        tol = ulp_of(dd)(exact) + U * np.abs(prod)
        assert_within(acc.get(), exact, tol, f"accumulate {rows}x{cols}")
        acc.check_sentinel("accumulate")
        src.check_sentinel("src")


@pytest.mark.parametrize("mask", range(8))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_act_bwd(ops, layout, mask):
    """dz = dy * act'(y) with act' computed in fp32 from the stored y: none and relu are exact,
    sigmoid is dy * (y * (1 - y)), three correctly rounded fp32 operations."""
    rng = np.random.default_rng(13)
    dyd, yd, zd = dtypes(mask, 3)
    for rows, cols in shapes(layout):
        dy = stored(randn(rng, rows, cols, 2.0), dyd)
        pre = randn(rng, rows, cols, 3.0)
        pre[0, 0] = -0.0
        for act, y32 in ((ops.ACT_NONE, pre), (ops.ACT_RELU, np.maximum(pre, np.float32(0))),
                         (ops.ACT_SIGMOID, (1 / (1 + np.exp(-pre))).astype(np.float32))):
            y = stored(y32, yd)
            dyb, yb = Buf(rows, cols, dyd, layout, dy), Buf(rows, cols, yd, layout, y)
            dz = Buf(rows, cols, zd, layout)
            ops.act_bwd(dyb.t, yb.t, dz.t, act)
            ref = R.act_grad_f32(dy, y, act)
            assert_bits(dz, ref, f"act {act} {rows}x{cols}")
            # and the sigmoid emulation is within 3 roundings of the fp64 product
            if act == ops.ACT_SIGMOID and zd == F32:
                exact = R.act_grad64(dy.astype(np.float64), y.astype(np.float64), act)
                assert np.all(np.abs(ref - exact) <= 3 * U * np.abs(exact))


ROUND_SPECIAL = np.array([0.5, -0.5, 1.5, -1.5, 2.5, -2.5, -0.4, 0.4, 3.5, -3.5, 0.49999997,
                          2 ** 22 + 0.5, 2 ** 22 + 1.5, 2 ** 23 - 0.5, 2 ** 23 - 1.5, -(2 ** 23 - 0.5),
                          2 ** 24, 2 ** 24 + 2, -(2 ** 25), 3e38, -0.0, 0.0], np.float32)


@pytest.mark.parametrize("mask", range(4))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_round_half_even(ops, layout, mask):
    """rint of the stored value, bit for bit (-0.4 -> -0.0 included), into out and out32."""
    rng = np.random.default_rng(14)
    xd, od = dtypes(mask, 2)
    for rows, cols in shapes(layout):
        x = randn(rng, rows, cols, 40.0)
        flat = x.reshape(-1)
        k = min(flat.size, ROUND_SPECIAL.size)
        flat[:k] = ROUND_SPECIAL[:k]
        flat[k:k + 2000] = (rng.integers(-400, 400, min(2000, flat.size - k)) + 0.5).astype(np.float32)
        xs = stored(x, xd)
        xb = Buf(rows, cols, xd, layout, xs)
        out, out32 = Buf(rows, cols, od, layout), Buf(rows, cols, F32, layout)
        ops.round_half_even(xb.t, out16=out.t, out32=out32.t)
        ref = np.rint(xs)
        assert_bits(out, ref, f"out {rows}x{cols}")
        assert_bits(out32, ref, f"out32 {rows}x{cols}")


@pytest.mark.parametrize("mask", range(4))
@pytest.mark.parametrize("layout", LAYOUTS)
def test_dropout_explicit_mask(ops, layout, mask):
    rng = np.random.default_rng(15)
    xd, od = dtypes(mask, 2)
    for rows, cols in shapes(layout):
        x = stored(randn(rng, rows, cols), xd)
        keep = (rng.random((rows, cols)) >= 0.15).astype(np.uint8)
        xb, mb = Buf(rows, cols, xd, layout, x), Buf(rows, cols, torch.uint8, layout, keep)
        for rate in (0.0, 0.15):
            out = Buf(rows, cols, od, layout)
            ops.dropout(xb.t, out.t, rate, mask=mb.t)
            assert_bits(out, R.dropout_ref(x, keep.astype(bool), rate), f"rate {rate} {rows}x{cols}")


# ------------------------------------------------------------------------------- RNG
RNG_CASES = [
    # rows, cols, layout, seed, counter (None: no device counter), stream id
    (64, 256, "pad", 1, 0, 0),
    (33, 9, "odd", 123, 7, 5),                    # cols % 4 == 1 (and % 8 == 1)
    (17, 10, "ld4", 77, 3, 1000),                 # cols % 4 == 2
    (5, 7, "off1", 5, 1, 1001),                   # cols % 4 == 3
    (40, 3, "pad", 9, 2, 6),                      # cols < 4
    (9, 1, "off3", 10, 4, 7),
    (12, 2, "odd", 11, 4, 8),
    (130, 1001, "pad", 12, 6, 9),                 # ld > cols, cols % 8 == 1
    (29, 12, "pad", 13, 6, 10),                   # cols % 8 == 4
    (1, "fallback", "pad", 14, 8, 11),
    (1, "fallback", "off3", 15, 8, 12),
    (31, 100, "pad", 16, None, 13),
    (31, 100, "odd", 17, (1 << 33) + 5, 14),      # device counter above 2^32
    (31, 100, "pad", (0xDEADBEEF << 32) | 17, 9, 15),   # key's high word set
    (31, 100, "pad", 18, 9, (1 << 24) - 1),       # the largest distinct stream id
    (3, 33, "off1", 19, (1 << 40) - 1, 0),        # the largest step below the id bits
]


@pytest.mark.parametrize("case", range(len(RNG_CASES)))
def test_rng_matches_host_philox(ops, case):
    """dropout / dropout_mask / uniform on the RNG path equal the host Philox bit for bit: the
    stream is a function of (seed, step, stream id, row, column) alone, whatever the layout and
    launch geometry.  uniform's bf16 copy is bf16_rn of its fp32 value (1.0 included)."""
    rows, cols, layout, seed, step, sid = RNG_CASES[case]
    if cols == "fallback":
        cols = R.fallback_cols(sms())
    rng = np.random.default_rng(16 + case)
    counter = None if step is None else torch.tensor([step], dtype=torch.int64, device="cuda")
    u = R.rng_uniform(seed, step or 0, sid, rows, cols)
    rate = 0.15
    keep = R.keep_mask(u, rate)
    for xd, od in ((F32, F32), (BF16, BF16), (F32, BF16)):
        x = stored(randn(rng, rows, cols), xd)
        xb, out = Buf(rows, cols, xd, layout, x), Buf(rows, cols, od, layout)
        ops.dropout(xb.t, out.t, rate, seed=seed, counter=counter, stream_id=sid)
        assert_bits(out, R.dropout_ref(x, keep, rate), f"dropout {xd}->{od}")
    m = Buf(rows, cols, torch.uint8, layout)
    ops.dropout_mask(m.t, rate, seed=seed, counter=counter, stream_id=sid)
    assert np.array_equal(m.get(), keep.astype(np.uint8))
    m.check_sentinel("mask")
    u32, u16 = Buf(rows, cols, F32, layout), Buf(rows, cols, BF16, layout)
    ops.uniform(out32=u32.t, out16=u16.t, seed=seed, counter=counter, stream_id=sid)
    assert_bits(u32, u, "uniform out32")
    assert_bits(u16, u, "uniform out16")          # bf16_rn(u): may be 1.0
    assert u.max() < 1.0
    if counter is not None:
        # the next step's stream after counter_add
        ops.counter_add(counter, 3)
        assert counter.item() == step + 3
        u32b = Buf(rows, cols, F32, layout)
        ops.uniform(out32=u32b.t, seed=seed, counter=counter, stream_id=sid)
        assert_bits(u32b, R.rng_uniform(seed, step + 3, sid, rows, cols), "after counter_add")


def test_rng_streams_are_distinct_and_bf16_reaches_one(ops):
    """Different stream ids / steps / seeds give different streams; ids alias modulo 2^24 (the
    documented limit); about 2^-9 of bf16 uniforms round up to exactly 1.0."""
    rows, cols = 256, 1024

    def draw(seed, step, sid):
        out = torch.empty(rows, cols, device="cuda")
        c = torch.tensor([step], dtype=torch.int64, device="cuda")
        ops.uniform(out32=out, seed=seed, counter=c, stream_id=sid)
        return out

    a = draw(1, 0, 0)
    for other in (draw(1, 0, 1), draw(1, 1, 0), draw(2, 0, 0), draw(1, 0, (1 << 24) - 1),
                  draw(1 << 32, 0, 0)):
        assert (a == other).float().mean().item() < 1e-3
    assert torch.equal(draw(1, 0, 5), draw(1, 0, 5 + (1 << 24)))
    u16 = torch.empty(rows, cols, dtype=BF16, device="cuda")
    ops.uniform(out16=u16, seed=3, stream_id=1000)
    ones = (u16 == 1.0).float().mean().item()
    assert 0.5 * 2 ** -9 < ones < 2 * 2 ** -9


# ============================================================================= reductions
RED_ROWS = [1, 8, 31, 64, 65, 300, 2047, 2048, 4096]


def red_cols():
    """Column counts, with the single-slab edge: 2 * SMs - 1 column blocks take two row slabs,
    2 * SMs blocks take one."""
    e = 128 * (2 * sms() - 1)
    return [1, 127, 128, 129, 3369, e, e + 1]


def dev_rand(rows, cols, dtype, layout, gen, offset=0.0, scale=1.0):
    """Random [rows, cols] view of `layout` on the device (what lies outside it is random too)."""
    ld, off = geometry(cols, layout)
    flat = (torch.randn(off + rows * ld, generator=gen, device="cuda") * scale + offset).to(dtype)
    return torch.as_strided(flat, (rows, cols), (ld, 1), off)


def vec_out(n, fill=None):
    """n fp32 outputs followed by 13 sentinel floats; returns (buffer, view)."""
    raw = torch.full((n + 13,), SENTINEL[F32][1], dtype=torch.int32, device="cuda")
    v = raw.view(F32)[:n]
    if fill is not None:
        v.copy_(fill)
    return raw, v


def tail_ok(raw, n):
    return bool((raw[n:] == SENTINEL[F32][1]).all())


def check_sum(got, ref, abs_sum, adds, what, roundings=0):
    tol = R.sum_bound(abs_sum, adds, roundings)
    err = (got.double() - ref).abs()
    bad = ~(err <= tol)
    if bad.any():
        i = int(bad.nonzero()[0, 0])
        raise AssertionError(f"{what}: {int(bad.sum())} columns outside the bound, first {i}: got "
                             f"{got[i].item()!r}, want {ref[i].item()!r}, bound {tol[i].item():.3g}")


@pytest.mark.parametrize("path", ["atomic", "ws"])
@pytest.mark.parametrize("kernel", ["colsum", "bias_grad", "bn_stats", "bn_bwd_stats"])
def test_column_reductions(ops, kernel, path):
    """Column sums against fp64: |got - exact| <= n_adds * u * sum |term| with n_adds the
    longest chain of fp32 additions of the launch (ceil(rows_per_slab / 8) + 8 + slabs).  The
    ws path uses ONE workspace, sized by cc_reduce_ws_floats for the largest shape, for every
    shape, and leaves its tickets zero."""
    gen = torch.Generator(device="cuda").manual_seed(21)
    cols_list = red_cols()
    ws = None
    if path == "ws":
        ws = torch.zeros(ops.reduce_ws_floats(max(RED_ROWS), max(cols_list)), device="cuda")
    i = 0
    for rows in RED_ROWS:
        for cols in cols_list:
            for offset in (0.0, 100.0):
                i += 1
                d0 = F32 if i % 2 else BF16
                d1 = F32 if (i // 2) % 2 else BF16
                layout = ("pad", "odd", "off1")[i % 3]
                adds = R.colreduce_adds(rows, cols, sms())
                what = f"{kernel} {path} {rows}x{cols} +{offset} {d0} {layout}"
                a = dev_rand(rows, cols, d0, layout, gen, offset)
                a64 = a.double()
                if kernel == "colsum":
                    beta = (i // 3) % 2
                    start = torch.randn(cols, generator=gen, device="cuda") if beta else None
                    raw, out = vec_out(cols, start)
                    ops.colsum(a, out, beta, ws=ws)
                    s0 = start.double() if beta else torch.zeros(cols, device="cuda", dtype=torch.float64)
                    # beta: the starting value joins the chain of additions
                    check_sum(out, a64.sum(0) + s0, a64.abs().sum(0) + s0.abs(), adds + beta, what)
                    assert tail_ok(raw, cols), what
                elif kernel == "bn_stats":
                    raw, sums = vec_out(2 * cols)
                    ops.bn_stats(a, sums, ws=ws)
                    check_sum(sums[:cols], a64.sum(0), a64.abs().sum(0), adds, what)
                    check_sum(sums[cols:], (a64 * a64).sum(0), (a64 * a64).sum(0), adds,
                              what + " x^2", roundings=1)
                    assert tail_ok(raw, 2 * cols), what
                elif kernel == "bn_bwd_stats":
                    dy = dev_rand(rows, cols, d1, layout, gen, 0.3)
                    x64 = a64
                    mean = x64.mean(0).float()
                    rstd = (1.0 / torch.sqrt(x64.var(0, unbiased=False) + 1e-3)).float()
                    xhat = (a.float() - mean) * rstd               # two fp32 roundings, as the kernel
                    raw, sums2 = vec_out(2 * cols)
                    ops.bn_bwd_stats(dy, a, mean, rstd, sums2, ws=ws)
                    dy64 = dy.double()
                    t1 = dy64 * xhat.double()
                    check_sum(sums2[:cols], dy64.sum(0), dy64.abs().sum(0), adds, what + " dy")
                    check_sum(sums2[cols:], t1.sum(0), t1.abs().sum(0), adds, what + " dy*xhat",
                              roundings=1)
                    assert tail_ok(raw, 2 * cols), what
                else:
                    act = i % 3
                    ypre = dev_rand(rows, cols, F32, layout, gen, 0.0, 3.0)
                    y32 = (torch.sigmoid(ypre) if act == 1 else torch.relu(ypre) if act == 2
                           else ypre)
                    y = y32.to(d1)
                    ys = y.float()
                    dyf = a.float()
                    v = (dyf * (ys * (1 - ys)) if act == 1 else dyf * (ys > 0).float() if act == 2
                         else dyf)
                    want_dz = (i // 3) % 2 == 0
                    zd = F32 if (i // 5) % 2 else BF16
                    dz = Buf(rows, cols, zd, layout) if want_dz else None
                    dzlo = Buf(rows, cols, BF16, layout) if want_dz and zd == BF16 and i % 4 < 2 else None
                    dz_only = want_dz and i % 7 == 0
                    beta = (i // 4) % 2 if not dz_only else 0
                    start = torch.randn(cols, generator=gen, device="cuda") if beta else None
                    raw, out = vec_out(cols, start)
                    ops.bias_grad(a, y, act, None if dz_only else out,
                                  dz=None if dz is None else dz.t, beta=beta,
                                  dz_lo=None if dzlo is None else dzlo.t, ws=ws)
                    if not dz_only:
                        s0 = start.double() if beta else 0
                        check_sum(out, v.double().sum(0) + s0,
                                  v.double().abs().sum(0) + (s0.abs() if beta else 0), adds + beta, what)
                    else:
                        assert (raw.view(torch.int32) == SENTINEL[F32][1]).all(), "dz-only wrote out"
                    assert tail_ok(raw, cols), what
                    if dz is not None:
                        assert torch.equal(dz.t.contiguous(), v.to(zd)), what + " dz"
                        dz.check_sentinel(what + " dz")
                    if dzlo is not None:
                        lo = (v - v.to(BF16).float()).to(BF16)
                        assert torch.equal(dzlo.t.contiguous(), lo), what + " dz_lo"
                        dzlo.check_sentinel(what + " dz_lo")
                del a, a64
    if ws is not None:
        assert int(ws[: 2 * sms()].view(torch.int32).abs().sum().item()) == 0, "tickets not reset"


def test_reduce_workspace_too_small_is_an_error(ops):
    from cellcomm_b200._lib import CCError
    x = torch.randn(4096, 1, device="cuda")
    # a one-column sum of 4096 rows: 2 * SMs tickets and one partial per row slab
    need = 2 * sms() + R.colreduce_grid(4096, 1, sms())[1]
    assert ops.reduce_ws_floats(4096, 1) >= need
    out = torch.empty(1, device="cuda")
    with pytest.raises(CCError, match="workspace"):
        ops.colsum(x, out, ws=torch.zeros(need - 1, device="cuda"))
    ws = torch.zeros(need, device="cuda")
    ops.colsum(x, out, ws=ws)
    assert abs(out.item() - x.double().sum().item()) <= R.sum_bound(
        x.double().abs().sum().item(), R.colreduce_adds(4096, 1, sms()))


# ============================================================================= BatchNorm
BN_OFFSETS = [(0.0, 1.0), (0.5, 0.05), (0.999, 0.001), (30.0, 1.0)]
BN_SHAPES = [(1, 7), (5, 8), (77, 515), (300, 129), (2048, 256)]


def _bn_forward(ops, x, cols, n_total, sums, gamma, beta, mm0, mv0, yd, layout):
    rows = x.shape[0]
    y = Buf(rows, cols, yd, layout)
    mm, mv = torch.tensor(mm0, device="cuda"), torch.tensor(mv0, device="cuda")
    sm, sr = torch.empty(cols, device="cuda"), torch.empty(cols, device="cuda")
    ops.bn_train_apply(x, y.t, sums, n_total, gamma, beta, 1e-3, 0.99, mm, mv, sm, sr)
    return y, mm, mv, sm, sr


@pytest.mark.parametrize("mask", range(8))
@pytest.mark.parametrize("layout", ["pad", "odd", "ld4", "off1"])
def test_batchnorm(ops, layout, mask):
    """bn_stats -> bn_train_apply -> bn_bwd_stats -> bn_bwd_apply (+ inference forms) against
    fp64 two-pass statistics and the closed-form gradients:
    - save_mean, save_rstd within 1e-3 relative (the one-pass E[x^2] - E[x]^2 limit, measured
      in test_bn_one_pass_limit);
    - y, dx within 1 ulp of the output dtype plus the fp32 evaluation error and the
      propagated error of the statistics;
    - n_total = 2 * rows with the sums doubled (two ranks holding the same batch) gives the
      single-rank result bit for bit;
    - moving statistics with the Keras momentum update."""
    rng = np.random.default_rng(30 + mask)
    xd, yd, dxd = dtypes(mask, 3)
    eps = np.float32(1e-3)
    for si, (rows, cols) in enumerate(BN_SHAPES):
        for mu, sd in BN_OFFSETS:
            what = f"{rows}x{cols} {mu}/{sd} {layout} mask {mask}"
            x = stored(randn(rng, rows, cols, sd, mu), xd)
            xb = Buf(rows, cols, xd, layout, x)
            ws = torch.zeros(ops.reduce_ws_floats(rows, cols), device="cuda") if si % 2 else None
            sums = torch.empty(2 * cols, device="cuda")
            ops.bn_stats(xb.t, sums, ws=ws)
            gamma32 = (rng.random(cols, dtype=np.float32) + np.float32(0.5))
            beta32 = rng.standard_normal(cols, dtype=np.float32)
            mm0 = rng.standard_normal(cols, dtype=np.float32)
            mv0 = rng.random(cols, dtype=np.float32) + np.float32(0.5)
            gamma, beta = torch.from_numpy(gamma32).cuda(), torch.from_numpy(beta32).cuda()
            y, mm, mv, sm, sr = _bn_forward(ops, xb.t, cols, rows, sums, gamma, beta, mm0, mv0, yd,
                                            layout)
            x64 = x.astype(np.float64)
            mean64, var64 = R.bn_moments64(x64)
            rstd64 = 1.0 / np.sqrt(var64 + float(eps))
            smh, srh = sm.cpu().numpy().astype(np.float64), sr.cpu().numpy().astype(np.float64)
            adds = R.colreduce_adds(rows, cols, sms())
            mean_tol = 1e-3 * np.abs(mean64) + R.sum_bound(np.abs(x64).sum(0), adds) / rows
            assert_within(smh, mean64, mean_tol, what + " save_mean")
            # one row has zero variance: var is then the rounding of the fp32 sum of x^2 alone
            # (a relative u of E[x^2]), which the one-pass bound of test_bn_one_pass_limit covers
            rstd_tol = (1e-3 if rows > 1 else
                        3 * adds * U * (x64 * x64).mean(0) / (2 * (var64 + float(eps))) + 1e-6)
            assert_within(srh, rstd64, rstd_tol * rstd64, what + " save_rstd")
            # y from the saved statistics: (x - mu) * (gamma * rstd) + beta in fp32
            gr = gamma32.astype(np.float64) * srh
            yref = (x64 - smh) * gr + beta32
            ytol = ulp_of(yd)(yref) + 4 * U * (np.abs(x64 - smh) * gr + np.abs(beta32))
            assert_within(y.get(), yref, ytol, what + " y")
            y.check_sentinel(what + " y")
            # moving statistics: moving * 0.99 + batch * 0.01; the batch variance carries the
            # one-pass error 3 * n_adds * u * E[x^2]
            var_tol = 3 * adds * U * (x64 * x64).mean(0) + 2e-3 * var64
            mm_ref = R.moving_update64(mm0.astype(np.float64), mean64, 0.99)
            mv_ref = R.moving_update64(mv0.astype(np.float64), var64, 0.99)
            assert_within(mm.cpu().numpy(), mm_ref, 4 * U * (np.abs(mm0) + np.abs(mean64))
                          + 0.01 * mean_tol, what + " moving_mean")
            assert_within(mv.cpu().numpy(), mv_ref, 4 * U * (np.abs(mv0) + var64) + 0.01 * var_tol,
                          what + " moving_var")
            # two ranks with the same batch: doubled sums, n_total = 2 * rows -> same bits
            y2, mm2, mv2, sm2, sr2 = _bn_forward(ops, xb.t, cols, 2 * rows, sums * 2, gamma, beta,
                                                 mm0, mv0, yd, layout)
            for a, b in ((y2.t, y.t), (mm2, mm), (mv2, mv), (sm2, sm), (sr2, sr)):
                assert torch.equal(a, b), what + " n_total = 2 rows"
            # ---- backward
            dy = stored(randn(rng, rows, cols, 1.0, 0.3), dxd if mask & 4 else xd)
            dyd = dxd if mask & 4 else xd
            dyb = Buf(rows, cols, dyd, layout, dy)
            sums2 = torch.empty(2 * cols, device="cuda")
            ops.bn_bwd_stats(dyb.t, xb.t, sm, sr, sums2, ws=ws)
            dx = Buf(rows, cols, dxd, layout)
            dg, db = torch.empty(cols, device="cuda"), torch.empty(cols, device="cuda")
            ops.bn_bwd_apply(dyb.t, xb.t, dx.t, gamma, sm, sr, sums2, rows, dg, db)
            assert torch.equal(db, sums2[:cols]) and torch.equal(dg, sums2[cols:])
            dy64 = dy.astype(np.float64)
            dx_ref, dg_ref, db_ref = R.bn_train_bwd64(dy64, x64, gamma32.astype(np.float64),
                                                      float(eps))
            # statistic errors the kernel's xhat inherits
            e_r = np.abs(srh / rstd64 - 1)
            e_m = np.abs(smh - mean64) * rstd64
            xhat = (x64 - mean64) * rstd64
            dxhat_err = np.abs(xhat) * e_r + e_m * (1 + e_r)
            s0n, s1n = np.abs(dy64.mean(0)), np.abs((dy64 * xhat).mean(0))
            b0 = R.sum_bound(np.abs(dy64).sum(0), adds) / rows
            b1 = (R.sum_bound(np.abs(dy64 * xhat).sum(0), adds, 4)
                  + (np.abs(dy64) * dxhat_err).sum(0)) / rows
            assert_within(db.cpu().numpy(), db_ref, b0 * rows, what + " dbeta")
            assert_within(dg.cpu().numpy(), dg_ref, b1 * rows, what + " dgamma")
            gr64 = gamma32.astype(np.float64) * rstd64
            mag = np.abs(dy64) + s0n + np.abs(xhat) * s1n
            dx_tol = (ulp_of(dxd)(dx_ref) + gr64 * (8 * U * mag + e_r * mag + dxhat_err * s1n
                                                     + b0 + (np.abs(xhat) + dxhat_err) * b1))
            assert_within(dx.get(), dx_ref, dx_tol, what + " dx")
            dx.check_sentinel(what + " dx")
            # two ranks: doubled sums, n_total = 2 * rows -> same dx bits
            dx2 = Buf(rows, cols, dxd, layout)
            ops.bn_bwd_apply(dyb.t, xb.t, dx2.t, gamma, sm, sr, sums2 * 2, 2 * rows)
            assert torch.equal(dx2.t, dx.t), what + " dx, n_total = 2 rows"
            # ---- inference forms from the moving statistics
            yi = Buf(rows, cols, yd, layout)
            ops.bn_infer(xb.t, yi.t, gamma, beta, mm, mv, float(eps))
            mmh, mvh = mm.cpu().numpy().astype(np.float64), mv.cpu().numpy().astype(np.float64)
            ri = 1.0 / np.sqrt(mvh + np.float64(eps))
            gri = gamma32 * ri
            yiref = (x64 - mmh) * gri + beta32
            yitol = ulp_of(yd)(yiref) + (4 * U + 2.0 ** -22) * np.abs(x64 - mmh) * gri + 4 * U * np.abs(beta32)
            assert_within(yi.get(), yiref, yitol, what + " bn_infer")
            yi.check_sentinel(what + " bn_infer")
            dxi = Buf(rows, cols, dxd, layout)
            ops.bn_infer_bwd(dyb.t, dxi.t, gamma, mv, float(eps))
            dxiref = dy64 * gri
            assert_within(dxi.get(), dxiref, ulp_of(dxd)(dxiref) + (4 * U + 2.0 ** -22) * np.abs(dxiref),
                          what + " bn_infer_bwd")
            dxi.check_sentinel(what + " bn_infer_bwd")


@pytest.mark.parametrize("mean_over_std", [100, 300, 1000])
def test_bn_one_pass_limit(ops, mean_over_std, record_property):
    """Diagnostic: the error of save_rstd when the batch mean is far above the spread (the
    statistics are one-pass fp32 sums, E[x^2] - E[x]^2).  Records the measured error; asserts
    it stays within the one-pass bound 3 * n_adds * u * E[x^2] / (2 (var + eps)).
    Measured on an NVIDIA B200 (1,000 W power limit), 2048 x 128 fp32, eps 1e-3: maximum relative
    error 2.7e-3 at mean/std 100, 2.5e-2 at 300, 0.48 at 1000."""
    rows, cols = 2048, 128
    g = torch.Generator(device="cuda").manual_seed(40)
    x = torch.randn(rows, cols, generator=g, device="cuda") + float(mean_over_std)
    sums = torch.empty(2 * cols, device="cuda")
    ops.bn_stats(x, sums)
    gamma, beta = torch.ones(cols, device="cuda"), torch.zeros(cols, device="cuda")
    y = torch.empty(rows, cols, device="cuda")
    sm, sr = torch.empty(cols, device="cuda"), torch.empty(cols, device="cuda")
    ops.bn_train_apply(x, y, sums, rows, gamma, beta, 1e-3, 0.99, None, None, sm, sr)
    x64 = x.double().cpu().numpy()
    _, var = R.bn_moments64(x64)
    rstd = 1 / np.sqrt(var + 1e-3)
    err = np.abs(sr.cpu().numpy() / rstd - 1)
    record_property("save_rstd_max_rel_err", float(err.max()))
    print(f"mean/std {mean_over_std}: save_rstd max relative error {err.max():.3g}")
    adds = R.colreduce_adds(rows, cols, sms())
    bound = 3 * adds * U * (x64 * x64).mean(0) / (2 * (var + 1e-3))
    assert np.all(err <= bound + 1e-6)


# ============================================================================ softmax / argmax
SOFTMAX_WIDTHS = [1, 2, 3, 10, 33, 128]


def _softmax_input(rng, rows, cols, scale):
    x = randn(rng, rows, cols, scale)
    x[1, :] = 0.25                                 # all equal
    x[2, 0] = 80.0                                 # +-80 in one row
    x[2, -1] = -80.0
    x[3, :] = -80.0
    x[3, cols // 2] = 80.0
    return x


@pytest.mark.parametrize("mask", range(8))
@pytest.mark.parametrize("layout", ["pad", "odd", "off1"])
def test_softmax(ops, layout, mask):
    """Forward against fp64: relative error of y_j at most
    e(d_j) + max_k e(d_k) + (cols + 1) u + rounding of the output,
    e(d) the __expf bound at d = x - max (tail_ref.expf_rel_bound): the sum's terms, its fp32
    summation, the reciprocal and the product.  Results below 2^-125 may be flushed to zero.
    Backward: dx = y (dy - sum dy y) with an fp32 dot of `cols` fused terms."""
    rng = np.random.default_rng(50 + mask)
    xd, yd, dyd = dtypes(mask, 3)
    rows = 300
    for cols in SOFTMAX_WIDTHS:
        for scale in (1.0, 30.0):
            what = f"{rows}x{cols} scale {scale} {layout} mask {mask}"
            x = stored(_softmax_input(rng, rows, cols, scale), xd)
            xb = Buf(rows, cols, xd, layout, x)
            y, y32 = Buf(rows, cols, yd, layout), Buf(rows, cols, F32, layout)
            ops.softmax_fwd(xb.t, y.t, y32.t)
            x64 = x.astype(np.float64)
            ref = R.softmax64(x64)
            d = x - x.max(-1, keepdims=True)          # fp32, as the kernel forms it
            e = R.expf_rel_bound(d)
            rel = e + e.max(-1, keepdims=True) + (cols + 1) * U
            tiny = 2.0 ** -125
            assert_within(y32.get(), ref, rel * ref + R.ulp32(ref) * 0.5 + tiny, what + " y32")
            assert_within(y.get(), ref, rel * ref + ulp_of(yd)(ref) + tiny, what + " y")
            y.check_sentinel(what + " y")
            y32.check_sentinel(what + " y32")
            # backward from the stored y
            ys = y.get().astype(np.float64)
            dy = stored(randn(rng, rows, cols), dyd)
            dyb = Buf(rows, cols, dyd, layout, dy)
            dxd = yd
            dx = Buf(rows, cols, dxd, layout)
            ops.softmax_bwd(dyb.t, y.t, dx.t)
            dy64 = dy.astype(np.float64)
            dref = R.softmax_bwd64(dy64, ys)
            dot_abs = np.abs(dy64 * ys).sum(-1, keepdims=True)
            dtol = ulp_of(dxd)(dref) + (cols + 2) * U * np.abs(ys) * (np.abs(dy64) + dot_abs)
            assert_within(dx.get(), dref, dtol, what + " dx")
            dx.check_sentinel(what + " dx")


@pytest.mark.parametrize("layout", ["pad", "odd", "off3"])
def test_argmax_onehot(ops, layout):
    """The first maximum wins (ties), -inf entries, width 1; out16 and out32, alone or both."""
    rng = np.random.default_rng(60)
    for rows, cols in [(1, 1), (300, 1), (300, 2), (257, 10), (64, 33)]:
        p = rng.integers(0, 4, (rows, cols)).astype(np.float32)       # many ties
        p[rng.random((rows, cols)) < 0.2] = -np.inf
        p[0, :] = -np.inf
        pb = Buf(rows, cols, F32, layout, p)
        ref = R.onehot_argmax(p)
        for want16, want32 in ((True, True), (True, False), (False, True)):
            o16 = Buf(rows, cols, BF16, layout) if want16 else None
            o32 = Buf(rows, cols, F32, layout) if want32 else None
            ops.argmax_onehot(pb.t, out16=o16.t if o16 else None, out32=o32.t if o32 else None)
            for o in (o16, o32):
                if o is not None:
                    assert_bits(o, ref, f"argmax {rows}x{cols}")


# ================================================================================== losses
BCE_LOGITS = [1e-3, -1e-3, 5, -5, 20, -20, 88, -88, 100, -100]
BCE_PROBS = [0.0, 1e-9, 0.5, 1 - 1e-9, 1.0]


@pytest.mark.parametrize("dzd", [F32, BF16])
@pytest.mark.parametrize("from_logits", [True, False])
def test_bce(ops, from_logits, dzd):
    """loss_out += sum_r bce_r / n_total against fp64 (relative 1e-5, plus for probabilities the
    rounding of 1 - q before its log, u per element); dz = (p - t) / n_total, p = sigmoid(x)
    (logits) or the unclipped input, within the fp32 error of p and the subtraction."""
    rng = np.random.default_rng(70)
    for rows in (1, 255, 256, 257, 2048):
        for target in (0.0, 0.95, 1.0):
            for n_total, l0 in ((rows, 0.0), (2 * rows, 0.25)):
                what = f"rows {rows} t {target} n {n_total} logits {from_logits}"
                vals = np.array(BCE_LOGITS if from_logits else BCE_PROBS, np.float32)
                x = np.resize(vals, rows).astype(np.float32)
                if rows > 64:
                    x[64:] = (randn(rng, rows - 64, 1, 4.0)[:, 0] if from_logits
                              else rng.random(rows - 64, dtype=np.float32))
                xb = Buf(rows, 3, F32, "odd", np.stack([x, x + 1, x + 2], 1))   # strided column
                loss = torch.full((1,), l0, device="cuda")
                dz = Buf(rows, 1, dzd, "pad")
                ops.bce_fwd_bwd(xb.t[:, :1], target, n_total, loss, dz.t, from_logits=from_logits)
                t32 = float(np.float32(target))
                x64 = x.astype(np.float64)
                per = R.bce_logits64(x64, t32) if from_logits else R.bce_probs64(x64, t32)
                L = per.sum() / n_total
                tol = 1e-5 * abs(L) + R.ulp32(l0 + L)
                if not from_logits:
                    tol += rows * U / n_total
                assert abs(loss.item() - (l0 + L)) <= tol, f"{what}: loss {loss.item()!r} vs {l0 + L!r}"
                p = R.sigmoid64(x64) if from_logits else x64
                inv = 1.0 / n_total
                ref = (p - t32) * inv
                # (+ inv * 2^-125: expf(-x) overflows for x < -88.7, so p is 0, not ~1e-39)
                dtol = ulp_of(dzd)(ref) + inv * (2.0 ** -21 * p + 2.0 ** -22 * np.abs(p - t32) + 2.0 ** -125)
                assert_within(dz.get()[:, 0], ref, dtol, what + " dz")
                dz.check_sentinel(what + " dz")


@pytest.mark.parametrize("path", ["atomic", "ws"])
@pytest.mark.parametrize("mask", range(8))
def test_mse(ops, mask, path):
    """loss_out += sum (pred - target)^2 / (n_total * cols) within 1e-5 of fp64;
    dpred = (2 (pred - target)) * (1 / (n_total * cols)) as the kernel forms it in fp32, exact."""
    rng = np.random.default_rng(80 + mask)
    pd, td, gd = dtypes(mask, 3)
    for rows in (1, 64, 300):
        for cols in (1, 3, 7, 9, 33694):
            for layout in ("pad", "odd", "off1"):
                n_total, l0 = (rows, 0.0) if cols % 2 else (3 * rows, 0.5)
                what = f"{rows}x{cols} {layout} n {n_total}"
                a, t = stored(randn(rng, rows, cols), pd), stored(randn(rng, rows, cols, 1, 0.2), td)
                ab, tb = Buf(rows, cols, pd, layout, a), Buf(rows, cols, td, layout, t)
                g = Buf(rows, cols, gd, layout)
                loss = torch.full((1,), l0, device="cuda")
                ws = torch.zeros(ops.reduce_ws_floats(rows, cols), device="cuda") if path == "ws" else None
                ops.mse_fwd_bwd(ab.t, n_total, loss, target=tb.t, dpred=g.t, ws=ws)
                L, _ = R.mse64(a.astype(np.float64), t.astype(np.float64), n_total)
                assert abs(loss.item() - (l0 + L)) <= 1e-5 * L + R.ulp32(l0 + L), \
                    f"{what}: loss {loss.item()!r} vs {l0 + L!r}"
                inv = np.float32(1) / (np.float32(n_total) * np.float32(cols))
                assert_bits(g, (np.float32(2) * (a - t)) * inv, what + " dpred")
                if ws is not None:
                    assert int(ws[: 2 * sms()].view(torch.int32).abs().sum().item()) == 0


# ================================================================================= RMSprop
LR, RHO, MOM, EPS = 0.0075, 0.85, 0.1, 1e-7


def _grads(rng, shape):
    """Magnitudes from 1e-6 to 10, exact zeros included (sqrt(ms + eps) with ms == 0)."""
    g = rng.standard_normal(shape).astype(np.float32) * (10.0 ** rng.uniform(-6, 1, shape)).astype(np.float32)
    g.reshape(-1)[::17] = 0.0
    return g


class Flat:
    """A 1-D slice [off, off + n) of a flat buffer pre-filled with a sentinel (a bias, or a range
    of the flat parameter buffer clipped to a shard boundary)."""

    def __init__(self, n, dtype, off, data):
        idt, self.pat = SENTINEL[dtype]
        self.raw = torch.full((off + n + 13,), self.pat, dtype=idt, device="cuda")
        self.off, self.n, self.dtype = off, n, dtype
        self.t = torch.as_strided(self.raw.view(dtype), (n,), (1,), off)
        self.t.copy_(torch.from_numpy(np.ascontiguousarray(data).reshape(n)).to(dtype))

    def bits(self):
        return Buf.bits(self)

    def get(self):
        return self.t.cpu().float().numpy()

    def check_sentinel(self, what=""):
        raw = self.raw.cpu().numpy()
        pat = np.array(self.pat).astype(raw.dtype)
        assert np.all(raw[: self.off] == pat) and np.all(raw[self.off + self.n:] == pat), what


@pytest.mark.parametrize("with_p16", [True, False])
@pytest.mark.parametrize("grad_scale", [1.0, 0.5])
def test_rmsprop(ops, grad_scale, with_p16):
    """Three steps of the Keras RMSprop(momentum) recurrence against fp64 (relative 1e-5 of the
    magnitudes involved), on 2-D padded views (padding untouched) and 1-D slices at base
    offsets 0-3 of lengths 1-9 and 10^5; p16 == bf16(p32) bit for bit."""
    rng = np.random.default_rng(90)
    lr, rho, mo, eps = (float(np.float32(v)) for v in (LR, RHO, MOM, EPS))
    cases = [(r, c, lay) for r, c in ((50, 103), (3, 9), (130, 1001), (7, 64))
             for lay in ("pad", "odd", "off1")]
    cases += [(0, n, off) for off in range(4) for n in list(range(1, 10)) + [100000]]
    for rows, cols, lay in cases:
        flat = rows == 0
        shape = (cols,) if flat else (rows, cols)
        what = f"{shape} {lay} scale {grad_scale}"

        def mk(dt, data):
            return Flat(cols, dt, lay, data) if flat else Buf(rows, cols, dt, lay, data)

        w0 = rng.standard_normal(shape).astype(np.float32)
        zero = np.zeros(shape, np.float32)
        bp, bs, bm, bg = mk(F32, w0), mk(F32, zero), mk(F32, zero), mk(F32, zero)
        b16 = mk(BF16, zero) if with_p16 else None
        w, s, m = w0.astype(np.float64), np.zeros(shape), np.zeros(shape)
        mom_abs, w_err = np.zeros(shape), np.zeros(shape)
        for step in range(3):
            g = _grads(rng, shape)
            bg.t.copy_(torch.from_numpy(g))
            ops.rmsprop_step(bp.t, None if b16 is None else b16.t, bg.t, bs.t, bm.t, LR, RHO, MOM,
                             EPS, grad_scale)
            g64 = g.astype(np.float64) * grad_scale
            w, s, m = R.rmsprop64(w, g64, s, m, lr, rho, mo, eps)
            mom_abs = mo * mom_abs + lr * np.abs(g64) / np.sqrt(s + eps)
            w_err += 1e-5 * mom_abs
            at = f"{what} step {step}"
            assert_within(bs.get(), s, 1e-5 * s, at + " ms")
            assert_within(bm.get(), m, 1e-5 * mom_abs, at + " mom")
            assert_within(bp.get(), w, 1e-5 * np.abs(w) + w_err, at + " w")
            if b16 is not None:
                assert np.array_equal(b16.bits(), R.bf16_bits(bp.get())), at + " p16"
        for b in (bp, bs, bm, bg) + ((b16,) if b16 is not None else ()):
            b.check_sentinel(what)


# ============================================================================ bias_act / fills
@pytest.mark.parametrize("layout", ["pad", "odd"])
@pytest.mark.parametrize("act", [0, 1, 2])
def test_bias_act(ops, act, layout):
    """y[r, c] = act(bias[c]) (Dense with zero input width): none and relu exact; sigmoid
    1 / (1 + __expf(-b)) within the __expf bound plus two roundings."""
    rng = np.random.default_rng(100 + act)
    for rows, cols in [(1, 1), (5, 8), (77, 515), (2048, 3)]:
        b = rng.standard_normal(cols, dtype=np.float32) * np.float32(5)
        b[: min(cols, 4)] = np.array([100, -100, 0, 1e-3], np.float32)[: min(cols, 4)]
        for with_bias in (True, False):
            bias = torch.from_numpy(b).cuda() if with_bias else None
            bv = b.astype(np.float64) if with_bias else np.zeros(cols)
            if act == 2:
                ref = np.maximum(bv, 0)
            elif act == 1:
                ref = R.sigmoid64(bv)
            else:
                ref = bv
            ref = np.broadcast_to(ref, (rows, cols))
            for want16, want32 in ((True, True), (True, False), (False, True)):
                o16 = Buf(rows, cols, BF16, layout) if want16 else None
                o32 = Buf(rows, cols, F32, layout) if want32 else None
                ops.bias_act(bias, act, rows, out16=o16.t if o16 else None,
                             out32=o32.t if o32 else None)
                what = f"act {act} bias {with_bias} {rows}x{cols}"
                for o in (o16, o32):
                    if o is None:
                        continue
                    if act != 1:
                        assert_bits(o, ref.astype(np.float32), what)
                    else:
                        e = 1 - ref        # = exp(-b) / (1 + exp(-b))
                        tol = (R.expf_rel_bound(bv) * e + 3 * U) * ref + ulp_of(o.dtype)(ref) + 2.0 ** -125
                        assert_within(o.get(), ref, tol, what)
                        o.check_sentinel(what)


def test_fill_and_counter_add(ops):
    for n in (1, 7, 1001, 70001):
        for off in (0, 1, 3):                 # "off" layouts: base 1 or 3 floats off alignment
            b = Buf(1, n, F32, ("pad", "off1", None, "off3")[off])
            flat = torch.as_strided(b.raw.view(F32), (n,), (1,), b.off)
            ops.fill_f32(flat, -2.5)
            assert torch.all(flat == -2.5)
            b.check_sentinel(f"fill {n} +{b.off}")
    c = torch.tensor([7, (1 << 32) - 1, 9], dtype=torch.int64, device="cuda")
    ops.counter_add(c[1:2], 1)
    assert c.tolist() == [7, 1 << 32, 9]
    ops.counter_add(c[1:2], 1 << 40)
    assert c.tolist() == [7, (1 << 40) + (1 << 32), 9]
    ops.counter_add(c[1:2], 0)
    assert c.tolist() == [7, (1 << 40) + (1 << 32), 9]
