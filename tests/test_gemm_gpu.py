"""tcgen05 GEMM (cc_gemm through the C ABI) against a plain PyTorch fp32 reference.

Floating-point kernel => torch fp32 reference of the same op on the same bf16-rounded inputs.
Tolerance: fp32 accumulation of bf16 products, so |err| <= 2e-3 * sqrt(K) * scale for fp32
outputs, plus one bf16 rounding (rel 2^-8) for bf16 outputs.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ops():
    from cellcomm_b200 import ops
    return ops


def _rand(rows, cols, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    t = (torch.randn(rows, cols, generator=g) * scale).to(torch.bfloat16)
    return t


def _dev2d(t_cpu, ops):
    """copy into a padded device buffer, return the [rows, cols] view"""
    out = ops.alloc2d(t_cpu.shape[0], t_cpu.shape[1], dtype=t_cpu.dtype)
    out.copy_(t_cpu)
    return out


def _check(got, ref, K, bf16_out, scale=1.0):
    got = got.float().cpu()
    ref = ref.float().cpu()
    atol = 2e-3 * (K ** 0.5) * scale + 1e-5
    rtol = 2 ** -7 if bf16_out else 1e-4
    err = (got - ref).abs()
    bound = atol + rtol * ref.abs()
    bad = (err > bound).sum().item()
    assert bad == 0, (f"{bad} / {err.numel()} elements off; max err {err.max().item():.4g} "
                      f"max ref {ref.abs().max().item():.4g}")


SHAPES = [
    (128, 128, 64),
    (128, 256, 128),
    (256, 384, 512),
    (200, 300, 1000),
    (77, 50, 33),
    (3, 1, 10),
    (130, 1684, 3369),
]


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("bn", [128, 256])
def test_dgrad_orientation_k_major(M, N, K, bn):
    """A [M,K] K-major, B [N,K] K-major (dX = dZ W^T)."""
    ops = _ops()
    a, b = _rand(M, K, 1), _rand(N, K, 2)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    out = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, [da], [db], [K], 0, 0, out32=out, bn=bn)
    torch.cuda.synchronize()
    _check(out, a.float() @ b.float().t(), K, False)


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("bn", [128, 256])
def test_fwd_orientation_b_mn_major(M, N, K, bn):
    """A [M,K] K-major, B [K,N] MN-major (Y = X W)."""
    ops = _ops()
    a, b = _rand(M, K, 3), _rand(K, N, 4)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    out = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, [da], [db], [K], 0, 1, out32=out, bn=bn)
    torch.cuda.synchronize()
    _check(out, a.float() @ b.float(), K, False)


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("bn", [128, 256])
def test_wgrad_orientation_both_mn_major(M, N, K, bn):
    """A stored [K,M], B stored [K,N] (dW = X^T dZ)."""
    ops = _ops()
    a, b = _rand(K, M, 5), _rand(K, N, 6)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    out = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, [da], [db], [K], 1, 1, out32=out, bn=bn)
    torch.cuda.synchronize()
    _check(out, a.float().t() @ b.float(), K, False)


def test_a_mn_b_k_major():
    ops = _ops()
    M, N, K = 192, 160, 200
    a, b = _rand(K, M, 7), _rand(N, K, 8)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    out = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, [da], [db], [K], 1, 0, out32=out)
    torch.cuda.synchronize()
    _check(out, a.float().t() @ b.float().t(), K, False)


@pytest.mark.parametrize("persistent", ["1", "0"])
@pytest.mark.parametrize("orient", ["fwd", "dgrad", "wgrad"])
@pytest.mark.parametrize("M,N,ks,splits", [(128, 300, (4000,), 5), (300, 100, (700, 1300), 6),
                                           (520, 1100, (2048, 2048, 2048), 24), (130, 257, (320, 64, 640), 16)])
def test_split_k_work_units(M, N, ks, splits, orient, persistent, monkeypatch):
    """Split-K as work units of the persistent kernel (tile x k-range; CC_GEMM_PERSISTENT_SPLITK=1,
    the default) and in the one-tile-per-CTA kernel (=0): all operand-major combinations,
    several accumulating segments whose boundaries fall inside a k-range, more k-ranges than
    k-blocks per segment, several row tiles (2-CTA clusters), N <= 128 (the 128-wide
    instantiation), bias + activation applied by the finalize pass.  Both kernels sum the same
    partials in the same order: bit-identical results."""
    ops = _ops()
    outs = []
    for mode in (persistent, "0"):
        monkeypatch.setenv("CC_GEMM_PERSISTENT_SPLITK", mode)
        As, Bs, ref = [], [], 0
        for i, k in enumerate(ks):
            if orient == "fwd":       # A [M,k] K-major, B [k,N] MN-major
                a, b = _rand(M, k, 20 + i, 0.3), _rand(k, N, 30 + i, 0.3)
                ref = ref + a.float() @ b.float()
            elif orient == "dgrad":   # A [M,k], B [N,k]: both K-major
                a, b = _rand(M, k, 20 + i, 0.3), _rand(N, k, 30 + i, 0.3)
                ref = ref + a.float() @ b.float().t()
            else:                     # A [k,M], B [k,N]: both MN-major
                a, b = _rand(k, M, 20 + i, 0.3), _rand(k, N, 30 + i, 0.3)
                ref = ref + a.float().t() @ b.float()
            As.append(_dev2d(a, ops))
            Bs.append(_dev2d(b, ops))
        bias = torch.randn(N, generator=torch.Generator().manual_seed(3)).cuda()
        out16 = ops.alloc2d(M, N)
        out32 = torch.full((M, ops.pad_ld(N)), 7.0, device="cuda")[:, :N]
        a_mn, b_mn = {"fwd": (0, 1), "dgrad": (0, 0), "wgrad": (1, 1)}[orient]
        ops.gemm(M, N, As, Bs, list(ks), a_mn, b_mn, bias=bias, act=ops.ACT_RELU, out16=out16,
                 out32=out32, splits=splits)
        torch.cuda.synchronize()
        want = torch.relu(ref + bias.cpu())
        _check(out32, want, sum(ks), False, scale=0.1)
        _check(out16, want, sum(ks), True, scale=0.1)
        assert float((out32.as_strided((M, ops.pad_ld(N)), (ops.pad_ld(N), 1))[:, N:] - 7.0).abs().sum()) == 0
        outs.append(out32.clone())
    if persistent == "1":
        assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("splits", [2, 3, 7])
def test_split_k(splits):
    ops = _ops()
    M, N, K = 128, 300, 4000
    a, b = _rand(M, K, 9), _rand(K, N, 10)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    bias = torch.randn(N, device="cuda")
    out16 = ops.alloc2d(M, N)
    out32 = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, [da], [db], [K], 0, 1, bias=bias, act=ops.ACT_RELU, out16=out16, out32=out32,
             splits=splits)
    torch.cuda.synchronize()
    ref = torch.relu(a.float() @ b.float() + bias.cpu())
    _check(out32, ref, K, False)
    _check(out16, ref, K, True)


def test_auto_split_k_small_m_long_k():
    ops = _ops()
    M, N, K = 128, 512, 33694
    a, b = _rand(M, K, 11, 0.1), _rand(K, N, 12, 0.1)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    out32 = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, [da], [db], [K], 0, 1, out32=out32)
    torch.cuda.synchronize()
    _check(out32, a.float() @ b.float(), K, False, scale=0.01)


def test_concat_segments_forward():
    """[h1, x] @ W without materialising the concat (E2/Dx2 in the reference nets)."""
    ops = _ops()
    M, N = 150, 200
    ks = [100, 333, 6]
    xs = [_rand(M, k, 20 + i) for i, k in enumerate(ks)]
    w = _rand(sum(ks), N, 30)
    dxs = [_dev2d(x, ops) for x in xs]
    dw = _dev2d(w, ops)
    bias = torch.randn(N, device="cuda")
    out16 = ops.alloc2d(M, N)
    ops.dense_fwd(dxs, dw, [0, 100, 433], bias, ops.ACT_SIGMOID, out16=out16)
    torch.cuda.synchronize()
    ref = torch.sigmoid(torch.cat([x.float() for x in xs], 1) @ w.float() + bias.cpu())
    _check(out16, ref, sum(ks), True)


def test_dgrad_with_act_derivative_and_accumulate():
    ops = _ops()
    M, K, N = 140, 260, 90
    dz, w = _rand(M, N, 40), _rand(K, N, 41)
    y = torch.sigmoid(_rand(M, K, 42).float()).to(torch.bfloat16)
    prev = _rand(M, K, 43)
    ddz, dw, dy = _dev2d(dz, ops), _dev2d(w, ops), _dev2d(y, ops)
    out = _dev2d(prev, ops)
    ops.dense_dgrad([ddz], [dw], out, dact_y=dy, dact=ops.ACT_SIGMOID, alpha=0.5, beta=1)
    torch.cuda.synchronize()
    ref = prev.float() + 0.5 * (dz.float() @ w.float().t()) * (y.float() * (1 - y.float()))
    _check(out, ref, N, True)


def test_dgrad_two_segments():
    """d(cell) = dZ1 W1^T + dZ2 W2x^T (sub-step 1 of trainings_step through D's skip concat)."""
    ops = _ops()
    M, K = 100, 500
    n1, n2 = 300, 120
    dz1, dz2 = _rand(M, n1, 50), _rand(M, n2, 51)
    w1, w2 = _rand(K, n1, 52), _rand(K + 40, n2, 53)
    out = ops.alloc2d(M, K)
    dw2 = _dev2d(w2, ops)
    ops.dense_dgrad([_dev2d(dz1, ops), _dev2d(dz2, ops)], [_dev2d(w1, ops), dw2[40:]], out)
    torch.cuda.synchronize()
    ref = dz1.float() @ w1.float().t() + dz2.float() @ w2[40:].float().t()
    _check(out, ref, n1 + n2, True)


def test_wgrad_into_row_block_and_beta():
    ops = _ops()
    B, K, N = 128, 200, 170
    x, dz = _rand(B, K, 60), _rand(B, N, 61)
    dw = ops.alloc2d(K + 30, N, dtype=torch.float32)
    dw.fill_(1.0)
    ops.dense_wgrad(_dev2d(x, ops), _dev2d(dz, ops), dw[30:], beta=1)
    torch.cuda.synchronize()
    ref = 1.0 + x.float().t() @ dz.float()
    _check(dw[30:], ref, B, False)
    assert torch.all(dw[:30] == 1.0)


def test_large_batch_shapes():
    ops = _ops()
    M, N, K = 1024, 1024, 2048
    a, b = _rand(M, K, 70), _rand(K, N, 71)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    out16 = ops.alloc2d(M, N)
    ops.gemm(M, N, [da], [db], [K], 0, 1, out16=out16)
    torch.cuda.synchronize()
    _check(out16, a.float() @ b.float(), K, True)


@pytest.mark.parametrize("K,N,B", [(200, 170, 128), (700, 40, 64), (129, 513, 300)])
def test_wgrad_with_fused_rmsprop_epilogue(K, N, B):
    """dW = X^T dZ consumed in the epilogue by Keras RMSprop(momentum): parameters, slots and
    the bf16 copy are updated in place; the gradient is optionally also written."""
    ops = _ops()
    x, dz = _rand(B, K, 80, 0.5), _rand(B, N, 81, 0.01)
    ld = ops.pad_ld(N)
    dev = "cuda"
    w0 = torch.randn(K, N) * 0.05
    ms0 = torch.rand(K, N) * 1e-4
    mom0 = torch.randn(K, N) * 1e-3
    mk = lambda t, dt=torch.float32: (lambda b: (b.copy_(t), b)[1])(
        torch.zeros(K, ld, dtype=dt, device=dev)[:, :N])
    p32, ms, mom = mk(w0), mk(ms0), mk(mom0)
    p16 = torch.zeros(K, ld, dtype=torch.bfloat16, device=dev)[:, :N]
    dw = torch.zeros(K, ld, device=dev)[:, :N]
    lr, rho, mo, eps = 0.0075, 0.85, 0.1, 1e-7
    ops.dense_wgrad(_dev2d(x, ops), _dev2d(dz, ops), dw, rms=(p32, p16, ms, mom, lr, rho, mo, eps))
    torch.cuda.synchronize()
    g = x.float().t() @ dz.float()
    _check(dw, g, B, False, scale=0.005)
    g = dw.cpu()                      # the kernel's own fp32 gradient
    ms_ref = rho * ms0 + (1 - rho) * g * g
    mom_ref = mo * mom0 + lr * g / torch.sqrt(ms_ref + eps)
    assert torch.allclose(ms.cpu(), ms_ref, rtol=1e-5, atol=1e-12)
    assert torch.allclose(mom.cpu(), mom_ref, rtol=1e-4, atol=1e-8)
    assert torch.allclose(p32.cpu(), w0 - mom_ref, rtol=1e-5, atol=1e-7)
    assert torch.equal(p16, p32.to(torch.bfloat16))
    # without a gradient output
    p32b, msb, momb = mk(w0), mk(ms0), mk(mom0)
    ops.dense_wgrad(_dev2d(x, ops), _dev2d(dz, ops), None,
                    rms=(p32b, None, msb, momb, lr, rho, mo, eps))
    torch.cuda.synchronize()
    assert torch.equal(p32b, p32) and torch.equal(msb, ms)


@pytest.mark.parametrize("nfast", ["0", "1"])
@pytest.mark.parametrize("K,N,B", [(1000, 1300, 256), (385, 2049, 96), (64, 300, 40),
                                   (700, 520, 2048)])
def test_fused_rmsprop_epilogue_paths(K, N, B, nfast, monkeypatch):
    """The fused-optimiser epilogue with row-major state (the register path of the generic
    persistent kernel) on both tile rasters, several row / column tiles with ragged edges, a
    single row tile (K = 64: no cluster), a long batch reduction (32 k-blocks: the operand ring
    wraps many times), with and without the bf16 copy, with and without the gradient output.
    Padding must stay untouched."""
    ops = _ops()
    monkeypatch.setenv("CC_GEMM_RMS_NFAST", nfast)
    x, dz = _rand(B, K, 90, 0.5), _rand(B, N, 91, 0.01)
    ld = ops.pad_ld(N)
    w0 = torch.randn(K, N) * 0.05
    ms0 = torch.rand(K, N) * 1e-4
    mom0 = torch.randn(K, N) * 1e-3
    lr, rho, mo, eps = 0.0075, 0.85, 0.1, 1e-7

    def mk(t, dt=torch.float32):
        full = torch.full((K, ld), 7.0, dtype=dt, device="cuda")
        full[:, :N].copy_(t)
        return full

    g = x.float().t() @ dz.float()
    ms_ref = rho * ms0 + (1 - rho) * g * g
    mom_ref = mo * mom0 + lr * g / torch.sqrt(ms_ref + eps)
    for with16, with_grad in ((True, False), (False, True), (True, True)):
        p32f, msf, momf = mk(w0), mk(ms0), mk(mom0)
        p16f = torch.full((K, ld), 7.0, dtype=torch.bfloat16, device="cuda")
        dwf = torch.full((K, ld), 7.0, device="cuda")
        ops.dense_wgrad(_dev2d(x, ops), _dev2d(dz, ops), dwf[:, :N] if with_grad else None,
                        rms=(p32f[:, :N], p16f[:, :N] if with16 else None, msf[:, :N], momf[:, :N],
                             lr, rho, mo, eps))
        torch.cuda.synchronize()
        # bf16 operands, fp32 accumulation: the gradient itself is checked loosely, the update
        # arithmetic against the kernel's own gradient where available
        assert torch.allclose(msf[:, :N].cpu(), ms_ref, rtol=2e-2, atol=1e-9)
        assert torch.allclose(momf[:, :N].cpu(), mom_ref, rtol=2e-2, atol=2e-5)
        assert torch.allclose(p32f[:, :N].cpu(), w0 - mom_ref, rtol=0, atol=3e-5)
        if with_grad:
            gk = dwf[:, :N].cpu()
            _check(dwf[:, :N], g, B, False, scale=0.005)
            ms_k = rho * ms0 + (1 - rho) * gk * gk
            mom_k = mo * mom0 + lr * gk / torch.sqrt(ms_k + eps)
            assert torch.allclose(msf[:, :N].cpu(), ms_k, rtol=1e-5, atol=1e-12)
            assert torch.allclose(momf[:, :N].cpu(), mom_k, rtol=1e-4, atol=1e-8)
            assert torch.allclose(p32f[:, :N].cpu(), w0 - mom_k, rtol=1e-5, atol=1e-7)
            assert float((dwf[:, N:] - 7.0).abs().sum()) == 0.0
        if with16:
            assert torch.equal(p16f[:, :N], p32f[:, :N].to(torch.bfloat16))
        # padding columns: untouched
        for t in (p32f, msf, momf, p16f):
            assert float((t[:, N:].float() - 7.0).abs().sum()) == 0.0


@pytest.mark.parametrize("nfast", ["0", "1"])
@pytest.mark.parametrize("K0,K1,N,B", [(300, 500, 1300, 256), (70, 0, 2049, 96), (1000, 333, 520, 2048),
                                       (33, 31, 257, 128)])
def test_fused_rmsprop_blocked_state(K0, K1, N, B, nfast, monkeypatch):
    """Fused optimiser with the fp32 state in the BLOCKED layout (cc_gemm_desc.rms_blocked): a
    layer of K0 + K1 rows updated by two weight-gradient GEMMs (Concatenate segments; the second
    starts at a row that is not a multiple of 32, so its lanes wrap across block rows), ragged
    N, short and long batch reductions, both rasters, with and without the gradient output.
    The result, converted back to rows, must equal the row-major register path's (same
    accumulators, same arithmetic up to FMA contraction); the gradient output is bit-identical;
    padding rows and padding columns of the state stay zero."""
    ops = _ops()
    monkeypatch.setenv("CC_GEMM_RMS_NFAST", nfast)
    K = K0 + K1
    R, ld = (K + 31) // 32 * 32, ops.pad_ld(N)
    lr, rho, mo, eps = 0.0075, 0.85, 0.1, 1e-7
    gen = torch.Generator().manual_seed(5)

    def rows(scale, positive=False):
        t = torch.zeros(R, ld)
        v = torch.rand(K, N, generator=gen) if positive else torch.randn(K, N, generator=gen)
        t[:K, :N] = v * scale
        return t.cuda()

    w0, ms0, mom0 = rows(0.05), rows(1e-4, True), rows(1e-3)
    xs = [_rand(B, k, 90 + i, 0.5) if k else None for i, k in enumerate((K0, K1))]
    dz = _rand(B, N, 93, 0.01)
    for with_grad in (False, True):
        # reference: the row-major register path on the same inputs
        ref = [t.clone() for t in (w0, ms0, mom0)]
        ref16 = torch.zeros(R, ld, dtype=torch.bfloat16, device="cuda")
        refdw = torch.full((R, ld), 7.0, device="cuda")
        blk = [ops.state_rows_to_blocked(t).contiguous() for t in (w0, ms0, mom0)]
        assert torch.equal(ops.state_blocked_to_rows(blk[0], R, ld), w0)
        p16 = torch.full((R, ld), 7.0, dtype=torch.bfloat16, device="cuda")
        dw = torch.full((R, ld), 7.0, device="cuda")
        lo16 = torch.full((R, ld), 7.0, dtype=torch.bfloat16, device="cuda")
        ro = 0
        for x, k in zip(xs, (K0, K1)):
            if k == 0:
                continue
            sl = slice(ro, ro + k)
            ops.dense_wgrad(_dev2d(x, ops), _dev2d(dz, ops), refdw[sl, :N] if with_grad else None,
                            rms=(ref[0][sl, :N], ref16[sl, :N], ref[1][sl, :N], ref[2][sl, :N],
                                 lr, rho, mo, eps))
            ops.dense_wgrad(_dev2d(x, ops), _dev2d(dz, ops), dw[sl, :N] if with_grad else None,
                            rms=(blk[0], p16[sl, :N], blk[1], blk[2], lr, rho, mo, eps), rms_row0=ro,
                            rms_lo=lo16[sl, :N] if with_grad else None)
            ro += k
        torch.cuda.synchronize()
        # same accumulators as the row-major path; the update expressions may be contracted
        # into FMAs differently by the compiler: a few ulp
        for b, r_, tol in zip(blk, ref, (1e-7, 1e-12, 1e-8)):
            got = ops.state_blocked_to_rows(b, R, ld)
            assert torch.allclose(got, r_, rtol=2e-5, atol=tol), float((got - r_).abs().max())
            assert float(got[K:].abs().sum()) == 0.0 and float(got[:, N:].abs().sum()) == 0.0
            assert torch.equal(got == 0, r_ == 0)
        assert float((p16[:K, :N].float() - ref16[:K, :N].float()).abs().max()) <= 1e-3
        assert torch.equal(p16[:K, :N], ops.state_blocked_to_rows(blk[0], R, ld)[:K, :N].to(torch.bfloat16))
        # the bf16 copy is written in whole 32-column chunks: padding columns up to the next
        # multiple of 32 receive bf16(0) (the engine's padding is zero), nothing beyond, no other row
        edge = min(ld, (N + 31) // 32 * 32)
        assert float((p16[:, edge:].float() - 7.0).abs().sum()) == 0.0
        assert float((p16[K:].float() - 7.0).abs().sum()) == 0.0
        assert bool(((p16[:K, N:edge] == 7.0) | (p16[:K, N:edge] == 0.0)).all())
        if with_grad:
            # low-order term of the hi + lo kernels: bf16(w - float(bf16(w))), exactly
            w_new = ops.state_blocked_to_rows(blk[0], R, ld)[:K, :N]
            assert torch.equal(lo16[:K, :N], (w_new - p16[:K, :N].float()).to(torch.bfloat16))
            assert float((lo16[K:].float() - 7.0).abs().sum()) == 0.0
            assert float((lo16[:, edge:].float() - 7.0).abs().sum()) == 0.0
            assert torch.equal(dw[:K, :N], refdw[:K, :N])
            assert float(dw[:K, N:edge].abs().sum()) == 0.0
            assert float((dw[:, edge:] - 7.0).abs().sum()) == 0.0 and float((dw[K:] - 7.0).abs().sum()) == 0.0


@pytest.mark.parametrize("bn_eff", [128, 160, 192, 224, 256])
@pytest.mark.parametrize("orient", ["fwd", "dgrad", "wgrad"])
def test_effective_tile_width(bn_eff, orient, monkeypatch):
    """Persistent kernel with a narrower effective tile (wave-quantisation heuristic of
    gemm_sm100.cu): every candidate width, all three operand-major combinations, N not a
    multiple of the width, bias + activation epilogue."""
    ops = _ops()
    monkeypatch.setenv("CC_GEMM_BN_EFF", str(bn_eff))
    M, N, K = 300, 1000, 200
    bias = torch.randn(N, device="cuda")
    if orient == "fwd":
        a, b = _rand(M, K, 21), _rand(K, N, 22)
        ref, am, bm = a.float() @ b.float(), 0, 1
    elif orient == "dgrad":
        a, b = _rand(M, K, 23), _rand(N, K, 24)
        ref, am, bm = a.float() @ b.float().t(), 0, 0
    else:
        a, b = _rand(K, M, 25), _rand(K, N, 26)
        ref, am, bm = a.float().t() @ b.float(), 1, 1
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    out16 = ops.alloc2d(M, N)
    out32 = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, [da], [db], [K], am, bm, bias=bias, act=ops.ACT_SIGMOID, out16=out16,
             out32=out32, use_ws=False)
    torch.cuda.synchronize()
    ref = torch.sigmoid(ref + bias.cpu())
    _check(out32, ref, K, False)
    _check(out16, ref, K, True)


@pytest.mark.parametrize("orient", ["fwd", "dgrad", "wgrad"])
@pytest.mark.parametrize("M,N,K,segs", [(300, 1000, 200, 1), (1000, 517, 2100, 1), (257, 264, 70, 1),
                                        (640, 2300, 96, 3)])
def test_cluster_multicast_mma(M, N, K, segs, orient, monkeypatch):
    """The 2-CTA multicast scheme (two CTAs on vertically adjacent tiles, each loading half of
    the shared B tile into both) against the fp32 product: all three operand-major
    combinations, odd row-tile counts (the second CTA of the last pair idles), ragged N, a long
    reduction that wraps the ring, and several accumulating segments."""
    ops = _ops()
    monkeypatch.setenv("CC_GEMM_BN_EFF", "256")
    bias = torch.randn(N, device="cuda")
    a_list, b_list, ref = [], [], 0
    for sgi in range(segs):
        if orient == "fwd":
            a, b = _rand(M, K, 41 + sgi), _rand(K, N, 51 + sgi)
            ref, am, bm = ref + a.float() @ b.float(), 0, 1
        elif orient == "dgrad":
            a, b = _rand(M, K, 43 + sgi), _rand(N, K, 53 + sgi)
            ref, am, bm = ref + a.float() @ b.float().t(), 0, 0
        else:
            a, b = _rand(K, M, 45 + sgi), _rand(K, N, 55 + sgi)
            ref, am, bm = ref + a.float().t() @ b.float(), 1, 1
        a_list.append(_dev2d(a, ops))
        b_list.append(_dev2d(b, ops))
    out16 = ops.alloc2d(M, N)
    out32 = ops.alloc2d(M, N, dtype=torch.float32)
    ops.gemm(M, N, a_list, b_list, [K] * segs, am, bm, bias=bias, act=ops.ACT_SIGMOID, out16=out16,
             out32=out32, use_ws=False)
    torch.cuda.synchronize()
    want = torch.sigmoid(ref + bias.cpu())
    _check(out32, want, K * segs, False)
    _check(out16, want, K * segs, True)


def test_effective_tile_width_auto_matches_full_width(monkeypatch):
    """The heuristic's pick (here 192 for N = 3369 at 16 row tiles) gives the same result as
    the full 256-wide tile."""
    ops = _ops()
    M, N, K = 2048, 3369, 320
    a, b = _rand(M, K, 31), _rand(K, N, 32)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    outs = []
    for forced in ("0", "256"):
        monkeypatch.setenv("CC_GEMM_BN_EFF", forced)
        o = ops.alloc2d(M, N, dtype=torch.float32)
        ops.gemm(M, N, [da], [db], [K], 0, 1, out32=o, use_ws=False)
        torch.cuda.synchronize()
        outs.append(o.cpu())
    assert torch.equal(outs[0], outs[1])
    _check(outs[0], a.float() @ b.float(), K, False)


def test_routed_wgrad_output_two_ranks_emulated():
    """cc_gemm_desc.route_*: the wgrad epilogue stores every element of dW to the staging
    buffer of the rank that owns it in the sharded optimiser (here both "ranks" live on one
    device).  Bucket = this GEMM's rows plus a neighbouring region before it; the shard
    boundary falls in the middle of a row."""
    ops = _ops()
    M, N, K = 300, 200, 192                     # dW[M, N] = X[K, M]^T dZ[K, N]
    ld = ops.pad_ld(N)                          # 256
    a, b = _rand(K, M, 41), _rand(K, N, 42)
    da, db = _dev2d(a, ops), _dev2d(b, ops)
    before = 1024                               # elements of the bucket ahead of this piece
    total = before + M * ld
    W = 2
    shard = (total // W + 7) // 8 * 8           # owner boundary inside row (shard-before)//ld
    stage = [torch.full((total,), float("nan"), device="cuda") for _ in range(W)]
    local = stage[0][before:].view(M, ld)[:, :N]            # "my" gradient view (rank 0 = me)
    ops.dense_wgrad([da], [db], local, route=(W, shard, before, [t.data_ptr() for t in stage]))
    torch.cuda.synchronize()
    ref = torch.full((M, ld), float("nan"))
    ref[:, :N] = a.float().t() @ b.float()
    flat_ref = torch.cat([torch.full((before,), float("nan")), ref.flatten()])
    owner = torch.clamp(torch.arange(total) // shard, max=W - 1)
    for r in range(W):
        got = stage[r].cpu()
        mine = (owner == r) & ~torch.isnan(flat_ref)
        assert torch.isnan(got[~mine]).all(), f"rank {r}: wrote outside its share"
        assert torch.allclose(got[mine], flat_ref[mine], rtol=1e-4, atol=2e-3 * K ** 0.5)
    assert (owner == 1).any() and ((owner == 0) & ~torch.isnan(flat_ref)).any()
