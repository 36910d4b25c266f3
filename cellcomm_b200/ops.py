"""Thin torch-tensor wrappers over the C ABI (include/cellcomm_b200.h).

PyTorch is plumbing here: it owns device memory and the current CUDA stream; every function
passes raw pointers + leading dimensions to libcellcomm_b200.so.  2-D tensors may be strided
views (stride(1) == 1), so column slices of padded buffers are passed without copies.

There is deliberately NO fallback: on a tensor that is not on a CUDA device, or when the
library is missing, these raise.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import GemmDesc, check

COMPUTE_DTYPE = torch.bfloat16   # GEMM operand / activation dtype
ACT_NONE, ACT_SIGMOID, ACT_RELU = 0, 1, 2
ACT_IDS = {None: 0, "none": 0, "linear": 0, "sigmoid": 1, "relu": 2}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _req(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise RuntimeError(f"cellcomm_b200.ops: {name} must be a CUDA tensor (no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"cellcomm_b200.ops: {name} must be {dtype}, got {t.dtype}")
    if t.dim() == 2 and t.shape[1] > 1 and t.stride(1) != 1:
        raise ValueError(f"cellcomm_b200.ops: {name} must be row-major (stride(1)==1)")


def _p(t):
    return None if t is None else t.data_ptr()


def _ld(t):
    if t is None:
        return 0
    if t.dim() == 1:
        return t.shape[0]
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def pad_ld(cols, mult=64):
    """Leading dimension used for activations / weights: multiple of 64 elements (128 B rows)."""
    return max(mult, (cols + mult - 1) // mult * mult)


def alloc2d(rows, cols, dtype=torch.bfloat16, device="cuda", zero=True):
    """[rows, cols] view of a zero-initialised [rows, pad_ld(cols)] buffer."""
    ld = pad_ld(cols)
    buf = (torch.zeros if zero else torch.empty)((max(rows, 1), ld), dtype=dtype, device=device)
    return buf[:rows, :cols]


_WS = {}


def workspace(device):
    """Per-device split-K scratch (fp32)."""
    key = str(device)
    ws = _WS.get(key)
    if ws is None:
        ws = torch.empty(296 * 128 * 256 * 2, dtype=torch.float32, device=device)
        _WS[key] = ws
    return ws


def launch_count():
    return int(_lib.load().cc_launch_count())


def reload_env():
    """Make the library re-read its CC_GEMM_* environment knobs (it reads them once)."""
    _lib.load().cc_reload_env()


# --------------------------------------------------------------------------- GEMM
def gemm(M, N, a_list, b_list, k_list, a_mn, b_mn, *, bias=None, act=0, dact_y=None, dact=0,
         alpha=1.0, out16=None, beta16=0, out32=None, beta32=0, splits=0, bn=0, use_ws=True,
         rms=None, route=None, out16_lo=None, rms_row0=None, rms_lo=None):
    lib = _lib.load()
    d = GemmDesc()
    d.M, d.N = int(M), int(N)
    d.a_mn_major, d.b_mn_major = int(a_mn), int(b_mn)
    d.nseg = len(a_list)
    for s, (a, b, k) in enumerate(zip(a_list, b_list, k_list)):
        _req(a, torch.bfloat16, "A")
        _req(b, torch.bfloat16, "B")
        d.a[s], d.lda[s] = a.data_ptr(), _ld(a)
        d.b[s], d.ldb[s] = b.data_ptr(), _ld(b)
        d.k[s] = int(k)
    d.alpha = float(alpha)
    _req(bias, torch.float32, "bias")
    d.bias = _p(bias)
    d.act = int(act)
    _req(dact_y, torch.bfloat16, "dact_y")
    d.dact_y, d.ld_dact, d.dact = _p(dact_y), _ld(dact_y), int(dact)
    _req(out16, torch.bfloat16, "out16")
    _req(out32, torch.float32, "out32")
    d.out16, d.ld16, d.beta16 = _p(out16), _ld(out16), int(beta16)
    d.out32, d.ld32, d.beta32 = _p(out32), _ld(out32), int(beta32)
    if out16_lo is not None:
        _req(out16_lo, torch.bfloat16, "out16_lo")
        if out16 is None or beta16:
            raise ValueError("gemm(out16_lo=...): needs a plain bf16 out16 (the high-order term)")
        d.out16_lo, d.ld16_lo = out16_lo.data_ptr(), _ld(out16_lo)
    if use_ws:
        ws = workspace(a_list[0].device)
        d.workspace, d.workspace_elems = ws.data_ptr(), ws.numel()
    d.force_splits, d.force_bn = int(splits), int(bn)
    if rms is not None and rms_row0 is not None:
        # blocked optimiser state (cc_gemm_desc.rms_blocked): p32 / ms / mom are the LAYER's flat
        # blocked arrays, p16 the row-major [M, N] slice this GEMM updates, rms_row0 its first
        # layer row
        p32, p16, ms, mom, lr, rho, momentum, eps = rms
        _req(p16, torch.bfloat16, "p16")
        if p16 is None or tuple(p16.shape) != (M, N):
            raise ValueError("gemm(rms=..., rms_row0=...): needs the [M, N] bf16 copy")
        ld = _ld(p16)
        need = (int(rms_row0) + M + 31) // 32 * 32 * ld
        for t, name in ((p32, "p32"), (ms, "ms"), (mom, "mom")):
            _req(t, torch.float32, name)
            if t.dim() != 1 or t.numel() < need:
                raise ValueError(f"gemm(rms_row0=...): {name} must be the layer's flat blocked array "
                                 f"of at least {need} elements")
        d.rms_p32, d.rms_ms, d.rms_mom, d.rms_p16 = p32.data_ptr(), ms.data_ptr(), \
            mom.data_ptr(), p16.data_ptr()
        d.rms_ld, d.rms_blocked, d.rms_row0 = ld, 1, int(rms_row0)
        if rms_lo is not None:          # low-order bf16 term of the updated weights
            _req(rms_lo, torch.bfloat16, "rms_lo")
            if tuple(rms_lo.shape) != (M, N) or _ld(rms_lo) != ld:
                raise ValueError("gemm(rms_lo=...): must be laid out like the bf16 copy")
            d.rms_p16_lo = rms_lo.data_ptr()
        d.rms_lr, d.rms_rho, d.rms_momentum, d.rms_eps = float(lr), float(rho), float(momentum), \
            float(eps)
    elif rms is not None:
        if rms_lo is not None:
            raise ValueError("gemm(rms_lo=...): only with the blocked state layout (rms_row0)")
        p32, p16, ms, mom, lr, rho, momentum, eps = rms
        for t, name in ((p32, "p32"), (ms, "ms"), (mom, "mom")):
            _req(t, torch.float32, name)
            if tuple(t.shape) != (M, N) or _ld(t) != _ld(p32):
                raise ValueError("gemm(rms=...): parameter / slot views must be [M, N] with one ld")
        d.rms_p32, d.rms_ms, d.rms_mom, d.rms_p16 = p32.data_ptr(), ms.data_ptr(), \
            mom.data_ptr(), _p(p16)
        if p16 is not None and _ld(p16) != _ld(p32):
            raise ValueError("gemm(rms=...): p16 must share the parameter's leading dimension")
        d.rms_ld = _ld(p32)
        d.rms_lr, d.rms_rho, d.rms_momentum, d.rms_eps = float(lr), float(rho), float(momentum), \
            float(eps)
    if route is not None:
        world, shard, off0, bases = route
        if out32 is None or beta32:
            raise ValueError("gemm(route=...): needs a plain fp32 output")
        d.route_world, d.route_shard, d.route_off0 = int(world), int(shard), int(off0)
        for q in range(world):
            d.route_base[q] = int(bases[q])
        d.workspace, d.workspace_elems = None, 0       # routed tiles are never split along K
    check(lib.cc_gemm(C.byref(d), _stream()))


def dense_fwd(xs, w16, row_offsets, bias, act, out16=None, out32=None, hi_lo=None):
    """out = act(sum_s xs[s] @ w16[roff_s : roff_s + xs[s].shape[1], :] + bias).

    xs: list of [M, K_s] bf16 (Concatenate segments, consumed without materialising);
    w16: [K_total, N] bf16 Keras-layout kernel.  Dense forward, src/bigan_classify.py:10-75."""
    ws = list(w16) if isinstance(w16, (list, tuple)) else [w16] * len(xs)   # per-segment kernels
    M, N = xs[0].shape[0], ws[0].shape[1]
    bs = [w[ro:ro + x.shape[1]] for x, w, ro in zip(xs, ws, row_offsets)]
    if out16 is not None and out16.dtype == torch.float32:   # fp32 activation (feeds a BN)
        if out32 is not None:
            raise ValueError("dense_fwd: two fp32 outputs")
        out16, out32 = None, out16
    lo = None
    if hi_lo is not None:       # (hi, lo): also emit the output's two-term bf16 expansion
        if out16 is not None:
            raise ValueError("dense_fwd: hi_lo goes with an fp32 output")
        out16, lo = hi_lo
    gemm(M, N, xs, bs, [x.shape[1] for x in xs], 0, 1, bias=bias, act=act, out16=out16, out32=out32,
         out16_lo=lo)


def dense_dgrad(dzs, ws16, out, *, dact_y=None, dact=0, alpha=1.0, beta=0):
    """out[M,K] (+)= alpha * (sum_s dzs[s] @ ws16[s]^T) * act'(dact_y); ws16[s]: [K, N_s].
    `out` is fp32 (activation gradients) or bf16."""
    M, K = out.shape
    kw = ({"out32": out, "beta32": beta} if out.dtype == torch.float32
          else {"out16": out, "beta16": beta})
    gemm(M, K, dzs, ws16, [dz.shape[1] for dz in dzs], 0, 0, dact_y=dact_y, dact=dact, alpha=alpha,
         **kw)


def state_rows_to_blocked(rows):
    """[R, ld] row-major fp32 (R % 32 == 0, ld % 32 == 0) -> the flat blocked order of
    cc_gemm_desc.rms_blocked: 32 x 32 blocks of 4 KB, inside a block (column group of 4, row,
    column in group)."""
    R, ld = rows.shape
    return rows.reshape(R // 32, 32, ld // 32, 8, 4).permute(0, 2, 3, 1, 4).reshape(-1)


def state_blocked_to_rows(flat, R, ld):
    """Inverse of state_rows_to_blocked -> [R, ld] row-major (a copy)."""
    return flat.reshape(R // 32, ld // 32, 8, 32, 4).permute(0, 3, 1, 2, 4).reshape(R, ld)


def dense_wgrad(x, dz, dw32, beta=0, rms=None, route=None, rms_row0=None, rms_lo=None):
    """dw32[K,N] (+)= x[M,K]^T @ dz[M,N].  x may be a list [hi, lo] (bf16 expansion): the
    terms accumulate as GEMM segments along the batch reduction.
    rms = (p32, p16, ms, mom, lr, rho, momentum, eps): fuse the Keras RMSprop update of that
    [K,N] parameter block into the epilogue (dw32 may then be None: the gradient is consumed
    in registers and never written).  With rms_row0 the fp32 state is the layer's BLOCKED
    arrays (state_rows_to_blocked) and this GEMM's rows start at layer row rms_row0; rms_lo
    (blocked only) also receives the low-order bf16 term of the updated weights."""
    K, N = (dw32.shape if dw32 is not None else rms[1 if rms_row0 is not None else 0].shape)
    xs = list(x) if isinstance(x, (list, tuple)) else [x]
    dzs = list(dz) if isinstance(dz, (list, tuple)) else [dz] * len(xs)
    # tiny layers (one or two output tiles, reduction over the whole batch) take the split-K
    # path; the fused-optimiser epilogue cannot be split
    # route = (world, shard, off0, bases): the epilogue stores every element of dw32 to the rank
    # that owns it in the sharded optimiser (see cc_gemm_desc.route_*)
    gemm(K, N, xs, dzs, [t.shape[0] for t in xs], 1, 1, out32=dw32, beta32=beta,
         use_ws=rms is None and route is None, rms=rms, route=route, rms_row0=rms_row0,
         rms_lo=rms_lo)


# --------------------------------------------------------------------------- data
def gather_rows(rowptr, colidx, values, n_cols, *, row_idx=None, row_start=0, n_rows=None,
                out16=None, out32=None):
    lib = _lib.load()
    _req(rowptr, torch.int64, "rowptr")
    _req(colidx, torch.int32, "colidx")
    _req(values, torch.float32, "values")
    _req(row_idx, torch.int64, "row_idx")
    _req(out16, torch.bfloat16, "out16")
    _req(out32, torch.float32, "out32")
    if n_rows is None:
        n_rows = row_idx.shape[0]
    check(lib.cc_gather_rows(rowptr.data_ptr(), colidx.data_ptr(), values.data_ptr(), _p(row_idx),
                             int(row_start), int(n_rows), int(n_cols), _p(out16), _ld(out16),
                             _p(out32), _ld(out32), _stream()))


def encode_scratch_bytes(plan):
    return int(_lib.load().cc_encode_scratch_bytes(C.byref(plan)))


def encode_stream(rowptr, colidx, values, row_begin, row_end, plan, out32):
    """The encode-all-cells pass over CSR rows [row_begin, row_end) in one C call
    (cc_encode_stream); plan: _lib.EncodePlan built by BiGanEngine.encode_plan()."""
    _req(rowptr, torch.int64, "rowptr")
    _req(colidx, torch.int32, "colidx")
    _req(values, torch.float32, "values")
    _req(out32, torch.float32, "out32")
    if out32.shape[0] != row_end - row_begin:
        raise ValueError("encode_stream: out32 must have one row per encoded cell")
    check(_lib.load().cc_encode_stream(rowptr.data_ptr(), colidx.data_ptr(), values.data_ptr(),
                                       int(row_begin), int(row_end), C.byref(plan),
                                       out32.data_ptr(), _ld(out32), _stream()))


# --------------------------------------------------------------------------- tail kernels
def _act_t(t, name):
    """bf16-or-fp32 activation operand"""
    if t is None:
        return
    if not t.is_cuda:
        raise RuntimeError(f"cellcomm_b200.ops: {name} must be a CUDA tensor (no CPU fallback)")
    if t.dtype not in (torch.bfloat16, torch.float32):
        raise TypeError(f"cellcomm_b200.ops: {name} must be bf16 or fp32, got {t.dtype}")
    if t.dim() == 2 and t.shape[1] > 1 and t.stride(1) != 1:
        raise ValueError(f"cellcomm_b200.ops: {name} must be row-major (stride(1)==1)")


def _mask(*ts):
    """dtypes bitmask of the C ABI: bit i set when the i-th activation operand is fp32"""
    m = 0
    for i, t in enumerate(ts):
        _act_t(t, f"operand {i}")
        if t is not None and t.dtype == torch.float32:
            m |= 1 << i
    return m


def reduce_ws_floats(rows, cols):
    """fp32 elements of a fixed-order reduction workspace that serves every `ws=` call below
    on at most rows x cols (zero it once before the first use; one workspace per stream)."""
    return int(_lib.load().cc_reduce_ws_floats(int(rows), int(cols)))


def _ws(ws):
    """(pointer, floats) of a fixed-order reduction workspace; ws=None: the atomic path"""
    if ws is None:
        return None, 0
    _req(ws, torch.float32, "ws")
    if not ws.is_contiguous():
        raise ValueError("cellcomm_b200.ops: ws must be contiguous")
    return ws.data_ptr(), ws.numel()


# colsum / bias_grad / bn_stats / bn_bwd_stats / mse_fwd_bwd: with ws (a zeroed fp32 buffer of
# reduce_ws_floats elements) the partial sums combine in a fixed order, so the result is
# bit-identical from run to run; without it they combine with atomics.
def colsum(x, out32, beta=0, *, ws=None):
    _req(out32, torch.float32, "out")
    check(_lib.load().cc_colsum_ws(_p(x), _ld(x), x.shape[0], x.shape[1], _p(out32), int(beta),
                                   _mask(x), *_ws(ws), _stream()))


def bias_grad(dy, y, act, out32, dz=None, beta=0, dz_lo=None, *, ws=None):
    """out32[c] (+)= sum_r dy[r,c] * act'(y[r,c])  (Dense bias gradient from the fp32 gradient);
    dz (optional): also store dy * act'(y) there (one pass instead of act_bwd + bias_grad);
    dz_lo (optional): and its low-order bf16 term (dz then holds the high-order one).
    out32 = None: only dz (/ dz_lo) is produced."""
    _req(out32, torch.float32, "out")
    _req(dz_lo, torch.bfloat16, "dz_lo")
    check(_lib.load().cc_bias_grad_ws(_p(dy), _ld(dy), _p(y), _ld(y), dy.shape[0], dy.shape[1],
                                      int(act), _p(out32), int(beta), _p(dz), _ld(dz), _p(dz_lo),
                                      _ld(dz_lo), _mask(dy, y, dz), *_ws(ws), _stream()))


def split_bf16(x, hi, lo):
    """hi + lo ~= x with hi, lo in bf16 (two accumulating GEMM segments)."""
    _req(hi, torch.bfloat16, "hi")
    _req(lo, torch.bfloat16, "lo")
    check(_lib.load().cc_split_bf16(_p(x), _ld(x), _p(hi), _ld(hi), _p(lo), _ld(lo), x.shape[0],
                                    x.shape[1], _mask(x), _stream()))


def dropout(x, out, rate, *, mask=None, seed=0, counter=None, stream_id=0):
    _req(mask, torch.uint8, "mask")
    _req(counter, torch.int64, "counter")
    check(_lib.load().cc_dropout(_p(x), _ld(x), _p(out), _ld(out), x.shape[0], x.shape[1],
                                 float(rate), _p(mask), _ld(mask), int(seed), _p(counter),
                                 int(stream_id), _mask(x, out), _stream()))


def dropout_mask(mask, rate, *, seed=0, counter=None, stream_id=0):
    _req(mask, torch.uint8, "mask")
    check(_lib.load().cc_dropout_mask(_p(mask), _ld(mask), mask.shape[0], mask.shape[1],
                                      float(rate), int(seed), _p(counter), int(stream_id),
                                      _stream()))


def uniform(out32=None, out16=None, *, seed=0, counter=None, stream_id=0):
    t = out32 if out32 is not None else out16
    _req(out32, torch.float32, "out32")
    _req(out16, torch.bfloat16, "out16")
    if out32 is not None and out16 is not None and _ld(out32) != _ld(out16):
        raise ValueError("uniform: out32/out16 must share a leading dimension")
    check(_lib.load().cc_uniform(_p(out32), _p(out16), _ld(t), t.shape[0], t.shape[1], int(seed),
                                 _p(counter), int(stream_id), _stream()))


def counter_add(counter, inc=1):
    check(_lib.load().cc_counter_add(_p(counter), int(inc), _stream()))


def act_bwd(dy, y, dz, act):
    check(_lib.load().cc_act_bwd(_p(dy), _ld(dy), _p(y), _ld(y), _p(dz), _ld(dz), dy.shape[0],
                                 dy.shape[1], int(act), _mask(dy, y, dz), _stream()))


def copy2d(src, dst, beta=0, scale=1.0):
    """dst (+)= scale*src; also the bf16<->fp32 cast."""
    check(_lib.load().cc_copy2d(_p(src), _ld(src), _p(dst), _ld(dst), src.shape[0], src.shape[1],
                                int(beta), float(scale), _mask(src, dst), _stream()))


def cast_f32_to_bf16(src32, dst16):
    copy2d(src32, dst16)


def cast_bf16_to_f32(src16, dst32, scale=1.0):
    copy2d(src16, dst32, scale=scale)


def bn_stats(x, sums, *, ws=None):
    check(_lib.load().cc_bn_stats_ws(_p(x), _ld(x), x.shape[0], x.shape[1], _p(sums), _mask(x),
                                     *_ws(ws), _stream()))


def bn_train_apply(x, y, sums, n_total, gamma, beta, eps, momentum, moving_mean, moving_var,
                   save_mean, save_rstd):
    check(_lib.load().cc_bn_train_apply(_p(x), _ld(x), _p(y), _ld(y), x.shape[0], x.shape[1],
                                        _p(sums), int(n_total), _p(gamma), _p(beta), float(eps),
                                        float(momentum), _p(moving_mean), _p(moving_var),
                                        _p(save_mean), _p(save_rstd), _mask(x, y), _stream()))


def bn_infer(x, y, gamma, beta, moving_mean, moving_var, eps):
    check(_lib.load().cc_bn_infer(_p(x), _ld(x), _p(y), _ld(y), x.shape[0], x.shape[1], _p(gamma),
                                  _p(beta), _p(moving_mean), _p(moving_var), float(eps),
                                  _mask(x, y), _stream()))


def bn_bwd_stats(dy, x, save_mean, save_rstd, sums2, *, ws=None):
    check(_lib.load().cc_bn_bwd_stats_ws(_p(dy), _ld(dy), _p(x), _ld(x), dy.shape[0],
                                         dy.shape[1], _p(save_mean), _p(save_rstd), _p(sums2),
                                         _mask(dy, x), *_ws(ws), _stream()))


def bn_bwd_apply(dy, x, dx, gamma, save_mean, save_rstd, sums2, n_total, dgamma=None, dbeta=None):
    check(_lib.load().cc_bn_bwd_apply(_p(dy), _ld(dy), _p(x), _ld(x), _p(dx), _ld(dx), dy.shape[0],
                                      dy.shape[1], _p(gamma), _p(save_mean), _p(save_rstd),
                                      _p(sums2), int(n_total), _p(dgamma), _p(dbeta),
                                      _mask(dy, x, dx), _stream()))


def bn_infer_bwd(dy, dx, gamma, moving_var, eps):
    check(_lib.load().cc_bn_infer_bwd(_p(dy), _ld(dy), _p(dx), _ld(dx), dy.shape[0], dy.shape[1],
                                      _p(gamma), _p(moving_var), float(eps), _mask(dy, dx),
                                      _stream()))


def softmax_fwd(x, y16=None, y32=None):
    _req(y32, torch.float32, "y32")
    check(_lib.load().cc_softmax_fwd(_p(x), _ld(x), _p(y16), _ld(y16), _p(y32), _ld(y32),
                                     x.shape[0], x.shape[1], _mask(x, y16), _stream()))


def softmax_bwd(dy, y, dx):
    check(_lib.load().cc_softmax_bwd(_p(dy), _ld(dy), _p(y), _ld(y), _p(dx), _ld(dx), dy.shape[0],
                                     dy.shape[1], _mask(dy, y, dx), _stream()))


def bce_fwd_bwd(x32, target, n_total, loss_out, dz=None, from_logits=True):
    _req(x32, torch.float32, "x")
    _req(loss_out, torch.float32, "loss_out")
    check(_lib.load().cc_bce_fwd_bwd(_p(x32), _ld(x32), x32.shape[0], int(bool(from_logits)),
                                     float(target), int(n_total), _p(loss_out), _p(dz), _ld(dz),
                                     _mask(dz), _stream()))


def mse_fwd_bwd(pred, n_total, loss_out, *, target, dpred=None, ws=None):
    _req(loss_out, torch.float32, "loss_out")
    check(_lib.load().cc_mse_fwd_bwd_ws(_p(pred), _ld(pred), _p(target), _ld(target),
                                        pred.shape[0], pred.shape[1], int(n_total), _p(loss_out),
                                        _p(dpred), _ld(dpred), _mask(pred, target, dpred),
                                        *_ws(ws), _stream()))


def round_half_even(x, out16=None, out32=None):
    _req(out32, torch.float32, "out32")
    check(_lib.load().cc_round_half_even(_p(x), _ld(x), _p(out16), _ld(out16), _p(out32),
                                         _ld(out32), x.shape[0], x.shape[1], _mask(x, out16),
                                         _stream()))


def argmax_onehot(p32, out16=None, out32=None):
    _req(p32, torch.float32, "p32")
    check(_lib.load().cc_argmax_onehot(_p(p32), _ld(p32), _p(out16), _ld(out16), _p(out32),
                                       _ld(out32), p32.shape[0], p32.shape[1], _stream()))


def rmsprop_step(p32, p16, g, ms, mom, lr, rho, momentum, eps, grad_scale=1.0):
    """In-place Keras RMSprop(momentum) on a [rows, cols] view; all fp32 views share p32's ld."""
    rows, cols = (p32.shape[0], p32.shape[1]) if p32.dim() == 2 else (1, p32.shape[0])
    ld = _ld(p32) if p32.dim() == 2 else cols
    for t in (g, ms, mom):
        if (t.dim() == 2 and _ld(t) != ld) or t.shape != p32.shape:
            raise ValueError("rmsprop_step: gradient/slots must share the parameter's layout")
    if p16 is not None and p16.dim() == 2 and _ld(p16) != ld:
        raise ValueError("rmsprop_step: p16 must share the parameter's leading dimension")
    check(_lib.load().cc_rmsprop_step(_p(p32), _p(p16), _p(g), _p(ms), _p(mom), rows, cols, ld,
                                      float(lr), float(rho), float(momentum), float(eps),
                                      float(grad_scale), _stream()))


def bias_act(bias, act, rows, out16=None, out32=None):
    t = out16 if out16 is not None else out32
    check(_lib.load().cc_bias_act(_p(bias), int(act), _p(out16), _ld(out16), _p(out32), _ld(out32),
                                  int(rows), t.shape[1], _stream()))


def fill_f32(t, value):
    check(_lib.load().cc_fill_f32(_p(t), float(value), t.numel(), _stream()))


# --------------------------------------------------------------------------- peer-memory optimiser
def peer_rmsprop(world, rank, grad_ptrs, p16_ptrs, p32, ms, mom, start, count, broadcast, lr, rho,
                 momentum, eps, ready_ptr, epoch, p16_multicast=0, epoch_ctr=None, lo=None):
    """Fused reduce-scatter -> Keras RMSprop -> bf16 all-gather over NVLink peer memory for the
    flat element range [start, start+count).  grad_ptrs / p16_ptrs: device pointers (ints) of
    every rank's flat gradient / bf16 weight buffer; p32, ms, mom: this rank's flat buffers."""
    for t, name in ((p32, "p32"), (ms, "ms"), (mom, "mom")):
        _req(t, torch.float32, name)
    d = _lib.PeerRmspropDesc()
    d.world, d.rank = int(world), int(rank)
    for q in range(world):
        d.grad[q], d.p16[q] = int(grad_ptrs[q]), int(p16_ptrs[q])
    d.p32, d.ms, d.mom = p32.data_ptr(), ms.data_ptr(), mom.data_ptr()
    d.start, d.count, d.broadcast = int(start), int(count), int(bool(broadcast))
    d.lr, d.rho, d.momentum, d.eps = float(lr), float(rho), float(momentum), float(eps)
    d.ready, d.epoch = int(ready_ptr), int(epoch) & 0xFFFFFFFF
    d.p16_multicast = int(p16_multicast) or None
    d.epoch_ctr = _p(epoch_ctr)
    if lo is not None:
        # lo = (p16lo_ptrs, p16lo_multicast, [(begin, end), ...]): low-order terms of the
        # kernels kept as hi + lo (at most two flat ranges)
        lo_ptrs, lo_mc, ranges = lo
        if len(ranges) > 2:
            raise ValueError("peer_rmsprop: at most two hi+lo ranges")
        for q in range(world):
            d.p16lo[q] = int(lo_ptrs[q])
        d.p16lo_multicast = int(lo_mc) or None
        for k, (a, b) in enumerate(ranges):
            d.lo_begin[k], d.lo_end[k] = int(a), int(b)
    check(_lib.load().cc_peer_rmsprop(C.byref(d), _stream()))


def peer_signal(target_ptrs, value, epoch_ctr=None):
    """After everything this stream has done so far, store `value` (+ *epoch_ctr) to every flag."""
    arr = (C.c_void_p * len(target_ptrs))(*[int(p) for p in target_ptrs])
    check(_lib.load().cc_peer_signal(arr, len(target_ptrs), int(value) & 0xFFFFFFFF,
                                     _p(epoch_ctr), _stream()))


def peer_wait(flags_ptr, n, value, epoch_ctr=None, bump=False):
    """Block the stream until n consecutive local uint32 flags are >= value (+ *epoch_ctr);
    bump: then advance the counter to that epoch."""
    check(_lib.load().cc_peer_wait(int(flags_ptr), int(n), int(value) & 0xFFFFFFFF, _p(epoch_ctr),
                                   int(bool(bump)), _stream()))


def peer_allreduce(data, world, rank, slot_ptrs, flag_ptrs, cap, epoch, epoch_ctr=None):
    """In-place sum all-reduce of a small contiguous fp32 tensor over peer memory (one kernel);
    with epoch_ctr the kernel uses epoch + *epoch_ctr and leaves that value in the counter."""
    _req(data, torch.float32, "data")
    if not data.is_contiguous():
        raise ValueError("peer_allreduce: data must be contiguous")
    sl = (C.c_void_p * world)(*[int(p) for p in slot_ptrs])
    fl = (C.c_void_p * world)(*[int(p) for p in flag_ptrs])
    check(_lib.load().cc_peer_allreduce(data.data_ptr(), data.numel(), int(world), int(rank), sl, fl,
                                        int(cap), int(epoch) & 0xFFFFFFFF, _p(epoch_ctr),
                                        _stream()))
