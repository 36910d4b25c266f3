"""Host references for the tail kernels (csrc/tail_kernels.cu); no GPU needed.

Three kinds:
- Philox-4x32-10 and the counter layout of the RNG kernels (dropout, dropout mask, uniform), a
  numpy port vectorised in uint64: the device streams must match it bit for bit.
- Exact helpers: bf16 round-to-nearest-even of fp32 values and the two-term split
  hi = bf16(x), lo = bf16(x - hi).
- fp64 references of the operations, written from the Keras formulas (SURVEY.md A.3-A.6), and
  the error bounds the fp32 kernels are held to.

The fp64 references take float64 numpy arrays; the BatchNormalization ones take an `xp`
module (numpy by default) so that they also run on float64 torch tensors.
"""
import numpy as np

U32 = np.uint64(0xFFFFFFFF)
PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85
FP32_U = 2.0 ** -24          # unit roundoff of fp32
EXPF_ULP_SLOPE = 1.173       # __expf(x): at most 2 + floor(1.173 |x|) ulp (CUDA C guide)


# --------------------------------------------------------------------------------- Philox
def philox_scalar(ctr, key):
    """One Philox-4x32-10 block with Python ints: ctr = 4 words, key = 2 words -> 4 words."""
    c, (k0, k1) = list(ctr), key
    m = 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = PHILOX_M0 * c[0], PHILOX_M1 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k0, p1 & m, (p0 >> 32) ^ c[3] ^ k1, p0 & m]
        k0, k1 = (k0 + PHILOX_W0) & m, (k1 + PHILOX_W1) & m
    return c


def philox_block(seed, ctr_hi, ctr_lo):
    """Philox::block of common.cuh, vectorised: seed is the 64-bit key, ctr_hi / ctr_lo the two
    64-bit counter halves (scalars or arrays, broadcast).  Returns uint64 array [..., 4] holding
    the four 32-bit output words."""
    seed = np.uint64(int(seed) & 0xFFFFFFFFFFFFFFFF)
    hi = np.asarray(ctr_hi, dtype=np.uint64)
    lo = np.asarray(ctr_lo, dtype=np.uint64)
    hi, lo = np.broadcast_arrays(hi, lo)
    c0, c1 = lo & U32, lo >> np.uint64(32)
    c2, c3 = hi & U32, hi >> np.uint64(32)
    k0, k1 = seed & U32, seed >> np.uint64(32)
    m0, m1 = np.uint64(PHILOX_M0), np.uint64(PHILOX_M1)
    w0, w1 = np.uint64(PHILOX_W0), np.uint64(PHILOX_W1)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2                     # < 2^64: exact in uint64
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & U32,
                          (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & U32)
        k0, k1 = (k0 + w0) & U32, (k1 + w1) & U32
    return np.stack([c0, c1, c2, c3], axis=-1)


def u32_to_unit(o):
    """u32_to_unit of common.cuh: the top 24 bits as a float32 in [0, 1)."""
    return ((np.asarray(o, dtype=np.uint64) >> np.uint64(8)).astype(np.float32)
            * np.float32(2.0 ** -24))


def rng_hi(step, stream_id):
    """High counter half of rng8: (stream_id << 40) ^ step in 64 bits.  stream_id is a uint32,
    so ids of 2^24 and above lose their top bits (they alias lower ids), and a step of 2^40 or
    more overlaps the id bits."""
    sid = int(stream_id) & 0xFFFFFFFF
    return ((sid << 40) ^ int(step)) & 0xFFFFFFFFFFFFFFFF


def rng_uniform(seed, step, stream_id, rows, cols):
    """u[r, c] of the RNG kernels: element (r, c) is lane c % 4 of Philox block
    r * ceil(cols / 4) + c // 4, key = seed, counter hi = rng_hi(step, stream_id).  The launch
    geometry does not enter."""
    bpr = (cols + 3) // 4
    blocks = (np.arange(rows, dtype=np.uint64)[:, None] * np.uint64(bpr)
              + np.arange(bpr, dtype=np.uint64)[None, :])
    o = philox_block(seed, np.uint64(rng_hi(step, stream_id)), blocks)   # [rows, bpr, 4]
    return u32_to_unit(o.reshape(rows, bpr * 4)[:, :cols])


def keep_mask(u, rate):
    return u >= np.float32(rate)


def dropout_scale(rate):
    """1.f / (1.f - rate) as the kernel computes it (fp32)."""
    return np.float32(1.0) / (np.float32(1.0) - np.float32(rate))


def dropout_ref(x32, keep, rate):
    """x * keep / (1 - rate) as the kernel computes it: x * scale in fp32, +0 where dropped."""
    out = np.asarray(x32, np.float32) * dropout_scale(rate)
    return np.where(keep, out, np.float32(0.0)).astype(np.float32)


# ------------------------------------------------------------------------------ bf16 / split
def bf16_bits(x32):
    """uint16 bit patterns of bf16 round-to-nearest-even of fp32 values (NaN stays NaN)."""
    b = np.ascontiguousarray(x32, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = (b + np.uint64(0x7FFF) + ((b >> np.uint64(16)) & np.uint64(1))) >> np.uint64(16)
    nan = np.isnan(np.asarray(x32, dtype=np.float32))
    r = np.where(nan, (b >> np.uint64(16)) | np.uint64(0x40), r)
    return r.astype(np.uint16)


def bf16_from_bits(h):
    return (np.asarray(h, dtype=np.uint16).astype(np.uint32) << np.uint32(16)).view(np.float32)


def bf16_round(x32):
    """fp32 -> bf16 (round to nearest even) -> fp32."""
    return bf16_from_bits(bf16_bits(x32))


def split_ref(x32):
    """Two-term bf16 expansion: hi = bf16(x), lo = bf16(x - hi) (x - hi is exact in fp32)."""
    x32 = np.asarray(x32, np.float32)
    hi = bf16_round(x32)
    return hi, bf16_round(x32 - hi)


def ulp32(x):
    """Spacing of fp32 numbers at |x| (the subnormal spacing below the normal range)."""
    a = np.maximum(np.abs(np.asarray(x, np.float64)), 2.0 ** -126)
    return 2.0 ** (np.floor(np.log2(a)) - 23)


def ulp16(x):
    a = np.maximum(np.abs(np.asarray(x, np.float64)), 2.0 ** -126)
    return 2.0 ** (np.floor(np.log2(a)) - 7)


# ---------------------------------------------------------------------- elementwise formulas
def act_grad_f32(dy32, y32, act):
    """dz = dy * act'(y) as the kernels compute it in fp32 (act: 0 none, 1 sigmoid, 2 relu);
    sigmoid' is y * (1 - y) of the stored output."""
    dy32, y32 = np.asarray(dy32, np.float32), np.asarray(y32, np.float32)
    if act == 1:
        return dy32 * (y32 * (np.float32(1.0) - y32))
    if act == 2:
        return dy32 * np.where(y32 > 0, np.float32(1.0), np.float32(0.0))
    return dy32.copy()


def act_grad64(dy, y, act):
    if act == 1:
        return dy * y * (1.0 - y)
    if act == 2:
        return dy * (y > 0)
    return dy


def sigmoid64(x):
    return 1.0 / (1.0 + np.exp(-x))


def expf_rel_bound(d):
    """Relative error bound of the fp32 __expf(d) the kernels use, d = x - max already rounded
    in fp32: 2 + floor(1.173 |d|) ulp of the result (ulp <= 2^-23 relative), plus the
    rounding of the subtraction d = x - max (relative 2^-24 of d moves exp by |d| 2^-24)."""
    d = np.abs(np.asarray(d, np.float64))
    return (2.0 + np.floor(EXPF_ULP_SLOPE * d)) * 2.0 ** -23 + d * FP32_U


# ----------------------------------------------------------------------- column reductions
def colreduce_grid(rows, cols, sms):
    """(column blocks, row slabs, rows per slab) of the column-reduction launch."""
    gx = (cols + 127) // 128
    gy = 1
    target = 2 * sms
    if gx < target:
        gy = (target + gx - 1) // gx
        gy = max(1, min(gy, (rows + 63) // 64))
    return gx, gy, (rows + gy - 1) // gy


def colreduce_adds(rows, cols, sms):
    """Additions on the longest path from one term to a column total: each thread sums
    ceil(rows_per_slab / 8) rows, then the 8 row groups of a CTA, then the slabs."""
    _, gy, rps = colreduce_grid(rows, cols, sms)
    return (rps + 7) // 8 + 8 + gy


def sum_bound(abs_sum, n_adds, term_roundings=0):
    """|fp32 recursive sum - exact| <= (n_adds + roundings per term) * u * sum |term|."""
    return (n_adds + term_roundings) * FP32_U * abs_sum


# ---------------------------------------------------------------------------- BatchNorm
def bn_moments64(x):
    """Two-pass fp64 batch statistics (tf.nn.moments): mean, biased variance per column."""
    mean = x.sum(0) / x.shape[0]
    d = x - mean
    return mean, (d * d).sum(0) / x.shape[0]


def bn_train64(x, gamma, beta, eps, xp=np):
    mean, var = bn_moments64(x)
    rstd = 1.0 / xp.sqrt(var + eps)
    return (x - mean) * rstd * gamma + beta, mean, rstd, var


def bn_train_bwd64(dy, x, gamma, eps, xp=np):
    """Gradients of y = (x - mean(x)) / sqrt(var(x) + eps) * gamma + beta (batch statistics) by
    the closed form of the chain rule: dx, dgamma, dbeta."""
    n = x.shape[0]
    mean, var = bn_moments64(x)
    rstd = 1.0 / xp.sqrt(var + eps)
    xhat = (x - mean) * rstd
    dbeta = dy.sum(0)
    dgamma = (dy * xhat).sum(0)
    dx = gamma * rstd * (dy - dbeta / n - xhat * dgamma / n)
    return dx, dgamma, dbeta


def moving_update64(moving, batch, momentum):
    """Keras moving statistics: moving * momentum + batch * (1 - momentum)."""
    return moving * momentum + batch * (1.0 - momentum)


# ------------------------------------------------------------------------- softmax / argmax
def softmax64(x):
    e = np.exp(x - x.max(-1)[..., None])
    return e / e.sum(-1)[..., None]


def softmax_bwd64(dy, y):
    return y * (dy - (dy * y).sum(-1)[..., None])


def onehot_argmax(p):
    """to_categorical(argmax(p, -1)): the first maximum wins."""
    p = np.asarray(p)
    out = np.zeros(p.shape, np.float32)
    out[np.arange(p.shape[0]), np.argmax(p, axis=-1)] = 1.0
    return out


# --------------------------------------------------------------------------------- losses
BCE_EPS32 = np.float32(1e-7)     # Keras backend epsilon, clip bounds as fp32 [eps, 1 - eps]


def bce_logits64(x, t):
    """tf.nn.sigmoid_cross_entropy_with_logits per element."""
    return np.maximum(x, 0.0) - x * t + np.log1p(np.exp(-np.abs(x)))


def bce_probs64(p, t):
    """Keras binary_crossentropy on probabilities clipped to [eps, 1 - eps] (fp32 bounds)."""
    q = np.clip(p, float(BCE_EPS32), float(np.float32(1.0) - BCE_EPS32))
    return -(t * np.log(q) + (1.0 - t) * np.log1p(-q))


def mse64(pred, target, n_total):
    d = pred - target
    return (d * d).sum() / (n_total * pred.shape[1]), 2.0 * d / (n_total * pred.shape[1])


# -------------------------------------------------------------------------------- RMSprop
def rmsprop64(w, g, ms, mom, lr, rho, momentum, eps):
    """Keras RMSprop with momentum (SURVEY.md A.6); returns the new (w, ms, mom)."""
    ms = rho * ms + (1.0 - rho) * g * g
    mom = momentum * mom + lr * g / np.sqrt(ms + eps)
    return w - mom, ms, mom


def round_half_even(x):
    return np.rint(x)


def fallback_cols(sms):
    """Width of a 1 x N row whose 8-column chunks outnumber the threads of the largest
    elementwise launch (8 blocks of 256 threads per SM): for_each_chunk8's grid-stride walk."""
    return 8 * (8 * sms * 256) + 13


def isclose_ulp(got, ref, n_ulp=1.0, ulp=ulp32):
    return np.abs(np.asarray(got, np.float64) - ref) <= n_ulp * ulp(ref)

