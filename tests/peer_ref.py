"""Host references for the peer-memory optimiser and all-reduce (csrc/peer_optimizer.cu); no
GPU needed.

- The rank-order fp32 sum: sequential float32 additions starting from +0.0, g = ((0 + g_0) +
  g_1) + ..., exactly what both kernels do; other orders for showing that a test can see it.
- Gradients on which the order is observable from three ranks on.
- The modular epoch comparison of wait_flag and the epoch arithmetic of the entry points.
- The all-reduce's parity-slot addressing and the optimiser kernel's launch geometry.

The RMSprop recurrence and the bf16 helpers are tests/tail_ref.py's.
"""
import numpy as np

U32 = 1 << 32
PEER_MAX = 16


def rank_order_sum(terms):
    """terms [W, ...] float32 -> sum over the first axis as the kernels compute it."""
    terms = np.asarray(terms, np.float32)
    s = np.zeros(terms.shape[1:], np.float32)
    for t in terms:
        s = s + t
    return s


def reverse_order_sum(terms):
    return rank_order_sum(np.asarray(terms, np.float32)[::-1])


def pairwise_sum(terms):
    """Tree sum of adjacent pairs, from +0.0 like the kernels."""
    t = list(np.asarray(terms, np.float32))
    while len(t) > 1:
        t = [t[i] + t[i + 1] if i + 1 < len(t) else t[i] for i in range(0, len(t), 2)]
    return np.float32(0.0) + t[0]


def order_terms(rng, world, n, frac=0.5):
    """[world, n] float32 gradients and the mask of the elements built so that the fp32 sum
    depends on the order (world >= 3).  There g_0 = x = +-2^k, g_1 = +-0.75 * 2^(k-24) (same
    sign: lost when added to x, kept when added to -x, where the spacing halves), g_2 = -x and
    the rest are small values of fine granularity.  Elsewhere: normal values of magnitudes from
    1e-6 to 10, with exact zeros (some -0.0 on every rank)."""
    g = (rng.standard_normal((world, n), dtype=np.float32)
         * (10.0 ** rng.uniform(-6, 1, (world, n))).astype(np.float32))
    zero = np.zeros(n, bool)
    zero[3::23] = True
    g[:, zero] = 0.0
    g[:, 5::46] = -0.0
    mask = np.zeros(n, bool)
    if world >= 3:
        mask = (rng.random(n) < frac) & ~zero
        m = int(mask.sum())
        k = rng.integers(-4, 5, m)
        sign = np.where(rng.random(m) < 0.5, -1.0, 1.0)
        x = np.ldexp(sign, k).astype(np.float32)
        g[0, mask] = x
        g[1, mask] = np.ldexp(0.75 * sign, k - 24).astype(np.float32)
        g[2, mask] = -x
        if world > 3:
            fine = rng.standard_normal((world - 3, m)) * np.ldexp(1.0, k - 14)
            g[3:, mask] = fine.astype(np.float32)
    return g, mask


# ------------------------------------------------------------------------------------- epochs
def u32(v):
    return int(v) % U32


def as_i32(v):
    """A uint32 value as the int32 a torch flag / counter tensor stores."""
    v = u32(v)
    return v - U32 if v >= 1 << 31 else v


def effective_epoch(epoch, ctr=None):
    """epoch_rel + *epoch_ctr modulo 2^32 (ctr None: the host value alone)."""
    return u32(int(epoch) + (0 if ctr is None else int(ctr)))


def flag_reached(flag, epoch):
    """wait_flag's exit test: (int32)(flag - epoch) >= 0."""
    return as_i32(int(flag) - int(epoch)) >= 0


# ---------------------------------------------------------------------------------- all-reduce
def ar_parity(epoch):
    return u32(epoch) & 1


def ar_slot_offset(epoch, world, cap, src):
    """Element offset of slot [parity(epoch)][src] in a rank's [2][world][cap] staging array."""
    return ar_parity(epoch) * world * cap + src * cap


def ar_threads(n):
    """Block size of the all-reduce launch: n rounded up to a warp, at most 1024."""
    return 1024 if n >= 1024 else max(32, (n + 31) // 32 * 32)


# ------------------------------------------------------------------------- optimiser geometry
def blocks_per_sm(env_value):
    """CC_PEER_BLOCKS_PER_SM as the library parses it (atoi, default 2, clamped to [1, 8] by
    falling back to 2)."""
    if env_value is None:
        return 2
    s = env_value.strip()
    digits = ""
    for i, ch in enumerate(s):
        if ch.isdigit() or (i == 0 and ch in "+-"):
            digits += ch
        else:
            break
    try:
        v = int(digits)
    except ValueError:
        v = 0
    return v if 1 <= v <= 8 else 2


def rmsprop_grid(count, sms, per_sm):
    """Blocks of 256 threads cc_peer_rmsprop launches for `count` elements (8 per thread)."""
    return min((count // 8 + 255) // 256, sms * per_sm)


def rmsprop_passes(count, sms, per_sm):
    """Grid-stride passes of the launch (0 for an empty range: nothing is launched)."""
    n8 = count // 8
    if n8 == 0:
        return 0
    threads = rmsprop_grid(count, sms, per_sm) * 256
    return (n8 + threads - 1) // threads


def lo_mask(offsets, ranges):
    """Elements the kernel gives a low-order term: the 8-element group starting at off = start
    + 8 i is in when begin <= off < end for one of the (at most two) ranges."""
    group = np.asarray(offsets) // 8 * 8
    m = np.zeros(np.shape(offsets), bool)
    for a, b in ranges:
        m |= (group >= a) & (group < b)
    return m
