"""cc_peer_rmsprop, cc_peer_allreduce and cc_peer_signal / cc_peer_wait (csrc/peer_optimizer.cu)
bit for bit, with W emulated ranks on one GPU; the real fabric through tests/peer_gpu_worker.py.

Every "rank" is a set of ordinary device buffers and its peer pointers are the other sets'
data_ptr()s.  Every buffer sits in a NaN-sentinel allocation with PAD elements of padding on
either side, and each check compares the whole allocation, padding included.

References (tests/peer_ref.py, tests/tail_ref.py): the rank-order fp32 sum on the host, with
gradients built so that the order is observable from three ranks on; the RMSprop result is
`ops.rmsprop_step` on that sum (bit for bit) and within tail_ref's fp64 bound.

Safety: wait_flag traps after ~10 s, so everything runs on one stream in protocol order and every
launch that waits goes through `guard`: it synchronises, reads the awaited flags and the rank's
epoch counter, and fails the test WITHOUT launching unless every awaited flag has reached the
effective epoch.  A broken kernel therefore shows as wrong bits, never as a spinning kernel.
"""
import os

import numpy as np
import pytest
import torch

import peer_ref as P
import tail_ref as R

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LR, RHO, MOM, EPS = 0.0075, 0.85, 0.1, 1e-7          # engine.LR, RHO, MOMENTUM, EPSILON
F32, BF16, I32 = torch.float32, torch.bfloat16, torch.int32
PAD = 64
# sentinel bit patterns: NaNs with a payload no kernel writes; flags get a large positive value
SENT = {F32: (torch.int32, 0x7FC0DEAD), BF16: (torch.int16, 0x7FC1), I32: (torch.int32, 0x5A5A5A5A)}


@pytest.fixture(scope="module")
def ops():
    from cellcomm_b200 import ops
    return ops


@pytest.fixture(scope="module")
def geom():
    """(SMs, blocks per SM) of cc_peer_rmsprop's grid cap.  The library reads
    CC_PEER_BLOCKS_PER_SM once per process (cc_reload_env does not reset it), so it is read the
    same way here rather than set."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return sms, P.blocks_per_sm(os.environ.get("CC_PEER_BLOCKS_PER_SM"))


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda() if isinstance(x, np.ndarray) else x


class Flat:
    """n elements of dtype at element PAD of an allocation filled with SENT[dtype]; `raw` (the
    whole allocation as integers) may be given, e.g. a symmetric-memory buffer."""

    def __init__(self, n, dtype, data=None, raw=None):
        idt, pat = SENT[dtype]
        if raw is None:
            raw = torch.empty(n + 2 * PAD, dtype=idt, device="cuda")
        self.raw = raw.view(idt)
        self.raw.fill_(pat)
        self.t = self.raw.view(dtype)[PAD:PAD + n]
        self.n, self.dtype = n, dtype
        if data is not None:
            self.t.copy_(_dev(data))

    @property
    def ptr(self):
        return self.t.data_ptr()


def bf16_dev(x32):
    """bf16 bit patterns (tail_ref's round-to-nearest-even) of fp32 host values, on the device."""
    return _dev(R.bf16_bits(x32).view(np.int16))


def assert_bits(got, want, what):
    if torch.equal(got, want):
        return
    bad = (got != want).nonzero().flatten()
    i = int(bad[0])
    raise AssertionError(f"{what}: {bad.numel()} of {got.numel()} differ, first at element "
                         f"{i - PAD} (got {int(got[i]) & 0xFFFFFFFF:#x}, "
                         f"want {int(want[i]) & 0xFFFFFFFF:#x})")


def with_range(raw, lo, hi, vals):
    """A copy of the raw allocation with view elements [lo, hi) replaced by vals (raw ints)."""
    out = raw.clone()
    out[PAD + lo:PAD + hi] = vals
    return out


def ctr_tensor(v):
    return None if v is None else torch.tensor([P.as_i32(v)], dtype=I32, device="cuda")


def ctr_value(ctr):
    return None if ctr is None else P.u32(int(ctr.item()))


# --------------------------------------------------------------------------- guarded launches
def guard(flags, idx, epoch, ctr, what):
    """Synchronise; fail (launching nothing) unless the int32 flags[idx] have all reached the
    effective epoch (+ *ctr, modulo 2^32, as wait_flag compares).  Returns that epoch."""
    torch.cuda.synchronize()
    e = P.effective_epoch(epoch, ctr_value(ctr))
    vals = flags.cpu().tolist()
    late = [(i, P.u32(vals[i])) for i in idx if not P.flag_reached(vals[i], e)]
    if late:
        pytest.fail(f"{what}: flags (index, value) {late} have not reached epoch {e}; not launched")
    return e


def run_rmsprop(ops, W, r, grad_ptrs, p16_ptrs, state, start, count, broadcast, ready, ready_off,
                epoch, ctr, lo=None, mc=0):
    """cc_peer_rmsprop for rank r; ready: rank r's int32 flag array, ready_off: index of the
    bucket's first flag in it."""
    guard(ready, range(ready_off, ready_off + W), epoch, ctr, f"rank {r} peer_rmsprop")
    p32, ms, mom = state
    ops.peer_rmsprop(W, r, grad_ptrs, p16_ptrs, p32, ms, mom, start, count, broadcast, LR, RHO, MOM,
                     EPS, ready.data_ptr() + 4 * ready_off, epoch, p16_multicast=mc,
                     epoch_ctr=ctr, lo=lo)


def run_allreduce(ops, data, W, r, slot_ptrs, flag_ptrs, my_flags, cap, epoch, ctr=None):
    """Rank r's kernel raises its own flag itself; it waits for every other rank's."""
    e = guard(my_flags, [q for q in range(W) if q != r], epoch, ctr, f"rank {r} peer_allreduce")
    ops.peer_allreduce(data, W, r, slot_ptrs, flag_ptrs, cap, epoch, epoch_ctr=ctr)
    return e


def run_wait(ops, flags, off, n, value, ctr, bump):
    guard(flags, range(off, off + n), value, ctr, "peer_wait")
    ops.peer_wait(flags.data_ptr() + 4 * off, n, value, epoch_ctr=ctr, bump=bump)


# ================================================================================ peer_rmsprop
BSTART = 192         # bucket start: a non-zero multiple of 64, like the engine's buckets
EPOCHS = {"host": (7, None), "ctr": (1, 2 ** 32 - 2), "wrap": (3, 2 ** 32 - 1)}
SIZES = [("zero", "ctr"), ("one", "host"), ("one", "wrap"), ("three", "ctr")]
# three grid-stride passes of a sharded bucket need W x 1.5 M elements per buffer: up to W = 4
RMS_CASES = [(w, b, s, e) for w in (1, 2, 3, 4, 8, 16) for b in (1, 0) for s, e in SIZES
             if not (s == "three" and b and w > 4)]


def shard_count(size, sms, per_sm):
    """Elements per rank: none; one pass of a partial grid with a ragged last block; two full
    passes of the capped grid and a ragged half."""
    cap = sms * per_sm
    return {"zero": 0, "one": 8 * (128 * cap + 3), "three": 8 * (640 * cap + 5)}[size]


def lo_ranges(broadcast, size, W, n):
    if broadcast:
        s1, sl = BSTART + min(1, W - 1) * n, BSTART + (W - 1) * n
        return [(s1 - 40, s1 + 56), (sl + 16, sl + 104)]   # across a shard start; in the last shard
    if size == "one":
        return [(BSTART + 64, BSTART + 64), (BSTART + n - 48, BSTART + n + 40)]  # empty; across the end
    return [(BSTART + n + 8, BSTART + n + 200), (BSTART + 8, BSTART + 120)]      # outside; inside


def _within(got, ref, tol, what):
    err = np.abs(np.asarray(got, np.float64) - ref)
    bad = err > tol
    assert not bad.any(), f"{what}: {bad.sum()} outside the fp64 bound, worst {err[bad].max()}"


@pytest.mark.parametrize("world,broadcast,size,epochs", RMS_CASES)
def test_peer_rmsprop_exact(ops, geom, world, broadcast, size, epochs):
    """Rank-order sum -> RMSprop -> bf16 (+ lo) stores, bit for bit against ops.rmsprop_step on
    the host sum; broadcast = 1 shards [BSTART, +W n) as _launch_bucket does, broadcast = 0 has
    every rank update the whole range and store its own copy only."""
    W, (sms, per_sm) = world, geom
    n = shard_count(size, sms, per_sm)
    assert P.rmsprop_passes(n, sms, per_sm) == {"zero": 0, "one": 1, "three": 3}[size]
    span = W * n if broadcast else n
    L = BSTART + span + 256
    rs = slice(BSTART, BSTART + span)
    epoch, c0 = EPOCHS[epochs]
    rng = np.random.default_rng([W, broadcast, n, epoch])
    G, order = P.order_terms(rng, W, span)
    w0 = rng.standard_normal(L, dtype=np.float32)
    s0 = rng.random(L, dtype=np.float32)
    s0[::7] = 0.0                                       # sqrt(ms + eps) of eps alone
    m0 = rng.standard_normal(L, dtype=np.float32) * np.float32(0.01)
    m0[5::46] = -0.0
    init = [Flat(L, F32, x) for x in (w0, s0, m0)]
    grads = []
    for q in range(W):
        grads.append(Flat(L, F32))
        grads[-1].t[rs].copy_(_dev(G[q]))
    g_before = [g.raw.clone() for g in grads]
    state = [[Flat(L, F32, x.t) for x in init] for _ in range(W)]
    p16 = [Flat(L, BF16) for _ in range(W)]
    p16lo = [Flat(L, BF16) for _ in range(W)]
    sent16 = p16[0].raw.clone()
    eff = P.effective_epoch(epoch, c0)
    ready = [Flat(W, I32, np.full(W, P.as_i32(eff), np.int32)) for _ in range(W)]
    r_before = ready[0].raw.clone()
    ctr = [ctr_tensor(c0) for _ in range(W)]
    ranges = lo_ranges(broadcast, size, W, n)
    lo = ([b.ptr for b in p16lo], 0, ranges)
    launches = ops.launch_count()
    for r in range(W):
        start = BSTART + r * n if broadcast else BSTART
        run_rmsprop(ops, W, r, [g.ptr for g in grads], [b.ptr for b in p16],
                    [x.t for x in state[r]], start, n, broadcast, ready[r].t, 0, epoch, ctr[r], lo)
        if not broadcast:
            torch.cuda.synchronize()
            for q in range(r + 1, W):
                assert_bits(p16[q].raw, sent16, f"rank {r} wrote rank {q}'s p16")
                assert_bits(p16lo[q].raw, sent16, f"rank {r} wrote rank {q}'s p16lo")
    torch.cuda.synchronize()
    assert ops.launch_count() - launches == (W if n else 0)

    gsum = P.rank_order_sum(G)
    if W >= 3 and span:
        rev = P.reverse_order_sum(G)
        assert np.mean(gsum.view(np.uint32)[order] != rev.view(np.uint32)[order]) > 0.99
    ref = [Flat(L, F32, x.t) for x in init]
    if span:
        ops.rmsprop_step(ref[0].t[rs], None, _dev(gsum), ref[1].t[rs], ref[2].t[rs], LR, RHO, MOM, EPS)
    w, s, m = (x.t[rs].cpu().numpy() for x in ref)
    lr, rho, mo, eps = (float(np.float32(v)) for v in (LR, RHO, MOM, EPS))
    g64 = gsum.astype(np.float64)
    w64, s64, m64 = R.rmsprop64(w0[rs].astype(np.float64), g64, s0[rs].astype(np.float64),
                                m0[rs].astype(np.float64), lr, rho, mo, eps)
    mom_abs = mo * np.abs(m0[rs]) + lr * np.abs(g64) / np.sqrt(s64 + eps)
    _within(s, s64, 1e-5 * s64, "ms")
    _within(m, m64, 1e-5 * mom_abs, "mom")
    _within(w, w64, 1e-5 * (np.abs(w64) + mom_abs), "w")

    for r in range(W):
        a, b = (BSTART + r * n, BSTART + (r + 1) * n) if broadcast else (BSTART, BSTART + span)
        for k, name in enumerate(("p32", "ms", "mom")):
            want = with_range(init[k].raw, a, b, ref[k].raw[PAD + a:PAD + b])
            assert_bits(state[r][k].raw, want, f"rank {r} {name}")
    hi, lo32 = R.split_ref(w)
    if span:     # the host split is cc_split_bf16's, so the kernel's lo term must be too
        sp = [torch.empty(1, span, dtype=BF16, device="cuda") for _ in range(2)]
        ops.split_bf16(ref[0].t[rs].view(1, span), *sp)
        assert torch.equal(sp[0].view(torch.int16)[0], bf16_dev(hi)), "split_bf16 hi"
        assert torch.equal(sp[1].view(torch.int16)[0], bf16_dev(lo32)), "split_bf16 lo"
    want16 = with_range(sent16, BSTART, BSTART + span, bf16_dev(hi))
    in_lo = P.lo_mask(np.arange(BSTART, BSTART + span), ranges)
    assert in_lo.any() or n == 0
    lo_bits = np.where(in_lo, R.bf16_bits(lo32), np.uint16(SENT[BF16][1])).view(np.int16)
    want_lo = with_range(sent16, BSTART, BSTART + span, _dev(lo_bits))
    for q in range(W):
        assert_bits(p16[q].raw, want16, f"p16[{q}]")
        assert_bits(p16lo[q].raw, want_lo, f"p16lo[{q}]")
        assert_bits(grads[q].raw, g_before[q], f"grad[{q}]")
        assert_bits(ready[q].raw, r_before, f"ready flags of rank {q}")
        assert ctr_value(ctr[q]) == c0


# ============================================================================== peer_allreduce
AR_CAP = 16384       # engine.TorchDist._AR_CAP (largest BatchNorm: 2 x 6738 = 13476)
AR_N = [1, 31, 32, 33, 1023, 1024, 1025, 13476]
AR_CASES = [(n, cap) for n in AR_N for cap in (n, AR_CAP)] + [(AR_CAP, AR_CAP)]
AR_WORLDS = [1, 2, 3, 5, 8, 16]


class Ranks:
    """W ranks' all-reduce state: [2][W][cap] slots, [W] flags (at `flag0`), data buffers."""

    def __init__(self, W, n, cap, flag0, c0=None):
        self.W, self.n, self.cap = W, n, cap
        self.slots = [Flat(2 * W * cap, F32) for _ in range(W)]
        self.flags = [Flat(W, I32, np.full(W, P.as_i32(flag0), np.int32)) for _ in range(W)]
        self.data = [Flat(n, F32) for _ in range(W)]
        self.ctr = [ctr_tensor(c0) for _ in range(W)]

    def call(self, ops, D, epoch, rel_epoch, use_ctr, what):
        """Ranks 0, 1, ... one after another.  Before rank r runs, the slots [parity][q] of r's
        array and r's flags are pre-filled / raised ONLY for q > r: slot [parity][r] and those
        of q < r must come from r's own push and the earlier ranks' kernels."""
        W, n, cap = self.W, self.n, self.cap
        Dd = _dev(D)
        want = _dev(P.rank_order_sum(D)).view(I32)
        off = [P.ar_slot_offset(epoch, W, cap, q) for q in range(W)]
        for r in range(W):
            self.data[r].t.copy_(Dd[r])
            for q in range(r + 1, W):
                self.slots[r].t[off[q]:off[q] + n].copy_(Dd[q])
                self.flags[r].t[q] = P.as_i32(epoch)
            before = [s.raw.clone() for s in self.slots]
            fbefore = [f.raw.clone() for f in self.flags]
            e = run_allreduce(ops, self.data[r].t, W, r, [s.ptr for s in self.slots],
                              [f.ptr for f in self.flags], self.flags[r].t, cap, rel_epoch,
                              self.ctr[r] if use_ctr else None)
            assert e == epoch
            torch.cuda.synchronize()
            at = f"{what} rank {r}"
            assert_bits(self.data[r].raw, with_range(self.data[r].raw, 0, n, want), at + " data")
            for q in range(W):
                # my values land in slot [parity][r] of every rank; nothing else moves
                assert_bits(self.slots[q].raw, with_range(before[q], off[r], off[r] + n,
                                                          Dd[r].view(I32)), f"{at} slots of {q}")
                fb = fbefore[q].clone()
                fb[PAD + r] = P.as_i32(epoch)
                assert_bits(self.flags[q].raw, fb, f"{at} flags of {q}")
            if use_ctr:
                assert ctr_value(self.ctr[r]) == epoch, at + " counter"


@pytest.mark.parametrize("n,cap", AR_CASES)
@pytest.mark.parametrize("world", AR_WORLDS)
def test_peer_allreduce_exact(ops, world, n, cap):
    """Every rank's data becomes the rank-order sum, bit-identical across ranks; after rank r
    runs, slot [parity][r] of every rank holds r's data; the other parity half, [n, cap) of
    every slot and the padding are untouched.  Both parities (epoch 6 / 7)."""
    epoch = 6 if cap == n else 7
    D, _ = P.order_terms(np.random.default_rng([world, n, cap]), world, n)
    Ranks(world, n, cap, epoch - 1).call(ops, D, epoch, epoch, False, f"W={world} n={n} cap={cap}")


@pytest.mark.parametrize("c0", [0, 2 ** 32 - 2])
@pytest.mark.parametrize("world", AR_WORLDS)
def test_peer_allreduce_epoch_counter(ops, world, c0):
    """The engine's form (epoch = 1 + *epoch_ctr, written back): three consecutive calls; the
    parity alternates, the counter advances by one per call (through 2^32 from c0 = 2^32 - 2),
    and a call never disturbs the previous epoch's slots."""
    n = 1025
    rk = Ranks(world, n, AR_CAP, c0, c0)
    rng = np.random.default_rng([world, c0 & 0xFF])
    for call in range(3):
        D, _ = P.order_terms(rng, world, n)
        rk.call(ops, D, P.u32(c0 + call + 1), 1, True, f"call {call}")
    assert [ctr_value(c) for c in rk.ctr] == [P.u32(c0 + 3)] * world


# ========================================================================= peer_signal / wait
@pytest.mark.parametrize("c0", [None, 5, 2 ** 32 - 1])
@pytest.mark.parametrize("n", [1, 16])
def test_peer_signal(ops, n, c0):
    """value + *ctr (mod 2^32) lands in each of the n targets and nowhere else."""
    buf = Flat(48, I32, np.zeros(48, np.int32))
    value = 2 ** 32 - 3
    ctr = ctr_tensor(c0)
    ops.peer_signal([buf.ptr + 4 * (3 * q + 1) for q in range(n)], value, epoch_ctr=ctr)
    torch.cuda.synchronize()
    want = torch.full((48,), 0, dtype=I32, device="cuda")
    want[1:3 * n:3] = P.as_i32(P.effective_epoch(value, c0))
    assert_bits(buf.raw, with_range(buf.raw, 0, 48, want), "signal targets")
    assert ctr_value(ctr) == c0


@pytest.mark.parametrize("c0", [None, 7, 2 ** 32 - 2])
@pytest.mark.parametrize("bump", [True, False])
@pytest.mark.parametrize("n", [1, 16, 200])
def test_peer_wait_satisfied(ops, n, bump, c0):
    """A satisfied wait (flags at, or up to 2^31 - 1 past, the epoch, across the wrap) returns,
    and bump leaves ctr = value + ctr_old; bump = 0 leaves the counter alone."""
    value = 3
    e = P.effective_epoch(value, c0)
    ahead = [0, 1, 2 ** 31 - 1, 5, 2 ** 16]
    flags = Flat(n + 8, I32, np.array([P.as_i32(e + ahead[i % 5]) for i in range(n + 8)], np.int32))
    before = flags.raw.clone()
    ctr = ctr_tensor(c0)
    run_wait(ops, flags.t, 4, n, value, ctr, bump)
    torch.cuda.synchronize()
    assert ctr_value(ctr) == (e if bump and c0 is not None else c0)
    assert_bits(flags.raw, before, "flags")


# ============================================================================ protocol replay
class Replay:
    """The engine's data-parallel update (Net._peer_update / _reduce_and_update) for W ranks:
    two sharded buckets with hi + lo terms, a gap, the replicated tail; flags
    [kind 0 ready / 1 done][bucket, tail = nb - 1][source], per-rank counters, and a closing
    peer_wait(bump=True) over every done flag.  Phases interleave across ranks so that every
    wait is satisfied at launch.

    `me`: the ranks this process drives (all of them when emulated); `alloc(n, dtype)` ->
    ({rank: Flat}, [peer pointer of every rank]); `barrier()` runs between phases."""
    N_FLAT, K = 5120, 4096
    BUCKETS = [(0, 2560), (2560, 3840)]            # [3840, K): a gap no bucket covers
    HILO = [(256, 1024), (2304, 2816)]             # the second crosses the bucket boundary

    def __init__(self, ops, W, me, alloc, c0, seed, mc=(0, 0), barrier=lambda: None):
        self.ops, self.W, self.me, self.c0, self.mc, self.barrier = ops, W, me, c0, mc, barrier
        self.nb = len(self.BUCKETS) + 1
        self.rng = np.random.default_rng(seed)
        N = self.N_FLAT
        self.stage, self.stage_p = alloc(W * N, F32)
        self.p16, self.p16_p = alloc(N, BF16)
        self.p16lo, self.p16lo_p = alloc(N, BF16)
        self.flags, self.flag_p = alloc(2 * self.nb * W, I32)
        w0 = self.rng.standard_normal(N, dtype=np.float32)
        s0 = self.rng.random(N, dtype=np.float32)
        m0 = self.rng.standard_normal(N, dtype=np.float32) * np.float32(0.01)
        hi, lo = R.split_ref(w0)
        self.ref = [Flat(N, F32, x) for x in (w0, s0, m0)]
        self.state = {r: [Flat(N, F32, x.t) for x in self.ref] for r in me}
        self.want = {r: [x.raw.clone() for x in self.ref] for r in me}
        self.ctr = {r: ctr_tensor(c0) for r in me}
        for r in me:
            self.p16[r].raw[PAD:PAD + N] = bf16_dev(hi)
            self.p16lo[r].raw[PAD:PAD + N] = bf16_dev(lo)
            self.flags[r].t.fill_(P.as_i32(c0))
        self.want16 = self.p16[me[0]].raw.clone()
        self.want_lo = self.p16lo[me[0]].raw.clone()
        torch.cuda.synchronize()
        self.barrier()

    def fptr(self, on, kind, bucket, src):
        return self.flag_p[on] + 4 * ((kind * self.nb + bucket) * self.W + src)

    def findex(self, kind, bucket, src):
        return (kind * self.nb + bucket) * self.W + src

    def _phase(self, fn):
        for r in self.me:
            fn(r)
        torch.cuda.synchronize()
        self.barrier()

    def update(self, u):
        ops, W, N, nb = self.ops, self.W, self.N_FLAT, self.nb
        G, _ = P.order_terms(self.rng, W, N)
        Gd = _dev(G)
        for r in self.me:                 # what the wgrad epilogues leave in r's staging slots
            st = self.stage[r].t
            for a, b in self.BUCKETS:
                n = (b - a) // W
                for q in range(W):
                    st[q * N + a + r * n:q * N + a + (r + 1) * n] = Gd[q, a + r * n:a + (r + 1) * n]
            st[r * N + self.K:(r + 1) * N] = Gd[r, self.K:]
        torch.cuda.synchronize()
        self.barrier()
        lo = (self.p16lo_p, self.mc[1], self.HILO)
        jobs = [(bi, a, (b - a) // W, True) for bi, (a, b) in enumerate(self.BUCKETS)]
        jobs.append((nb - 1, self.K, N - self.K, False))
        for bucket, a, n, bc in jobs:
            self._phase(lambda r: ops.peer_signal([self.fptr(t, 0, bucket, r) for t in range(W)], 1,
                                                  epoch_ctr=self.ctr[r]))

            def kernel(r):
                if bc:
                    grads = [self.stage_p[r] + 4 * q * N for q in range(W)]
                else:
                    grads = [self.stage_p[q] + 4 * q * N for q in range(W)]
                run_rmsprop(ops, W, r, grads, self.p16_p, [x.t for x in self.state[r]],
                            a + r * n if bc else a, n, bc, self.flags[r].t,
                            self.findex(0, bucket, 0), 1, self.ctr[r], lo if bc else None,
                            self.mc[0])
                ops.peer_signal([self.fptr(t, 1, bucket, r) for t in range(W)], 1,
                                epoch_ctr=self.ctr[r])
            self._phase(kernel)
        self._phase(lambda r: run_wait(ops, self.flags[r].t, self.findex(1, 0, 0), nb * W, 1,
                                       self.ctr[r], True))
        self._expect(P.rank_order_sum(G), u)

    def _expect(self, gsum, u):
        """Advance the reference by one update and compare every driven rank with it."""
        W, N = self.W, self.N_FLAT
        gd = _dev(gsum)
        for a, b in self.BUCKETS + [(self.K, N)]:
            self.ops.rmsprop_step(self.ref[0].t[a:b], None, gd[a:b], self.ref[1].t[a:b],
                                  self.ref[2].t[a:b], LR, RHO, MOM, EPS)
        torch.cuda.synchronize()
        w = self.ref[0].t.cpu().numpy()
        hi, lo = R.split_ref(w)
        hi_d, lo_d = bf16_dev(hi), bf16_dev(lo)
        lo_in = P.lo_mask(np.arange(N), self.HILO)
        for a, b in self.BUCKETS + [(self.K, N)]:
            self.want16[PAD + a:PAD + b] = hi_d[a:b]
            m = _dev(lo_in[a:b])
            self.want_lo[PAD + a:PAD + b] = torch.where(m, lo_d[a:b], self.want_lo[PAD + a:PAD + b])
        e = P.u32(self.c0 + u + 1)
        for r in self.me:
            mine = [(a + r * ((b - a) // W), a + (r + 1) * ((b - a) // W)) for a, b in self.BUCKETS]
            for a, b in mine + [(self.K, N)]:          # my shards and the replicated tail
                for k in range(3):
                    self.want[r][k][PAD + a:PAD + b] = self.ref[k].raw[PAD + a:PAD + b]
            at = f"update {u} rank {r}"
            for k, name in enumerate(("p32", "ms", "mom")):
                assert_bits(self.state[r][k].raw, self.want[r][k], f"{at} {name}")
            assert_bits(self.p16[r].raw, self.want16, at + " p16")
            assert_bits(self.p16lo[r].raw, self.want_lo, at + " p16lo")
            fl = torch.full((2 * self.nb * W,), P.as_i32(e), dtype=I32, device="cuda")
            assert_bits(self.flags[r].raw, with_range(self.flags[r].raw, 0, fl.numel(), fl),
                        at + " flags")
            assert ctr_value(self.ctr[r]) == e, at + " counter"


def local_alloc(W):
    def alloc(n, dtype):
        fl = [Flat(n, dtype) for _ in range(W)]
        return dict(enumerate(fl)), [f.ptr for f in fl]
    return alloc


@pytest.mark.parametrize("c0", [0, 2 ** 32 - 2])
@pytest.mark.parametrize("world", [2, 4])
def test_protocol_replay(ops, world, c0):
    """Three consecutive updates with the engine's call sequence and flag layout: every rank's
    p32 / ms / mom / p16 / p16lo equal the host reference bit for bit after each."""
    rp = Replay(ops, world, list(range(world)), local_alloc(world), c0, seed=[world, c0 & 0xFF])
    for u in range(3):
        rp.update(u)


# ======================================================================= rejected descriptors
def test_rejected_descriptors(ops):
    """Each malformed call raises before any launch and leaves every buffer as it was; a valid
    call still works afterwards."""
    from cellcomm_b200._lib import CCError
    W, n = 2, 64
    L = BSTART + W * n + 64
    grads = [Flat(L, F32, np.ones(L, np.float32)) for _ in range(W)]
    p16 = [Flat(L, BF16) for _ in range(W)]
    p16lo = [Flat(L, BF16) for _ in range(W)]
    st = [Flat(L, F32, np.zeros(L, np.float32)) for _ in range(3)]
    odd = [Flat(L + 1, F32, np.zeros(L + 1, np.float32)) for _ in range(3)]   # views 4 B off
    ready = Flat(W, I32, np.full(W, 5, np.int32))
    ar = Ranks(W, 8, 32, 0)
    sig = Flat(20, I32, np.zeros(20, np.int32))
    bufs = grads + p16 + p16lo + st + odd + [ready, sig] + ar.slots + ar.flags + ar.data
    g_p, h_p, l_p = [g.ptr for g in grads], [b.ptr for b in p16], [b.ptr for b in p16lo]

    def rms(world=W, rank=0, gp=g_p, hp=h_p, state=None, start=BSTART, count=n, bc=1, lo=None,
            mc=0):
        s = state or [x.t for x in st]
        ops.peer_rmsprop(world, rank, gp, hp, *s, start, count, bc, LR, RHO, MOM, EPS, ready.ptr, 5,
                         p16_multicast=mc, lo=lo)

    def c_world17():
        """world = 17 straight into the C entry point (ops.peer_rmsprop cannot build it: the
        descriptor holds CC_PEER_MAX = 16 pointers per array)."""
        import ctypes as C
        from cellcomm_b200 import _lib
        d = _lib.PeerRmspropDesc()
        d.world, d.rank, d.start, d.count, d.broadcast = 17, 0, BSTART, n, 1
        for q in range(len(d.grad)):
            d.grad[q], d.p16[q] = g_p[q % W], h_p[q % W]
        d.p32, d.ms, d.mom = (x.ptr for x in st)
        d.lr, d.rho, d.momentum, d.eps = LR, RHO, MOM, EPS
        d.ready, d.epoch = ready.ptr, 5
        _lib.check(_lib.load().cc_peer_rmsprop(C.byref(d), torch.cuda.current_stream().cuda_stream))

    def shifted(ptrs, q, by):
        return [p + by if i == q else p for i, p in enumerate(ptrs)]

    lo_ok = (l_p, 0, [(BSTART, BSTART + 64)])
    bad = {
        "world 0": lambda: rms(world=0, gp=[], hp=[]),
        "world 17": lambda: rms(world=17, gp=g_p * 9, hp=h_p * 9),
        "world 17, C entry point": c_world17,
        "rank = world": lambda: rms(rank=W),
        "rank = world, replicated": lambda: rms(rank=W, bc=0),
        "rank -1": lambda: rms(rank=-1),
        "count % 8": lambda: rms(count=n - 4),
        "start = 4 mod 8": lambda: rms(start=BSTART + 4),
        "p32 4 B off": lambda: rms(state=[odd[0].t[1:], st[1].t, st[2].t]),
        "ms 4 B off": lambda: rms(state=[st[0].t, odd[1].t[1:], st[2].t]),
        "mom 4 B off": lambda: rms(state=[st[0].t, st[1].t, odd[2].t[1:]]),
        "grad[1] 4 B off": lambda: rms(gp=shifted(g_p, 1, 4)),
        "grad[0] 8 B off": lambda: rms(gp=shifted(g_p, 0, 8)),
        "p16[1] 2 B off": lambda: rms(hp=shifted(h_p, 1, 2)),
        "p16[0] 8 B off, replicated": lambda: rms(hp=shifted(h_p, 0, 8), bc=0),
        "p16lo[1] 2 B off": lambda: rms(lo=(shifted(l_p, 1, 2), 0, lo_ok[2])),
        "p16lo[1] missing": lambda: rms(lo=([l_p[0], 0], 0, lo_ok[2])),
        "multicast 8 B off": lambda: rms(mc=h_p[0] + 8),
        "lo multicast 2 B off": lambda: rms(lo=(l_p, l_p[0] + 2, lo_ok[2])),
        "lo range begin % 8": lambda: rms(lo=(l_p, 0, [(BSTART + 4, BSTART + 64)])),
        "lo range end % 8": lambda: rms(lo=(l_p, 0, [(BSTART, BSTART + 60)])),
        "three lo ranges": lambda: rms(lo=(l_p, 0, [(0, 8), (16, 24), (32, 40)])),
        "allreduce n > cap": lambda: ops.peer_allreduce(
            torch.zeros(33, device="cuda"), W, 0, [s.ptr for s in ar.slots],
            [f.ptr for f in ar.flags], 32, 1),
        "allreduce rank = world": lambda: ops.peer_allreduce(
            ar.data[0].t, W, W, [s.ptr for s in ar.slots], [f.ptr for f in ar.flags], 32, 1),
        "allreduce world 17": lambda: ops.peer_allreduce(
            ar.data[0].t, 17, 0, [ar.slots[0].ptr] * 17, [ar.flags[0].ptr] * 17, 32, 1),
        "signal n = 0": lambda: ops.peer_signal([], 1),
        "signal n = 17": lambda: ops.peer_signal([sig.ptr] * 17, 1),
    }
    snap = [b.raw.clone() for b in bufs]
    for what, call in bad.items():
        launches = ops.launch_count()
        with pytest.raises((CCError, ValueError)):
            call()
        torch.cuda.synchronize()
        assert ops.launch_count() == launches, what
        for b, s in zip(bufs, snap):
            assert_bits(b.raw, s, what)
    guard(ready.t, range(W), 5, None, "valid call")
    rms(lo=lo_ok)
    torch.cuda.synchronize()
    assert ops.launch_count() == launches + 1
    w = st[0].t[BSTART:BSTART + n].cpu().numpy()
    assert np.all(w < 0) and np.array_equal(p16[1].t[BSTART:BSTART + n].view(torch.int16).cpu().numpy(),
                                            R.bf16_bits(w).view(np.int16))


# ============================================================================== real fabric
def test_real_fabric():
    """The replay and three all-reduces over real peer memory under torchrun
    (tests/peer_gpu_worker.py) on 8 GPUs, or 2: P2P stores, and the NVLS multicast address when
    the fabric has one; every rank checks its bits against its local reference and all ranks
    agree.  Skipped with fewer than 2 GPUs or without symmetric memory."""
    import subprocess
    import sys
    n_gpus = torch.cuda.device_count()
    if n_gpus < 2:
        pytest.skip("needs 2 GPUs")
    world = 8 if n_gpus >= 8 else 2
    port = 29900 + (os.getpid() % 97)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
           f"--nproc-per-node={world}", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(HERE, "peer_gpu_worker.py")]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    if "peer_check skip:" in out.stdout:
        pytest.skip(out.stdout.split("peer_check skip:", 1)[1].strip().splitlines()[0])
    assert "peer_check ok" in out.stdout
    print([ln for ln in out.stdout.splitlines() if "peer_check ok" in ln][0])
