"""Network graphs + forward/backward executor over the C-ABI kernels.

This is the host side of what TensorFlow/Keras does for the reference inside
`Model.train_on_batch` / `Model.predict` (src/bigan_classify.py:83-155): a static layer graph
per network (G, E, D), a forward pass that saves activations, a reverse pass that emits
dgrad / wgrad GEMMs and the tail kernels, and a fused-layout RMSprop update.  All arithmetic
is in libcellcomm_b200.so (cellcomm_b200.ops); torch only owns buffers and streams.

Semantics follow Keras 2.4.0 as used by the reference (SURVEY.md Appendix A):
  * Dense: y = act(x W + b), W[in,out]; Concatenate inputs are consumed as GEMM segments.
  * BatchNormalization: eps 1e-3, momentum 0.99, biased batch variance; a frozen
    (trainable=False) BN runs in inference mode even inside train_on_batch.
  * Dropout: active inside frozen sub-models during train_on_batch, off in predict.
"""
import math
import os

import torch

from . import ops as _ops_module

# tests may swap this for an emulator to exercise the host logic without a GPU
ops = _ops_module

BN_EPS, BN_MOMENTUM = 1e-3, 0.99                  # Keras BatchNormalization defaults
LR, RHO, MOMENTUM, EPSILON = 0.0075, 0.85, 0.1, 1e-7   # src/bigan_classify.py:88 (+ Keras eps)
REAL_LABEL = 0.95                                 # src/bigan_classify.py:128

_ACT = {"none": 0, "sigmoid": 1, "relu": 2, "softmax": 0}
# two-term bf16 expansion for the inputs of Dense layers that feed a BatchNormalization
# 0: none; 1: narrow tensors only (free); 2: also the wide inputs of BN-feeding Dense layers;
# 3: also their dL/dz.  Default "auto": level 3 for the generator (its relu+BN trunk is the
# only place where bf16 operands cost more than 2 % gradient cosine; +3.4 % GEMM work per
# step), level 1 for E and D.  Level 3 everywhere costs +17 %.  See DESIGN.md.
_SPLIT_ENV = os.environ.get("CELLCOMM_B200_SPLIT", "auto")
_SPLIT_PRECISION = None if _SPLIT_ENV == "auto" else int(_SPLIT_ENV)
_SMALL_WIDTH = int(os.environ.get("CELLCOMM_B200_SMALL_WIDTH", "512"))
# data parallel: reduce-scatter + sharded RMSprop + bf16 all-gather instead of all-reduce + full sweep
_SHARD_OPTIMIZER = os.environ.get("CELLCOMM_B200_SHARD_OPT", "1") != "0"
# ... in buckets of about this many parameters, each reduce-scattered on the side stream as soon
# as the backward pass has produced its gradient (big layers are cut along their rows)
# diagnostic: data-parallel step without gradient exchange / update (compute-only lower bound)
_DP_SKIP_UPDATE = os.environ.get("CELLCOMM_B200_DP_SKIP_UPDATE", "0") == "1"
_BUCKET_ELEMS = int(os.environ.get("CELLCOMM_B200_BUCKET_ELEMS", str(48 << 20)))
# hi + lo bf16 compute copies of the BN-feeding kernels of level-3 networks (the generator)
_HILO_WEIGHTS = os.environ.get("CELLCOMM_B200_HILO_WEIGHTS", "1") != "0"
# fused-optimiser mode: Dense kernels of at most this many elements are NOT updated inside their
# wgrad epilogue (their weight-gradient GEMM has one or two output tiles, i.e. runs on one or two
# SMs for the whole batch reduction: ~45 us each at batch 2048, ~1.9 ms per step over the ~30
# narrow layers); they take the split-K wgrad and one flat RMSprop sweep per contiguous range
_NARROW_ELEMS = int(os.environ.get("CELLCOMM_B200_NARROW_ELEMS", str(1 << 20)))
# fused-optimiser mode: keep the fp32 master weights and RMSprop slots of the wide kernels in the
# BLOCKED layout of cc_gemm_desc.rms_blocked (4 KB blocks in accumulator order) while training;
# they are converted back to rows whenever anything else reads them (Net._rows)
_BLOCKED_STATE = os.environ.get("CELLCOMM_B200_BLOCKED_STATE", "1") != "0"


# =========================================================================== graph specs
class GraphBuilder:
    """Records a network as nodes over tensor ids; layers keep the reference's creation order."""

    def __init__(self, name):
        self.name = name
        self.widths = []
        self.nodes = []
        self.inputs = {}
        self.layers = []       # ("dense", in_widths, units, act) | ("bn", width)
        self.n_dropout = 0
        self.output = None

    def _new(self, width):
        self.widths.append(int(width))
        return len(self.widths) - 1

    def input(self, name, width):
        t = self._new(width)
        self.inputs[name] = t
        return t

    def dense(self, ins, units, act):
        ins = list(ins) if isinstance(ins, (list, tuple)) else [ins]
        out = self._new(units)
        self.layers.append(("dense", [self.widths[i] for i in ins], int(units), act))
        self.nodes.append({"kind": "dense", "ins": ins, "out": out, "layer": len(self.layers) - 1,
                           "act": act})
        if act == "softmax":
            sm = self._new(units)
            self.nodes.append({"kind": "softmax", "ins": [out], "out": sm})
            return sm
        return out

    def bn(self, x):
        out = self._new(self.widths[x])
        self.layers.append(("bn", self.widths[x]))
        self.nodes.append({"kind": "bn", "ins": [x], "out": out, "layer": len(self.layers) - 1})
        return out

    def dropout(self, x, rate):
        out = self._new(self.widths[x])
        self.nodes.append({"kind": "dropout", "ins": [x], "out": out, "rate": float(rate),
                           "drop": self.n_dropout})
        self.n_dropout += 1
        return out

    def concat(self, xs):
        out = self._new(sum(self.widths[i] for i in xs))
        self.nodes.append({"kind": "concat", "ins": list(xs), "out": out})
        return out


def cont_generator_graph(Z, G):
    """src/bigan_cont.py:7-25"""
    w = [int(G * f) for f in (0.2, 0.1)]
    b = GraphBuilder("cell_generator")
    z, r = b.input("z", Z), b.input("r", Z)
    all_in = b.concat([z, r])
    x = b.dense(all_in, 50, "sigmoid")
    x = b.dropout(b.concat([x, all_in]), 0.1)
    x = b.dense(x, 256, "sigmoid")
    x = b.dense(x, 256, "sigmoid")
    x = b.bn(x)
    x = b.dropout(b.concat([x, all_in]), 0.1)
    x = b.dense(x, w[1], "sigmoid")
    x = b.dense(x, w[0], "relu")
    x = b.bn(x)
    b.output = b.dense(x, G, "relu")
    return b


def cont_encoder_graph(Z, G):
    """src/bigan_cont.py:28-41"""
    w = [int(G * f) for f in (0.1, 0.05)]
    b = GraphBuilder("cell_encoder")
    cell = b.input("cell", G)
    x = b.dense(cell, w[0], "sigmoid")
    x = b.dropout(x, 0.15)
    x = b.dense([x, cell], w[1], "sigmoid")      # Concatenate()([x, cell_in]) as two GEMM segments
    x = b.dropout(x, 0.1)
    x = b.bn(x)
    x = b.dense(x, 150, "sigmoid")
    x = b.dense(x, 150, "sigmoid")
    b.output = b.dense(x, Z, "sigmoid")
    return b


def classify_generator_graph(Z, G):
    """src/bigan_classify.py:10-25"""
    b = GraphBuilder("cell_generator")
    z, r = b.input("z", Z), b.input("r", Z)
    all_in = b.concat([z, r])
    x = b.dense(all_in, 50, "sigmoid")
    x = b.dropout(b.concat([x, all_in]), 0.1)
    x = b.dense(x, 256, "sigmoid")
    x = b.bn(x)
    x = b.dropout(b.concat([x, all_in]), 0.1)
    x = b.dense(x, 256, "sigmoid")
    x = b.dropout(x, 0.1)
    x = b.dense(x, 1024, "relu")
    b.output = b.dense(x, G, "relu")
    return b


def classify_encoder_graph(Z, G):
    """src/bigan_classify.py:28-40"""
    b = GraphBuilder("cell_encoder")
    cell = b.input("cell", G)
    proc = b.dense(cell, 1000, "sigmoid")
    x = b.dropout(proc, 0.15)
    x = b.dense(x, 300, "sigmoid")
    x = b.dropout(x, 0.15)
    x = b.dense([x, proc], 150, "sigmoid")
    b.output = b.dense(x, Z, "softmax")
    return b


def discriminator_graph(Z, G):
    """src/bigan_classify.py:43-75 (shared by both variants, bigan_cont.py:46-50)"""
    l = [int(G * f) for f in (0.3, 0.1, 0.05)]
    b = GraphBuilder("cell_discriminator")
    z, cell = b.input("z", Z), b.input("cell", G)
    a = b.dense(z, 50, "sigmoid")
    a2 = b.dense(z, 50, "sigmoid")
    x = b.dropout(b.concat([a, a2, z]), 0.15)
    x = b.bn(x)
    x = b.dense(x, 256, "sigmoid")
    x = b.dense(x, 256, "sigmoid")
    se = b.dense(x, 256, "sigmoid")
    x = b.dense(cell, l[0], "sigmoid")
    x = b.dropout(x, 0.15)
    x = b.dense([x, cell], l[1], "sigmoid")
    x = b.bn(x)
    x = b.dropout(x, 0.15)
    x = b.dense(x, l[2], "sigmoid")
    x = b.dense(x, 256, "sigmoid")
    sg = b.dense(x, 256, "sigmoid")
    x = b.dense([se, sg], 300, "sigmoid")
    x = b.bn(x)
    x = b.dropout(x, 0.15)
    x = b.dense(x, 50, "sigmoid")
    x = b.dense(x, 50, "sigmoid")
    x = b.dense(x, 10, "sigmoid")
    b.output = b.dense(x, 1, "sigmoid")
    return b


# =========================================================================== runtime
def _pad(n, m=64):
    return (n + m - 1) // m * m


class _NoDist:
    world_size = 1
    rank = 0

    def all_reduce(self, t):
        return t

    all_reduce_grad = all_reduce

    def broadcast(self, t):
        return t

    def broadcast_object(self, obj=None):
        return obj


class TorchDist:
    """Data-parallel plumbing over torch.distributed (NCCL over NVLink on the GPU box, gloo in
    the CPU tests): sum all-reduces of BN statistics, flat gradients and the loss buffer.
    Every rank holds the full weights and 1/world_size of each batch's rows."""

    def __init__(self, group=None, grad_group=None):
        import torch.distributed as dist
        self._dist, self.group = dist, group
        self.world_size = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        # gradient reduce-scatter / weight all-gather run on a side stream while the backward
        # pass keeps issuing small BatchNorm all-reduces on the main stream.  torch serialises
        # the collectives of ONE process group on its NCCL stream, so the bulk traffic gets a
        # communicator of its own (collective call: every rank constructs TorchDist).
        self.grad_group = grad_group
        if grad_group is None and self.world_size > 1 and group is None and \
                dist.get_backend() == "nccl":
            self.grad_group = dist.new_group(ranks=list(range(self.world_size)))
        if self.grad_group is None:
            self.grad_group = group

    def symmetric_zeros(self, numel, dtype, device):
        """A zeroed buffer mapped into every rank's address space over NVLink (torch symmetric
        memory; collective call) -> (tensor, [device pointer of rank q's copy], handle), or None
        when peer memory is unavailable (CPU / gloo tests, several nodes, CELLCOMM_B200_PEER_OPT=0).
        The peer-memory optimiser kernel (csrc/peer_optimizer.cu) is the only consumer."""
        if (self.world_size not in (2, 4, 8) or torch.device(device).type != "cuda"
                or os.environ.get("CELLCOMM_B200_PEER_OPT", "1") == "0"
                or self._dist.get_backend(self.group) != "nccl"
                or int(os.environ.get("LOCAL_WORLD_SIZE", self.world_size)) != self.world_size):
            return None
        if getattr(self, "_symm_failed", False):
            return None
        try:
            import torch.distributed._symmetric_memory as symm
            t = symm.empty(int(numel), dtype=dtype, device=device)
            t.zero_()
            hdl = symm.rendezvous(t, self._dist.group.WORLD if self.group is None else self.group)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
        except Exception as exc:      # fails on every rank alike: fall back to the NCCL path
            self._symm_failed = True
            if self.rank == 0:
                import sys
                print(f"cellcomm_b200: symmetric memory unavailable ({exc}); data-parallel "
                      f"updates use NCCL reduce-scatter / all-gather", file=sys.stderr, flush=True)
            return None
        assert ptrs[self.rank] == t.data_ptr(), "symmetric memory: local pointer mismatch"
        return t, ptrs, hdl

    _AR_CAP = 16384      # floats per small all-reduce over peer memory (largest BN: 2 x 6738)

    def _peer_allreduce_state(self, device):
        """Peer-mapped staging slots + flags for the one-kernel small all-reduce (lazy,
        collective: the first all-reduce happens at the same point on every rank)."""
        st = getattr(self, "_ar", None)
        if st is None:
            st = False
            if os.environ.get("CELLCOMM_B200_PEER_ALLREDUCE", "1") != "0":
                W = self.world_size
                a = self.symmetric_zeros(2 * W * self._AR_CAP, torch.float32, device)
                if a is not None:
                    b = self.symmetric_zeros(W, torch.int32, device)
                    # epoch counter on the device (advanced by the kernel itself): the call
                    # is identical every time, so a captured CUDA graph can replay it
                    st = {"slots": a[1], "flags": b[1], "keep": (a, b),
                          "ctr": torch.zeros(1, dtype=torch.int32, device=device)}
            self._ar = st
        return st or None

    def all_reduce(self, t):
        """Sum all-reduce of a small tensor (BN statistics, loss buffer)."""
        if self.world_size > 1:
            st = None
            if t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and \
                    t.numel() <= self._AR_CAP:
                st = self._peer_allreduce_state(t.device)
            if st is not None:
                ops.peer_allreduce(t, self.world_size, self.rank, st["slots"], st["flags"],
                                   self._AR_CAP, 1, epoch_ctr=st["ctr"])
            else:
                self._dist.all_reduce(t, op=self._dist.ReduceOp.SUM, group=self.group)
        return t

    def broadcast(self, t):
        """rank 0's tensor to every rank (start-up only)."""
        if self.world_size > 1:
            self._dist.broadcast(t, src=self._dist.get_global_rank(self.group, 0)
                                 if self.group is not None else 0, group=self.group)
        return t

    def broadcast_object(self, obj=None):
        """rank 0's picklable object to every rank (control messages, RNG states)."""
        box = [obj if self.rank == 0 else None]
        if self.world_size > 1:
            self._dist.broadcast_object_list(
                box, src=self._dist.get_global_rank(self.group, 0) if self.group is not None else 0,
                group=self.group)
        return box[0]

    def all_reduce_grad(self, t):
        """Sum all-reduce on the gradient communicator (side-stream traffic)."""
        if self.world_size > 1:
            self._dist.all_reduce(t, op=self._dist.ReduceOp.SUM, group=self.grad_group)
        return t

    def reduce_scatter(self, out_shard, full):
        """out_shard = this rank's 1/world slice of sum_over_ranks(full)."""
        if self._dist.get_backend(self.group) == "nccl":
            self._dist.reduce_scatter_tensor(out_shard, full, op=self._dist.ReduceOp.SUM,
                                             group=self.grad_group)
        else:   # gloo (CPU tests) has no reduce-scatter: all-reduce and slice
            self._dist.all_reduce(full, op=self._dist.ReduceOp.SUM, group=self.grad_group)
            n = out_shard.numel()
            out_shard.copy_(full[self.rank * n:(self.rank + 1) * n])

    def all_gather(self, full, shard):
        """full = concat over ranks of `shard` (shard may be the matching slice of full)."""
        if self._dist.get_backend(self.group) == "nccl":
            self._dist.all_gather_into_tensor(full, shard, group=self.grad_group)
        else:
            parts = [torch.empty_like(shard) for _ in range(self.world_size)]
            self._dist.all_gather(parts, shard.clone(), group=self.grad_group)
            full.copy_(torch.cat(parts))


def default_dist():
    """TorchDist when a process group is initialised (torchrun), else single-process."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return TorchDist()
    except Exception:
        pass
    return _NoDist()


def _on_main_stream(reduce_kw, opt_stream):
    """reduce_kw for a reduction about to be enqueued.  Deterministic mode shares ONE workspace
    between all reductions of a step, which is safe only because they all run on the main
    stream; the optimiser side stream must never run one (two reductions in flight at once
    would mix their partials and tickets)."""
    if reduce_kw and opt_stream is not None:
        assert torch.cuda.current_stream(opt_stream.device) != opt_stream, \
            "a fixed-order reduction was enqueued on the optimiser side stream"
    return reduce_kw


class Net:
    """One network (G, E or D): parameters in flat fused-layout buffers, activation buffers for
    up to `max_rows` rows, forward / backward / RMSprop."""

    def __init__(self, graph, max_rows, device, generator=None, dist=None, precision=1):
        self.precision = precision if _SPLIT_PRECISION is None else _SPLIT_PRECISION
        self.g = graph
        self.name = graph.name
        self.max_rows = int(max_rows)
        self.device = device
        self.dist = dist or _NoDist()
        self.hp, self.split = self._high_precision_tensors()
        self.blockable, self.state_blocked = [], False
        self._opt_event = None
        self._alloc_params(generator)
        self._build_buckets()
        self._find_narrow_layers()
        self.act = {}      # forward activations (bf16; fp32 for tensors in self.hp)
        self.shadow = {}   # bf16 copies of fp32 activations that also feed a GEMM
        self.grad = {}     # activation gradients, always fp32
        self.tmp = {}      # fp32 scratch for accumulating a second gradient contribution
        self.dzb = {}      # bf16 gradient w.r.t. a Dense pre-activation (GEMM operand)
        # optimiser sweeps (and their gradient all-reduce) run on a side stream and overlap the
        # next network's forward pass; every use of this net's parameters waits for the event
        self.opt_stream = None
        self._opt_event = None
        self.on_grow = None
        self._gshard = None
        self._master_stale = False
        self._slots_stale = False
        self.fuse_optimizer = False   # kernels updated inside the wgrad epilogue (1 GPU)
        self.keep_grads = False       # fused mode: also write dW (parity tests)
        self.split_lo = {}  # bf16 low-order terms of the split tensors
        self._needs_cache = {}
        self._ctx = None
        self.logits32 = None
        # {"ws": workspace} in deterministic mode (BiGanEngine): passed to every column
        # reduction, which then sums its partials in a fixed order; {} keeps the atomic path
        self.reduce_kw = {}

    def _reduce_args(self):
        return _on_main_stream(self.reduce_kw, self.opt_stream)

    # ------------------------------------------------------------------ parameters
    def _alloc_params(self, generator):
        dev = self.device
        off = 0
        meta = []
        # flat layout: every Dense kernel first, then all biases and BN gamma/beta ("small"
        # parameters) contiguously, so that with the kernels updated inside the wgrad epilogue
        # one extra launch over the tail updates everything else
        for lay in self.g.layers:
            if lay[0] == "dense":
                K, N = sum(lay[1]), lay[2]
                ldn = ops.pad_ld(N)
                # 4096-element alignment: any layer / 64-row boundary can delimit a gradient
                # bucket whose 1/world shards (world <= 16) stay 256-element aligned
                off = (off + 4095) // 4096 * 4096
                # blocked optimiser-state layout (Net._state_layout): every Concatenate segment
                # of the kernel gets its own whole 32-row blocks ("virtual rows" seg_vrow[s] =
                # sum of the earlier segments' rows rounded up to 32), so the region holds
                # Kv >= K rows; in the row-major layout the rows beyond K are zero padding
                vrow, v = [], 0
                for k_s in lay[1]:
                    vrow.append(v)
                    v += (k_s + 31) // 32 * 32
                meta.append({"kind": "dense", "K": K, "N": N, "ld": ldn, "w_off": off,
                             "act": lay[3], "in_widths": lay[1], "seg_vrow": vrow,
                             "Kv": max(v, (K + 31) // 32 * 32)})
                off += meta[-1]["Kv"] * ldn
            else:
                meta.append({"kind": "bn", "n": lay[1]})
        off = (off + 4095) // 4096 * 4096     # kernel region: shardable across up to 16 ranks
        self.small_off = off
        for m in meta:
            if m["kind"] == "dense":
                m["b_off"] = off
                off += _pad(m["N"])
            else:
                m["g_off"], m["be_off"] = off, off + _pad(m["n"])
                off += 2 * _pad(m["n"])
        # padded so that 1/world shards (world <= 16) stay 256-element aligned
        self.n_flat = max((off + 4095) // 4096 * 4096, 4096)
        self.p32 = torch.zeros(self.n_flat, dtype=torch.float32, device=dev)
        self.ms = torch.zeros_like(self.p32)
        self.mom = torch.zeros_like(self.p32)
        # data parallel on one node: the gradient and the bf16 weights live in peer-mapped
        # memory so that the fused optimiser kernel can read every rank's gradient and write
        # every rank's weights directly over NVLink
        self.peer = None
        sym = getattr(self.dist, "symmetric_zeros", None)
        got = None
        if sym is not None and _SHARD_OPTIMIZER and 64 % self.dist.world_size == 0:
            got = sym(self.n_flat * self.dist.world_size, torch.float32, dev)
        if got is not None:
            # stage[q] on rank r = rank q's gradient contribution for the elements r owns (the
            # wgrad GEMM epilogues push it there); stage[r] on rank r is r's own gradient buffer
            W, me = self.dist.world_size, self.dist.rank
            self.stage, s_ptrs, h1 = got
            self.g32 = self.stage[me * self.n_flat:(me + 1) * self.n_flat]
            self.p16, w_ptrs, h2 = sym(self.n_flat, ops.COMPUTE_DTYPE, dev)
            mc = 0
            if os.environ.get("CELLCOMM_B200_MULTICAST", "1") != "0":
                try:
                    mc = int(h2.multicast_ptr or 0)     # NVSwitch multimem mapping (0: none)
                except Exception:
                    mc = 0
            # update counter on the device: every hand-shake of update u uses epoch ctr + 1 and
            # the update's last kernel advances ctr, so the step is CUDA-graph capturable
            self.peer = {"stage": s_ptrs, "p16": w_ptrs, "p16_mc": mc, "handles": [h1, h2],
                         "ctr": torch.zeros(1, dtype=torch.int32, device=dev)}
        else:
            self.g32 = torch.zeros_like(self.p32)
            self.p16 = torch.zeros(self.n_flat, dtype=ops.COMPUTE_DTYPE, device=dev)
        # low-order bf16 term of the kernels kept as hi + lo (flat, same layout; only the
        # ranges of the `hilo` layers are ever non-zero / read)
        self.p16lo = None
        if self.hilo:
            if self.peer is not None:
                self.p16lo, lo_ptrs, h4 = sym(self.n_flat, ops.COMPUTE_DTYPE, dev)
                lo_mc = 0
                if self.peer["p16_mc"]:
                    try:
                        lo_mc = int(h4.multicast_ptr or 0)
                    except Exception:
                        lo_mc = 0
                self.peer.update(p16lo=lo_ptrs, p16lo_mc=lo_mc)
                self.peer["handles"].append(h4)
            else:
                self.p16lo = torch.zeros(self.n_flat, dtype=ops.COMPUTE_DTYPE, device=dev)
        self.layers = []
        for m in meta:
            L = dict(m)
            if m["kind"] == "dense":
                K, N, ld = m["K"], m["N"], m["ld"]
                wv = lambda buf: buf[m["w_off"]:m["w_off"] + K * ld].view(K, ld)[:, :N]
                bv = lambda buf: buf[m["b_off"]:m["b_off"] + N]
                L.update(w32=wv(self.p32), w16=wv(self.p16), dw=wv(self.g32), b32=bv(self.p32),
                         db=bv(self.g32), ms_w=wv(self.ms), mom_w=wv(self.mom))
                if len(self.layers) in self.hilo:
                    L["w16lo"] = wv(self.p16lo)
                fan = K + N
                if K > 0 and N > 0:
                    limit = math.sqrt(6.0 / fan)      # glorot_uniform (Keras Dense default)
                    u = torch.rand((K, N), generator=generator, dtype=torch.float32)
                    L["w32"].copy_(((u * 2 - 1) * limit).to(dev))
            else:
                n = m["n"]
                L.update(gamma=self.p32[m["g_off"]:m["g_off"] + n],
                         beta=self.p32[m["be_off"]:m["be_off"] + n],
                         dgamma=self.g32[m["g_off"]:m["g_off"] + n],
                         dbeta=self.g32[m["be_off"]:m["be_off"] + n],
                         moving_mean=torch.zeros(n, dtype=torch.float32, device=dev),
                         moving_var=torch.ones(n, dtype=torch.float32, device=dev),
                         sums=torch.zeros(2 * max(n, 1), dtype=torch.float32, device=dev),
                         sums2=torch.zeros(2 * max(n, 1), dtype=torch.float32, device=dev),
                         save_mean=torch.zeros(max(n, 1), dtype=torch.float32, device=dev),
                         save_rstd=torch.zeros(max(n, 1), dtype=torch.float32, device=dev))
                L["gamma"].fill_(1.0)
            self.layers.append(L)
        self.sync_compute_copy()

    def _build_buckets(self):
        """Gradient buckets of the data-parallel sharded update: contiguous ranges of the flat
        kernel region [0, small_off).  A `piece` is the row range of one Dense kernel that one
        wgrad GEMM writes (input segments of a Concatenate are separate GEMMs; segments of
        more than two buckets' worth are cut at segment-relative multiples of 64 rows, which
        keeps the X column slices TMA-aligned).  Consecutive pieces are grouped into buckets;
        a bucket is reduce-scattered when its last piece has been issued."""
        self.pieces, self.buckets = {}, []
        dense = [(i, L) for i, L in enumerate(self.layers) if L["kind"] == "dense"]
        flat = []
        for n, (i, L) in enumerate(dense):
            region_end = dense[n + 1][1]["w_off"] if n + 1 < len(dense) else self.small_off
            ro, ld = 0, L["ld"]
            segs = [k for k in L["in_widths"]]
            for si, k in enumerate(segs):
                if k == 0 or L["N"] == 0:
                    ro += k
                    continue
                nchunk = max(1, round(k * ld / _BUCKET_ELEMS))
                rows_per = max(64, ((k + nchunk - 1) // nchunk + 63) // 64 * 64) if nchunk > 1 else k
                lo = 0
                while lo < k:
                    hi = min(k, lo + rows_per)
                    last_of_layer = (si == len(segs) - 1 or not any(segs[si + 1:])) and hi == k
                    piece = {"layer": i, "seg": si, "lo": ro + lo, "hi": ro + hi,
                             "start": L["w_off"] + (ro + lo) * ld,
                             "end": region_end if last_of_layer else L["w_off"] + (ro + hi) * ld}
                    flat.append(piece)
                    self.pieces.setdefault((i, si), []).append(piece)
                    lo = hi
                ro += k
        cur = None
        for pc in flat:
            size = pc["end"] - pc["start"]
            if cur is None or cur["end"] != pc["start"] or \
                    (cur["end"] - cur["start"]) + size > _BUCKET_ELEMS * 5 // 4:
                cur = {"start": pc["start"], "end": pc["end"], "pieces": 0, "pending": 0,
                       "launched": False}
                self.buckets.append(cur)
            cur["end"] = pc["end"]
            cur["pieces"] += 1
            pc["bucket"] = cur
        # gaps (alignment padding before a region, zero-width layers) carry zero gradients and
        # zero weights: they can stay out of the collectives
        self._bucket_scratch = None
        for n, bk in enumerate(self.buckets):
            bk["index"] = n
        if self.peer is not None:
            # hand-shake flags [kind: 0 ready / 1 done][bucket, last = replicated tail][source rank]
            W, nb = self.dist.world_size, len(self.buckets) + 1
            flags, f_ptrs, h3 = self.dist.symmetric_zeros(2 * nb * W, torch.int32, self.device)
            self.peer.update(flags=flags, f=f_ptrs, nb=nb)
            self.peer["handles"].append(h3)

    def _find_narrow_layers(self):
        """Narrow Dense kernels at the head and at the tail of the flat layout (the latents' and
        the 50-300-wide trunks): `narrow` = their layer indices, `narrow_ranges` = the (at most
        two) flat ranges one RMSprop sweep each updates in fused-optimiser mode; the tail range
        runs on through the biases / BN parameters to the end of the buffer."""
        dense = [(i, L) for i, L in enumerate(self.layers) if L["kind"] == "dense"]
        small = lambda L: L["K"] * L["ld"] <= _NARROW_ELEMS
        head = []
        for i, L in dense:
            if not small(L):
                break
            head.append(i)
        tail = []
        for i, L in reversed(dense):
            if not small(L) or i in head:
                break
            tail.append(i)
        self.narrow = set(head) | set(tail)
        # wide kernels whose fp32 state may live in the blocked layout
        self.blockable = [i for i, L in dense if i not in self.narrow
                          and L["K"] > 0 and L["N"] > 128] if _BLOCKED_STATE else []
        self.state_blocked = False
        self.narrow_ranges = []
        if head:
            last = self.layers[head[-1]]
            self.narrow_ranges.append((self.layers[head[0]]["w_off"], last["w_off"] + last["K"] * last["ld"]))
        tail_start = self.layers[tail[-1]]["w_off"] if tail else self.small_off
        if self.n_flat > tail_start:
            self.narrow_ranges.append((tail_start, self.n_flat))

    def _state_layout(self, blocked):
        """Convert p32 / ms / mom of the `blockable` kernels between rows (the layout every
        view in `layers`, every flat sweep and every collective assumes) and the blocked layout
        the fused weight-gradient epilogue streams (ops.state_rows_to_blocked; include/
        cellcomm_b200.h, cc_gemm_desc.rms_blocked).  The bf16 compute copy, the gradients and
        everything else are always rows.  One layer at a time: the temporary is one kernel."""
        blocked = bool(blocked) and bool(self.blockable)
        if blocked == self.state_blocked:
            return
        if self.device.type == "cuda" and torch.cuda.is_current_stream_capturing():
            raise RuntimeError(f"{self.name}: optimiser-state layout change inside a CUDA graph "
                               f"capture (convert before capturing)")
        self._wait_optimizer()
        for i in self.blockable:
            L = self.layers[i]
            R, ld = L["Kv"], L["ld"]
            segs = [(ro, vr, k) for ro, vr, k in zip(self._seg_rows(L), L["seg_vrow"],
                                                     L["in_widths"]) if k > 0]
            moved = any(ro != vr for ro, vr, _ in segs)
            for buf in (self.p32, self.ms, self.mom):
                reg = buf[L["w_off"]:L["w_off"] + R * ld]
                if blocked:
                    rows = reg.view(R, ld)
                    if moved:     # every segment to its own block-aligned virtual rows
                        virt = torch.zeros_like(rows)
                        for ro, vr, k in segs:
                            virt[vr:vr + k] = rows[ro:ro + k]
                        rows = virt
                    reg.copy_(ops.state_rows_to_blocked(rows))
                else:
                    virt = ops.state_blocked_to_rows(reg, R, ld)
                    if moved:
                        rows = torch.zeros_like(virt)
                        for ro, vr, k in segs:
                            rows[ro:ro + k] = virt[vr:vr + k]
                        virt = rows
                    reg.copy_(virt.reshape(-1))
        self.state_blocked = blocked

    @staticmethod
    def _seg_rows(L):
        """first kernel row of every Concatenate segment in the row-major layout"""
        out, ro = [], 0
        for k in L["in_widths"]:
            out.append(ro)
            ro += k
        return out

    def _rows(self):
        """fp32 master / slots back in rows before anything but the fused epilogue touches them"""
        self._state_layout(False)

    def sync_compute_copy(self):
        """bf16 compute copy (and the low-order terms of the hi + lo kernels) <- fp32 master
        (after init / set_weights)."""
        self._rows()
        self.p16.copy_(self.p32)
        self.refresh_lo()

    def hilo_ranges(self):
        """flat [start, end) ranges of the kernels kept as hi + lo"""
        return [(self.layers[i]["w_off"], self.layers[i]["w_off"] + self.layers[i]["K"] * self.layers[i]["ld"])
                for i in sorted(self.hilo)]

    def refresh_lo(self, start=None, end=None):
        """lo = bf16(w32 - bf16(w32)) over the hi + lo kernels (restricted to the flat range
        [start, end) when given: the shard this rank just updated)."""
        for a, b in self.hilo_ranges():
            if start is not None:
                a, b = max(a, start), min(b, end)
            if b > a:
                ops.split_bf16(self.p32[a:b].view(1, -1), self.p16[a:b].view(1, -1),
                               self.p16lo[a:b].view(1, -1))

    def param_count(self):
        n = 0
        for L in self.layers:
            n += (L["K"] * L["N"] + L["N"]) if L["kind"] == "dense" else 4 * L["n"]
        return n

    def trainable_count(self):
        n = 0
        for L in self.layers:
            n += (L["K"] * L["N"] + L["N"]) if L["kind"] == "dense" else 2 * L["n"]
        return n

    def get_weights(self):
        """Creation order; Dense -> kernel[in,out], bias; BN -> gamma, beta, mean, var (host)."""
        self._wait_optimizer()
        self.gather_master()
        self._rows()
        out = []
        for L in self.layers:
            keys = ("w32", "b32") if L["kind"] == "dense" else (
                "gamma", "beta", "moving_mean", "moving_var")
            out += [L[k].detach().float().cpu().numpy().copy() for k in keys]
        return out

    def set_weights(self, arrays):
        self._wait_optimizer()
        self._rows()
        it = iter(arrays)
        for L in self.layers:
            keys = ("w32", "b32") if L["kind"] == "dense" else (
                "gamma", "beta", "moving_mean", "moving_var")
            for k in keys:
                a = torch.as_tensor(next(it), dtype=torch.float32)
                if tuple(a.shape) != tuple(L[k].shape):
                    raise ValueError(f"{self.name}: weight shape {tuple(a.shape)} != "
                                     f"{tuple(L[k].shape)}")
                if a.numel():
                    L[k].copy_(a.to(self.device))
        self.ms.zero_()
        self.mom.zero_()
        self._master_stale = self._slots_stale = False
        self.sync_compute_copy()

    # ------------------------------------------------------------------ precision policy
    def _high_precision_tensors(self):
        """(hp, split): tensors stored in fp32, and the subset consumed by GEMMs as a two-term
        bf16 expansion (hi + lo segments).

        BatchNormalization divides by the batch standard deviation, which for sigmoid features
        is ~0.02-0.05 while bf16 resolves values near 0.5 to only 0.002-0.004, so 16-bit
        storage on the way INTO a BN costs several percent of the signal (measured against the
        oracle: gradient cosines of 0.3-0.97; see DESIGN.md "precision policy").  Hence
          * everything from a Dense output to a BN input (through Dropout / Concatenate) is fp32;
          * the inputs of those Dense layers are fp32 too and enter the GEMM as hi + lo.
        Network inputs stay as fed."""
        g = self.g
        producer = {n["out"]: n for n in g.nodes}

        def closure(seeds):
            out, stack = set(), list(seeds)
            while stack:
                t = stack.pop()
                n = producer.get(t)
                if n is None or t in out:
                    continue
                out.add(t)
                if n["kind"] in ("dropout", "concat"):
                    stack.extend(n["ins"])
            return out

        hp = closure(n["ins"][0] for n in g.nodes if n["kind"] == "bn")
        split = set()
        # Dense outputs on the way into a BN: their dL/dz (the BN-backward output) sums to ~0
        # over the batch, so wgrad / dgrad / the bias gradient of the layer below are
        # cancellation-dominated and need dz as hi + lo as well.
        self.prebn = set()
        # layers whose bf16 compute copy of the KERNEL is kept as hi + lo as well (level 3): the
        # rounding of a BN-feeding kernel is amplified by 1/std of the batch like everything else
        # on the way into the BN; with W = hi + lo the forward and the input gradient of these
        # layers see the fp32 master weights to 16 mantissa bits (DESIGN.md "precision policy")
        self.hilo = set()
        if self.precision >= 2:
            for n in g.nodes:
                if n["kind"] == "dense" and n["out"] in hp:
                    if self.precision >= 3:
                        self.prebn.add(n["out"])
                        if _HILO_WEIGHTS and g.widths[n["out"]] > 0 and \
                                sum(g.widths[i] for i in n["ins"]) > 0:
                            self.hilo.add(n["layer"])
                    split.update(i for i in n["ins"] if i in producer and g.widths[i] > 0)
        if self.precision >= 1:
            # narrow tensors (latents, the 50..256-wide trunks, the encoder tail): fp32 + hi/lo
            # costs nothing and keeps the small-variance sigmoid features exact
            for n in g.nodes:
                if 0 < g.widths[n["out"]] <= _SMALL_WIDTH:
                    split.add(n["out"])
                    if n["kind"] == "dense":
                        self.prebn.add(n["out"])
        return hp | closure(split), split

    def get_slots(self):
        """RMSprop slots (ms, mom) per trainable tensor in creation order (kernel, bias | gamma,
        beta), as host arrays: checkpointing and parity tests.  Data parallel: collective (the
        sharded optimiser only keeps each rank's own 1/world of the slots current)."""
        self._wait_optimizer()
        self.gather_slots()
        self._rows()
        out = []
        for L in self.layers:
            for key in (("w32", "b32") if L["kind"] == "dense" else ("gamma", "beta")):
                out.append((self._like(L[key], self.ms).detach().cpu().numpy().copy(),
                            self._like(L[key], self.mom).detach().cpu().numpy().copy()))
        return out

    def set_slots(self, slots):
        self._wait_optimizer()
        self._rows()
        it = iter(slots)
        for L in self.layers:
            for key in (("w32", "b32") if L["kind"] == "dense" else ("gamma", "beta")):
                ms, mom = next(it)
                if L[key].numel():
                    self._like(L[key], self.ms).copy_(torch.as_tensor(ms, dtype=torch.float32))
                    self._like(L[key], self.mom).copy_(torch.as_tensor(mom, dtype=torch.float32))
        self._slots_stale = False

    def _like(self, view, flat):
        """The view of `flat` (ms / mom / g32) laid out like the parameter view `view` of p32."""
        off = view.storage_offset() - self.p32.storage_offset()
        return torch.as_strided(flat, view.shape, view.stride(), flat.storage_offset() + off)

    # ------------------------------------------------------------------ buffers
    def reserve(self, rows):
        """Grow the activation/gradient buffers to hold `rows` rows (drops the old ones)."""
        if rows > self.max_rows:
            if self.on_grow is not None:
                self.on_grow()      # captured CUDA graphs point into the buffers dropped below
            self.max_rows = int(rows)
            self.act, self.grad, self.tmp, self.shadow, self.dzb = {}, {}, {}, {}, {}
            self.split_lo = {}
            self.logits32 = None
            self._ctx = None

    def _buf(self, store, tid):
        b = store.get(tid)
        if b is None:
            wid = tid[1] if isinstance(tid, tuple) else tid
            if store is self.grad or store is self.tmp or (store is self.act and tid in self.hp):
                dtype = torch.float32
            else:
                dtype = ops.COMPUTE_DTYPE
            b = ops.alloc2d(self.max_rows, self.g.widths[wid], dtype=dtype, device=self.device)
            store[tid] = b
        return b

    def _gemm_operands(self, A, tid, rows):
        """bf16 GEMM operand(s) for activation `tid`: [x] for bf16 tensors, [hi, lo] for split
        tensors, [bf16 copy] for other fp32 tensors (prepared once per forward)."""
        ops_ = self._ctx_operands.get(tid)
        if ops_ is None:
            x = A[tid]
            if x.dtype != torch.float32:
                ops_ = [x]
            elif tid in self.split:
                hi = self._buf(self.shadow, tid)[:rows]
                lo = self._buf(self.split_lo, tid)[:rows]
                ops.split_bf16(x, hi, lo)
                ops_ = [hi, lo]
            else:
                sh = self._buf(self.shadow, tid)[:rows]
                ops.copy2d(x, sh)
                ops_ = [sh]
            self._ctx_operands[tid] = ops_
        return ops_

    def _feeds_dense(self, tid, dropout_off):
        """Is tensor `tid` consumed by a Dense layer -- directly, or (dropout_off: predict mode)
        through a Dropout, which is then the identity?  Decides whether its producer emits the
        hi / lo operands."""
        cache = self._needs_cache.setdefault(("feeds_dense", bool(dropout_off)), {})
        if tid not in cache:
            hit = False
            for n in self.g.nodes:
                if tid in n["ins"]:
                    hit = hit or n["kind"] == "dense" or \
                        (dropout_off and n["kind"] == "dropout"
                         and self._feeds_dense(n["out"], True))
            cache[tid] = hit
        return cache[tid]

    def _needs(self, train, want):
        key = (bool(train), tuple(sorted(want)))
        nd = self._needs_cache.get(key)
        if nd is None:
            nd = [False] * len(self.g.widths)
            for name, t in self.g.inputs.items():
                nd[t] = name in want
            for node in self.g.nodes:
                has_params = node["kind"] in ("dense", "bn")
                nd[node["out"]] = (train and has_params) or any(nd[i] for i in node["ins"])
            self._needs_cache[key] = nd
        return nd

    # ------------------------------------------------------------------ forward
    def forward(self, feed, rows, *, bn_train, dropout="off", masks=None, rng=None,
                pre_activation=False, out32=None):
        """feed: {input name: [rows, width] bf16 view}.  dropout: 'off' (predict), 'masks'
        (explicit uint8 keep-masks in call order) or 'rng' (rng = (seed, counter, base_id)).
        Returns the output activation ([rows, width] bf16), or fp32 logits when pre_activation."""
        self.reserve(rows)
        self._wait_optimizer()
        g = self.g
        A = {}
        for name, t in g.inputs.items():
            x = feed[name]
            if x.shape != (rows, g.widths[t]):
                raise ValueError(f"{self.name}: input '{name}' has shape {tuple(x.shape)}, "
                                 f"expected {(rows, g.widths[t])}")
            A[t] = x
        n_total = rows * self.dist.world_size
        last = g.nodes[-1]
        self._ctx_operands = {}
        for node in g.nodes:
            kind, out = node["kind"], node["out"]
            width = g.widths[out]
            if kind == "dense":
                L = self.layers[node["layer"]]
                y = self._buf(self.act, out)[:rows]
                is_last = node is last or (last["kind"] == "softmax" and last["ins"][0] == out)
                act = _ACT[node["act"]]
                wants_out32 = is_last and out32 is not None and last["kind"] != "softmax"
                dest16, dest32, copy_out = y, None, None
                if is_last and pre_activation:
                    if self.logits32 is None:
                        self.logits32 = ops.alloc2d(self.max_rows, width, dtype=torch.float32,
                                                    device=self.device)
                    dest16, dest32, act = None, self.logits32[:rows], 0
                elif y.dtype == torch.float32:           # fp32 activation (precision policy)
                    dest16, dest32 = None, y
                    copy_out = out32 if wants_out32 else None
                elif wants_out32:
                    dest32 = out32
                if width > 0:
                    segs, second, ro = [], [], 0          # (operand, kernel row offset, kernel)
                    wlo = L.get("w16lo")
                    for i in node["ins"]:
                        if g.widths[i] > 0:
                            terms = self._gemm_operands(A, i, rows)
                            segs += [(t, ro, L["w16"]) for t in terms]
                            if wlo is not None:
                                # kernel kept as hi + lo: x_hi @ W_lo, and the second-order
                                # x_lo @ W_lo while the segment list has room for it
                                segs.append((terms[0], ro, wlo))
                                second += [(t, ro, wlo) for t in terms[1:]]
                        ro += g.widths[i]
                    # (second-order terms, 2^-16 relative, only where arithmetic is emulated
                    # exactly: the host-logic tests compare at 1e-4; on the GPU they would cost
                    # a fourth GEMM segment for less than the bf16 rounding of everything else)
                    if second and self.device.type != "cuda" and len(segs) + len(second) <= 4:
                        segs += second
                    xs, offs, ws = ([sg[j] for sg in segs] for j in range(3))
                    hi_lo = None
                    if (dest32 is y and dest16 is None and out in self.split
                            and self._feeds_dense(out, dropout == "off")):
                        # a Dense consumes this fp32 output as hi + lo: the epilogue emits both
                        # bf16 terms next to the fp32 value (no split pass before the consumer)
                        hi_lo = (self._buf(self.shadow, out)[:rows],
                                 self._buf(self.split_lo, out)[:rows])
                        self._ctx_operands[out] = list(hi_lo)
                    if xs:
                        ops.dense_fwd(xs, ws, offs, L["b32"], act, out16=dest16, out32=dest32,
                                      hi_lo=hi_lo)
                    else:
                        ops.bias_act(L["b32"], act, rows, out16=dest16, out32=dest32)
                        self._ctx_operands.pop(out, None)     # (nothing emitted hi / lo)
                    if copy_out is not None:
                        ops.copy2d(y, copy_out)
                A[out] = y
            elif kind == "softmax":
                y = self._buf(self.act, out)[:rows]
                if width > 0:
                    ops.softmax_fwd(A[node["ins"][0]], y16=y, y32=out32)
                A[out] = y
            elif kind == "bn":
                L = self.layers[node["layer"]]
                x = A[node["ins"][0]]
                y = self._buf(self.act, out)[:rows]
                if width > 0:
                    if bn_train:
                        ops.bn_stats(x, L["sums"], **self._reduce_args())
                        self.dist.all_reduce(L["sums"])
                        ops.bn_train_apply(x, y, L["sums"], n_total, L["gamma"], L["beta"],
                                           BN_EPS, BN_MOMENTUM, L["moving_mean"], L["moving_var"],
                                           L["save_mean"], L["save_rstd"])
                    else:
                        ops.bn_infer(x, y, L["gamma"], L["beta"], L["moving_mean"],
                                     L["moving_var"], BN_EPS)
                A[out] = y
            elif kind == "dropout":
                x = A[node["ins"][0]]
                if dropout == "off":
                    A[out] = x
                    src = node["ins"][0]     # predict: the identity; reuse prepared operands
                    if src in self._ctx_operands and (out in self.split) == (src in self.split):
                        self._ctx_operands[out] = self._ctx_operands[src]
                else:
                    y = self._buf(self.act, out)[:rows]
                    if width > 0:
                        self._dropout(node, x, y, dropout, masks, rng)
                    A[out] = y
            elif kind == "concat":
                y = self._buf(self.act, out)[:rows]
                c = 0
                for i in node["ins"]:
                    w = g.widths[i]
                    if w > 0:
                        ops.copy2d(A[i], y[:, c:c + w])
                    c += w
                A[out] = y
        self._ctx = {"rows": rows, "bn_train": bn_train, "dropout": dropout, "masks": masks,
                     "rng": rng, "A": A, "pre_activation": pre_activation, "n_total": n_total,
                     "operands": self._ctx_operands}
        if pre_activation:
            return self.logits32[:rows]
        return A[g.output]

    def _dropout(self, node, x, y, mode, masks, rng):
        if mode == "masks":
            m = masks[node["drop"]]
            if m.shape != x.shape:
                raise ValueError(f"{self.name}: dropout mask {node['drop']} has shape "
                                 f"{tuple(m.shape)}, expected {tuple(x.shape)}")
            ops.dropout(x, y, node["rate"], mask=m)
        else:
            seed, counter, base = rng
            ops.dropout(x, y, node["rate"], seed=seed, counter=counter,
                        stream_id=base + node["drop"])

    # ------------------------------------------------------------------ backward
    def _emit(self, tid, rows, state, fn):
        """Write (first contribution) or accumulate (later ones) a gradient for tensor `tid`."""
        dst = self._buf(self.grad, tid)[:rows]
        if not state[tid]:
            fn(dst)
            state[tid] = True
        else:
            t = self._buf(self.tmp, tid)[:rows]
            fn(t)
            ops.copy2d(t, dst, beta=1)

    def output_grad(self, rows):
        """fp32 buffer for dL/d(output); a loss kernel may write it in place and pass it to
        backward(), which then skips the seed copy."""
        return self._buf(self.grad, self.g.output)[:rows]

    def backward(self, dout, *, train, want=()):
        """dout: gradient w.r.t. the output (bf16 [rows, width]); for a pre_activation forward it
        is the gradient w.r.t. the final layer's logits.  train=True fills this net's parameter
        gradients; `want` names the inputs whose gradients are returned."""
        c = self._ctx
        self._wait_optimizer()
        g, rows, A = self.g, c["rows"], c["A"]
        needs = self._needs(train, want)
        state = [False] * len(g.widths)
        if train and self._bucketed():
            for bk in self.buckets:
                bk["pending"], bk["launched"] = bk["pieces"], False
        if train:
            # wide kernels' fp32 state in the blocked layout while the fused epilogue owns them
            # (a no-op from the second step on), in rows for every other update path
            self._state_layout(self.fuse_optimizer)
        if train and self.n_flat > self.small_off:
            # ONE fill for every bias gradient of the network (they lie contiguously behind the
            # kernels in the flat gradient buffer); the per-layer reductions then accumulate
            ops.fill_f32(self.g32[self.small_off:], 0.0)

        out_t = g.output
        ext = {}      # gradient tensors read in place instead of from this net's own buffers
        if dout.dtype == torch.float32 and dout.dim() == 2 and dout.stride(1) == 1 and \
                dout.shape[1] == g.widths[out_t]:
            # e.g. dL/d(cell) out of the frozen discriminator's backward: 276 MB at batch 2048
            # that would otherwise be copied into this net's seed buffer
            ext[out_t] = dout[:rows]
        elif g.widths[out_t] > 0:
            ops.copy2d(dout, self._buf(self.grad, out_t)[:rows])
        state[out_t] = True
        last = g.nodes[-1]
        for node in reversed(g.nodes):
            kind, out = node["kind"], node["out"]
            if not state[out] or not needs[out]:
                continue
            width = g.widths[out]
            dy = ext[out] if out in ext else self.grad[out][:rows]
            if kind == "dense":
                L = self.layers[node["layer"]]
                if width == 0:
                    continue
                is_last = node is last or (last["kind"] == "softmax" and last["ins"][0] == out)
                act = _ACT[node["act"]]
                if is_last and c["pre_activation"]:
                    act = 0
                # fp32 dL/dy -> bf16 dL/dz = dy * act'(y): the GEMM operand of wgrad / dgrad
                dz = self._buf(self.dzb, out)[:rows]
                if out in self.prebn:
                    # dz as hi + lo (two GEMM segments), and the bias gradient from the fp32
                    # product, in ONE pass over dy and y (frozen layers: no bias gradient)
                    dz_lo = self._buf(self.split_lo, ("dz", out))[:rows]
                    ops.bias_grad(dy, A[out], act, L["db"] if train else None, dz=dz, beta=1,
                                  dz_lo=dz_lo, **self._reduce_args())
                    dzs = [dz, dz_lo]
                elif train:
                    # one pass over dy and y: dz for the GEMMs and the bias gradient
                    ops.bias_grad(dy, A[out], act, L["db"], dz=dz, beta=1, **self._reduce_args())
                    dzs = [dz]
                else:
                    ops.act_bwd(dy, A[out], dz, act)
                    dzs = [dz]
                ro = 0
                for seg_index, i in enumerate(node["ins"]):
                    k = g.widths[i]
                    if k > 0:
                        # input gradient first: it must see this layer's weights BEFORE the
                        # fused wgrad epilogue below updates them
                        if needs[i]:
                            wseg = L["w16"][ro:ro + k]
                            dst = self._buf(self.grad, i)[:rows]
                            d_terms, w_terms = list(dzs), [wseg] * len(dzs)
                            if "w16lo" in L:         # dz_hi @ W_lo^T (+ dz_lo @ W_lo^T, see forward)
                                n_lo = 1 if self.device.type == "cuda" else 4 - len(dzs)
                                for d_ in dzs[:n_lo]:
                                    d_terms.append(d_)
                                    w_terms.append(L["w16lo"][ro:ro + k])
                            ops.dense_dgrad(d_terms, w_terms, dst, beta=1 if state[i] else 0)
                            state[i] = True
                        if train:
                            xs = c["operands"][i]
                            # all hi/lo cross terms except lo*lo
                            pairs = [(x, d) for a, x in enumerate(xs) for b, d in enumerate(dzs)
                                     if a + b < 2]
                            rms, row0, lo_out = None, None, None
                            if self.fuse_optimizer and node["layer"] not in self.narrow:
                                sl = slice(ro, ro + k)
                                if self.state_blocked and node["layer"] in self.blockable:
                                    lo_out = L["w16lo"][sl] if "w16lo" in L else None
                                    # the layer's blocked arrays + this segment's first row
                                    a = L["w_off"]
                                    b = a + L["Kv"] * L["ld"]
                                    rms = (self.p32[a:b], L["w16"][sl], self.ms[a:b], self.mom[a:b],
                                           LR, RHO, MOMENTUM, EPSILON)
                                    row0 = L["seg_vrow"][seg_index]   # block-aligned
                                else:
                                    rms = (L["w32"][sl], L["w16"][sl], L["ms_w"][sl], L["mom_w"][sl],
                                           LR, RHO, MOMENTUM, EPSILON)
                            if self._bucketed():
                                # data parallel: one GEMM per gradient piece, and the piece's
                                # bucket goes to the side stream as soon as it is complete
                                for pc in self.pieces.get((node["layer"], seg_index), ()):
                                    a, b = pc["lo"] - ro, pc["hi"] - ro
                                    ops.dense_wgrad([p_[0][:, a:b] for p_ in pairs],
                                                    [p_[1] for p_ in pairs],
                                                    L["dw"][pc["lo"]:pc["hi"]],
                                                    route=self._route(pc))
                                    self._piece_done(pc)
                            else:
                                dw = L["dw"][ro:ro + k] if (rms is None or self.keep_grads) else None
                                ops.dense_wgrad([p_[0] for p_ in pairs], [p_[1] for p_ in pairs],
                                                dw, rms=rms, rms_row0=row0, rms_lo=lo_out)
                    ro += k
                if train:
                    if self.fuse_optimizer and "w16lo" in L and node["layer"] not in self.narrow \
                            and not (self.state_blocked and node["layer"] in self.blockable):
                        # the wgrad epilogues above just updated this kernel: new low-order term
                        ops.split_bf16(L["w32"], L["w16"], L["w16lo"])
            elif kind == "softmax":
                i = node["ins"][0]
                if width > 0 and needs[i]:
                    self._emit(i, rows, state, lambda d: ops.softmax_bwd(dy, A[out], d))
            elif kind == "bn":
                L = self.layers[node["layer"]]
                i = node["ins"][0]
                if width == 0:
                    continue
                x = A[i]
                if c["bn_train"]:
                    ops.bn_bwd_stats(dy, x, L["save_mean"], L["save_rstd"], L["sums2"],
                                     **self._reduce_args())
                    if train:
                        # dgamma / dbeta from the LOCAL sums: the flat gradient all-reduce in
                        # apply_rmsprop() adds the other ranks' shares
                        ops.bn_bwd_apply(dy, x, None, L["gamma"], L["save_mean"], L["save_rstd"],
                                         L["sums2"], c["n_total"], L["dgamma"], L["dbeta"])
                    self.dist.all_reduce(L["sums2"])
                    if needs[i]:
                        self._emit(i, rows, state, lambda d: ops.bn_bwd_apply(
                            dy, x, d, L["gamma"], L["save_mean"], L["save_rstd"], L["sums2"],
                            c["n_total"]))
                else:
                    if train:
                        raise RuntimeError("training a BatchNormalization in inference mode")
                    if needs[i]:
                        self._emit(i, rows, state, lambda d: ops.bn_infer_bwd(
                            dy, d, L["gamma"], L["moving_var"], BN_EPS))
            elif kind == "dropout":
                i = node["ins"][0]
                if width > 0 and needs[i]:
                    if c["dropout"] == "off":
                        self._emit(i, rows, state, lambda d: ops.copy2d(dy, d))
                    else:
                        self._emit(i, rows, state, lambda d: self._dropout(
                            node, dy, d, c["dropout"], c["masks"], c["rng"]))
            elif kind == "concat":
                col = 0
                for i in node["ins"]:
                    w = g.widths[i]
                    if w > 0 and needs[i]:
                        src = dy[:, col:col + w]
                        dst = self._buf(self.grad, i)[:rows]
                        ops.copy2d(src, dst, beta=1 if state[i] else 0)
                        state[i] = True
                    col += w
        grads = {}
        for name in want:
            t = g.inputs[name]
            if not state[t]:
                # zero-width layers (the 5-gene fixture's Dense(0)) cut the path: gradient is 0
                self._buf(self.grad, t).zero_()
            grads[name] = self.grad[t][:rows]
        return grads

    # ------------------------------------------------------------------ optimiser
    def apply_rmsprop(self):
        """Keras RMSprop(lr=0.0075, rho=0.85, momentum=0.1) over the flat parameter buffer in
        one launch; padding has zero gradient and stays zero.  In data-parallel runs the flat
        gradient is all-reduced (sum of per-rank partial sums) first.  With `fuse_optimizer`
        the Dense kernels were already updated inside their wgrad epilogues (the gradient
        never went to HBM) and only the small tail (biases, BN gamma/beta) is updated here."""
        if self.fuse_optimizer:
            # the narrow kernels (gradient in g32, written by their split-K wgrad) and the
            # biases / BN parameters: one flat sweep per contiguous range
            for a, b in self.narrow_ranges:
                sl = slice(a, b)
                ops.rmsprop_step(self.p32[sl], self.p16[sl], self.g32[sl], self.ms[sl],
                                 self.mom[sl], LR, RHO, MOMENTUM, EPSILON)
                self.refresh_lo(a, b)
            return
        if self.opt_stream is None:
            self._reduce_and_update()
            return
        main = torch.cuda.current_stream()
        self.opt_stream.wait_stream(main)           # gradients are complete
        with torch.cuda.stream(self.opt_stream):
            self._reduce_and_update()
            self._opt_event = torch.cuda.Event()
            self._opt_event.record(self.opt_stream)

    def _bucketed(self):
        """Data-parallel sharded update in per-bucket collectives (world a power of two <= 16:
        every bucket is a multiple of 64 elements, so 1/world shards stay 16-byte aligned)."""
        W = self.dist.world_size
        return (W > 1 and _SHARD_OPTIMIZER and not self.fuse_optimizer and 64 % W == 0
                and len(self.buckets) > 0)

    def _piece_done(self, pc):
        bk = pc["bucket"]
        bk["pending"] -= 1
        if bk["pending"] == 0:
            self._launch_bucket(bk)

    def _launch_bucket(self, bk):
        """reduce-scatter -> RMSprop on this rank's shard -> all-gather of the bf16 weights, for
        one bucket, on the optimiser stream (ordered after the gradient's wgrad GEMMs)."""
        if bk["launched"]:
            return
        bk["launched"] = True
        if _DP_SKIP_UPDATE:
            return
        W, r = self.dist.world_size, self.dist.rank
        n = (bk["end"] - bk["start"]) // W
        sl = slice(bk["start"] + r * n, bk["start"] + (r + 1) * n)
        if self._bucket_scratch is None and self.peer is None:
            biggest = max(b["end"] - b["start"] for b in self.buckets) // W
            self._bucket_scratch = torch.empty(biggest, dtype=torch.float32, device=self.device)
        shard = self._bucket_scratch[:n] if self.peer is None else None

        def run_peer():
            self._peer_update(bk["index"], bk["start"] + r * n, n, broadcast=True)

        def run():
            if self.peer is not None:
                return run_peer()
            self.dist.reduce_scatter(shard, self.g32[bk["start"]:bk["end"]])
            ops.rmsprop_step(self.p32[sl], self.p16[sl], shard, self.ms[sl], self.mom[sl], LR, RHO,
                             MOMENTUM, EPSILON)
            has_lo = any(a < bk["end"] and b > bk["start"] for a, b in self.hilo_ranges())
            if has_lo:
                self.refresh_lo(sl.start, sl.stop)
            self.dist.all_gather(self.p16[bk["start"]:bk["end"]], self.p16[sl])
            if has_lo:
                self.dist.all_gather(self.p16lo[bk["start"]:bk["end"]], self.p16lo[sl])

        if self.opt_stream is None:
            run()
            return
        self.opt_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.opt_stream):
            run()

    def _flag_ptr(self, on_rank, kind, bucket, source):
        pr = self.peer
        return pr["f"][on_rank] + 4 * ((kind * pr["nb"] + bucket) * self.dist.world_size + source)

    def _route(self, pc):
        """cc_gemm_desc.route_* for the wgrad GEMM of gradient piece `pc`: every element goes
        straight to the rank that owns it in the sharded update (my slot of its staging buffer)."""
        if self.peer is None:
            return None
        W, me, bk = self.dist.world_size, self.dist.rank, pc["bucket"]
        base = 4 * (me * self.n_flat + bk["start"])
        return (W, (bk["end"] - bk["start"]) // W, pc["start"] - bk["start"],
                [self.peer["stage"][r] + base for r in range(W)])

    def _peer_update(self, bucket, start, count, broadcast):
        """signal "my gradient of this bucket is complete" -> fused peer-memory optimiser kernel
        -> signal "consumed / my shard is written" (csrc/peer_optimizer.cu)."""
        pr, W, r = self.peer, self.dist.world_size, self.dist.rank
        ops.peer_signal([self._flag_ptr(t, 0, bucket, r) for t in range(W)], 1, epoch_ctr=pr["ctr"])
        if broadcast:   # sharded bucket: all contributions were pushed into MY staging slots
            grads = [pr["stage"][r] + 4 * q * self.n_flat for q in range(W)]
        else:           # replicated tail: pull every rank's own (small) gradient
            grads = [pr["stage"][q] + 4 * q * self.n_flat for q in range(W)]
        lo = None
        if self.hilo and broadcast:
            lo = (pr["p16lo"], pr["p16lo_mc"], self.hilo_ranges())
        ops.peer_rmsprop(W, r, grads, pr["p16"], self.p32, self.ms, self.mom, start, count,
                         broadcast, LR, RHO, MOMENTUM, EPSILON, self._flag_ptr(r, 0, bucket, 0),
                         1, p16_multicast=pr["p16_mc"], epoch_ctr=pr["ctr"], lo=lo)
        ops.peer_signal([self._flag_ptr(t, 1, bucket, r) for t in range(W)], 1, epoch_ctr=pr["ctr"])

    def _reduce_and_update(self):
        """Data-parallel update.  world == 1: one sweep.  world > 1 (ZeRO-1 style): reduce-scatter
        the fp32 gradient, RMSprop on this rank's 1/world shard of the flat buffers (1/world of
        the 30 B/parameter optimiser traffic), all-gather the bf16 compute copy.  The fp32
        master copy is then only current on its owner shard; gather_master() refreshes it."""
        W = self.dist.world_size
        K = self.small_off                      # Dense kernels: [0, K); biases + BN: [K, n_flat)
        if self._bucketed():
            # most buckets were launched from backward(); flush the rest (layers the backward
            # pass did not reach), then the replicated update of biases and BN gamma/beta
            for bk in self.buckets:
                self._launch_bucket(bk)
            if _DP_SKIP_UPDATE:
                return
            if self.peer is not None:
                # biases + BN gamma/beta: replicated update from the sum of all ranks' gradients,
                # then wait until every rank has consumed every bucket of this update (my
                # gradient buffer may be rewritten, my bf16 weights are complete)
                pr = self.peer
                self._peer_update(pr["nb"] - 1, K, self.n_flat - K, broadcast=False)
                ops.peer_wait(self._flag_ptr(self.dist.rank, 1, 0, 0),
                              pr["nb"] * self.dist.world_size, 1, epoch_ctr=pr["ctr"], bump=True)
                self.mark_updated()
                return
            tail = slice(K, self.n_flat)
            self.dist.all_reduce_grad(self.g32[tail])
            ops.rmsprop_step(self.p32[tail], self.p16[tail], self.g32[tail], self.ms[tail],
                             self.mom[tail], LR, RHO, MOMENTUM, EPSILON)
            self.mark_updated()
            return
        if W == 1 or not _SHARD_OPTIMIZER or K == 0 or K % (W * 256) != 0:
            self.dist.all_reduce(self.g32)
            ops.rmsprop_step(self.p32, self.p16, self.g32, self.ms, self.mom, LR, RHO, MOMENTUM,
                             EPSILON)
            self.refresh_lo()
            return
        n = K // W
        sl = slice(self.dist.rank * n, (self.dist.rank + 1) * n)
        if self._gshard is None:
            self._gshard = torch.empty(n, dtype=torch.float32, device=self.device)
        self.dist.reduce_scatter(self._gshard, self.g32[:K])
        ops.rmsprop_step(self.p32[sl], self.p16[sl], self._gshard, self.ms[sl], self.mom[sl], LR,
                         RHO, MOMENTUM, EPSILON)
        if self.hilo:
            self.refresh_lo(sl.start, sl.stop)
        self.dist.all_gather(self.p16[:K], self.p16[sl])
        if self.hilo:
            self.dist.all_gather(self.p16lo[:K], self.p16lo[sl])
        # biases and BN gamma/beta are read in fp32 by the forward kernels: replicated update
        tail = slice(K, self.n_flat)
        self.dist.all_reduce(self.g32[tail])
        ops.rmsprop_step(self.p32[tail], self.p16[tail], self.g32[tail], self.ms[tail],
                         self.mom[tail], LR, RHO, MOMENTUM, EPSILON)
        self.mark_updated()

    def _gather_sharded(self, flat):
        """all-gather every rank's owner shard of a flat fp32 buffer (p32 / ms / mom)"""
        W, r = self.dist.world_size, self.dist.rank
        if self._bucketed():
            ranges = [(b["start"], b["end"]) for b in self.buckets]
        else:
            ranges = [(0, self.small_off)]
        for a, b in ranges:
            n = (b - a) // W
            self.dist.all_gather(flat[a:b], flat[a + r * n:a + (r + 1) * n].clone())

    def mark_updated(self):
        """The sharded optimiser ran (possibly inside a replayed CUDA graph, where no Python
        executes): the non-owned parts of p32 / ms / mom are stale until gathered."""
        if self.dist.world_size > 1 and _SHARD_OPTIMIZER and not self.fuse_optimizer:
            self._master_stale = self._slots_stale = True

    def gather_master(self):
        """Make the fp32 master weights current on every rank (sharded-optimiser runs).
        Collective: every rank calls it."""
        if self._master_stale and self.dist.world_size > 1:
            self._gather_sharded(self.p32)
        self._master_stale = False

    def gather_slots(self):
        """Same for the RMSprop slots: each rank updates ms / mom only on its own shard, so a
        checkpoint (or any reader of the slots) needs the owners' values.  Collective."""
        if self._slots_stale and self.dist.world_size > 1:
            self._gather_sharded(self.ms)
            self._gather_sharded(self.mom)
        self._slots_stale = False

    def _wait_optimizer(self):
        """Order the current stream after a pending side-stream update of this net."""
        if self._opt_event is not None:
            torch.cuda.current_stream().wait_event(self._opt_event)
            self._opt_event = None

    def synchronize(self):
        self._wait_optimizer()


class LossScalar:
    """A loss that stays on the device until someone needs the number (float(), format, print).
    `CellTraining.run` sums these per iteration (src/cell_type_training.py:45-48) without a
    host sync per step."""

    __slots__ = ("t",)

    def __init__(self, t):
        self.t = t

    def __float__(self):
        return float(self.t)

    def item(self):
        return float(self.t)

    def _v(self, o):
        return o.t if isinstance(o, LossScalar) else o

    def __add__(self, o):
        return LossScalar(self.t + self._v(o))

    __radd__ = __add__

    def __sub__(self, o):
        return LossScalar(self.t - self._v(o))

    def __mul__(self, o):
        return LossScalar(self.t * self._v(o))

    __rmul__ = __mul__

    def __truediv__(self, o):
        return LossScalar(self.t / self._v(o))

    def __format__(self, spec):
        return format(float(self), spec)

    def __repr__(self):
        return repr(float(self))

    def __lt__(self, o):
        return float(self) < float(o)

    def __gt__(self, o):
        return float(self) > float(o)

    def __eq__(self, o):
        return float(self) == float(o)

    def __hash__(self):
        return id(self)


class GraphedStep:
    """One trainings_step on `batch` rows captured as a CUDA graph (see capture_step)."""

    def __init__(self, eng, csr, n_cols, batch, latents):
        self.eng, self.batch, self.latents = eng, int(batch), latents
        rowptr, colidx, values = csr
        dev = eng.device
        eng.reserve(batch)
        self.idx = torch.zeros(batch, dtype=torch.int64, device=dev)
        self.x16 = ops.alloc2d(batch, n_cols, device=dev)
        saved = [(n, n.opt_stream) for n in eng.nets.values()]
        for n, _ in saved:
            n._wait_optimizer()
            if eng.dist.world_size == 1:         # single GPU: nothing runs on the side stream
                n.opt_stream = None
        # data parallel (peer-memory path): the gradient exchange / update kernels stay on the
        # optimiser stream; it forks from and joins the capturing stream inside the graph

        def body():
            ops.gather_rows(rowptr, colidx, values, n_cols, row_idx=self.idx, out16=self.x16)
            if latents == "device":
                eng.draw_latents(batch)
            else:
                ops.cast_f32_to_bf16(eng.z32[:batch], eng.z16[:batch])
                ops.cast_f32_to_bf16(eng.r32[:batch], eng.r16[:batch])
            out = eng.train_step(self.x16)
            eng.join()                           # side-stream work joins before the capture ends
            return out

        try:
            # warm-up run (allocates lazy buffers, sets kernel attributes, fills the tensor-map
            # cache) on a side stream as torch requires; it is a real training step, so the
            # model / optimiser / RNG state is snapshotted and restored around it
            for n in eng.nets.values():
                n._state_layout(n.fuse_optimizer)        # not inside the capture
            self._layouts = {k: n.state_blocked for k, n in eng.nets.items()}
            snap = eng.snapshot_state()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                body()
            torch.cuda.current_stream().wait_stream(side)
            eng.restore_state(snap)
            del snap
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            l0 = ops.launch_count()
            with torch.cuda.graph(self.graph):
                self.losses = body()
            # kernels of libcellcomm_b200.so captured in the graph (each replay runs them all)
            self.launches_per_replay = ops.launch_count() - l0
        finally:
            for n, st in saved:
                n.opt_stream = st

    def replay(self, idx=None):
        """idx: batch row positions (host or device int64); None keeps the current buffer."""
        if idx is not None:
            self.idx.copy_(torch.as_tensor(idx), non_blocking=True)
        for k, n in self.eng.nets.items():
            n._state_layout(self._layouts[k])      # e.g. get_weights() put the state back in rows
        self.graph.replay()
        for n in self.eng.nets.values():
            n.mark_updated()          # no Python ran inside the graph (sharded data-parallel update)
        # fresh device scalars: the graph's own loss tensors are overwritten by the next replay
        # (train_on_batch returns independent floats in the reference)
        return tuple(LossScalar(l.t.clone()) for l in self.losses)


class BiGanEngine:
    """G, E, D plus the eight sub-steps of `trainings_step` (src/bigan_classify.py:126-155)."""

    SUBSTEP_NETS = {1: ("G", "D"), 2: ("E", "G"), 3: ("E", "D"), 4: ("G", "E"), 6: ("D",),
                    8: ("D",)}

    def __init__(self, variant, encoding_size, gene_size, max_batch=128, device="cuda", seed=None,
                 dist=None, graphs=None, deterministic=False):
        """variant 'cont' | 'classify' picks the reference graphs and whether sub-step 7 feeds
        one_hot(argmax) (classify, src/bigan_classify.py:121-124) or the raw encoding (cont,
        src/bigan_cont.py:55-56) to D.  `graphs` = {"G","E","D": GraphBuilder} overrides them.

        deterministic=True: every column reduction (bias gradients, BatchNormalization
        statistics and backward sums) and the MSE losses sum their partials in a fixed order
        through one workspace, so a run is a pure function of its inputs and seed on a given
        GPU count and build (DESIGN.md section 2).  One workspace serves the whole step because
        every reduction runs on the current (main) stream; the optimiser side stream runs only
        RMSprop sweeps and gradient exchanges."""
        if variant not in ("cont", "classify"):
            raise ValueError(f"unknown variant {variant}")
        self.variant, self.Z, self.Gn = variant, int(encoding_size), int(gene_size)
        self.device = torch.device(device)
        self.dist = dist or _NoDist()
        gen = torch.Generator()
        if seed is None:
            gen.seed()
        else:
            gen.manual_seed(int(seed))
        if graphs is None:
            gg = cont_generator_graph if variant == "cont" else classify_generator_graph
            eg = cont_encoder_graph if variant == "cont" else classify_encoder_graph
            graphs = {"G": gg(self.Z, self.Gn), "E": eg(self.Z, self.Gn),
                      "D": discriminator_graph(self.Z, self.Gn)}
        self.G = Net(graphs["G"], max_batch, self.device, gen, self.dist, precision=3)
        self.E = Net(graphs["E"], max_batch, self.device, gen, self.dist)
        self.D = Net(graphs["D"], max_batch, self.device, gen, self.dist)
        self.nets = {"G": self.G, "E": self.E, "D": self.D}
        self._graphs = {}
        for n in self.nets.values():
            n.on_grow = self._graphs.clear
        # single GPU: Keras RMSprop is applied inside the wgrad GEMM epilogues (the accumulator IS
        # the gradient: 26 B/parameter of optimiser traffic instead of a 4 B gradient write plus a
        # 30 B/parameter sweep; -2.9 ms per 2048-cell step, profiles/README.md).  Data parallel
        # runs must reduce the gradient first and use the sharded flat sweep instead.
        # CELLCOMM_B200_FUSE_OPT=0 selects the flat sweep on one GPU too.
        self.set_fused_optimizer(self.dist.world_size == 1 and self.device.type == "cuda" and
                                 os.environ.get("CELLCOMM_B200_FUSE_OPT", "1") == "1")
        if self.device.type == "cuda" and os.environ.get("CELLCOMM_B200_ASYNC_OPT", "1") != "0":
            side = torch.cuda.Stream(device=self.device)
            for n in self.nets.values():
                n.opt_stream = side
        self.loss_buf = torch.zeros(8, dtype=torch.float32, device=self.device)
        self.rng_seed = int(torch.randint(0, 2 ** 62, (1,), generator=gen).item())
        if self.dist.world_size > 1:
            # replicas start from rank 0's weights and RNG key (seed=None draws a different
            # initialisation in every process); the rank is folded into the Philox stream ids
            # below, so every rank draws its own dropout masks / priors for its rows
            bcast = getattr(self.dist, "broadcast", None)
            if bcast is not None:
                key = torch.tensor([self.rng_seed], dtype=torch.int64, device=self.device)
                bcast(key)
                self.rng_seed = int(key.item())
                for n in self.nets.values():
                    bcast(n.p32)
                    n.sync_compute_copy()
        self._rank_stream = (self.dist.rank & 0xFFF) << 12
        self.rng_counter = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.deterministic = bool(deterministic)
        self.reduce_kw = {}
        self.max_batch = 0
        self.reserve(max_batch)

    def _reduce_args(self):
        return _on_main_stream(self.reduce_kw, self.G.opt_stream)   # one side stream for all nets

    def set_fused_optimizer(self, on, keep_grads=False):
        """Single-GPU: apply RMSprop to every Dense kernel inside its wgrad GEMM epilogue.
        keep_grads also writes the gradients (parity tests compare them)."""
        if on and self.dist.world_size > 1:
            raise ValueError("the fused optimiser needs the gradient all-reduce to be a no-op")
        for n in self.nets.values():
            n.fuse_optimizer, n.keep_grads = bool(on), bool(keep_grads)

    def reserve(self, rows):
        """(Re)allocate the per-step staging buffers for batches of up to `rows` rows."""
        rows = int(rows)
        if rows <= self.max_batch:
            return
        self._graphs.clear()           # captured steps hold pointers into the old buffers
        self.max_batch = mb = rows
        Z, dev = self.Z, self.device
        for n in self.nets.values():
            n.reserve(mb)
        self.z16 = ops.alloc2d(mb, Z, device=dev)
        self.r16 = ops.alloc2d(mb, Z, device=dev)
        self.z32 = ops.alloc2d(mb, Z, dtype=torch.float32, device=dev)
        self.r32 = ops.alloc2d(mb, Z, dtype=torch.float32, device=dev)
        self.gen_cells = None
        self.gen_enc16 = ops.alloc2d(mb, Z, device=dev)
        self.gen_enc32 = ops.alloc2d(mb, Z, dtype=torch.float32, device=dev)
        if self.deterministic:
            # fixed-order reduction workspace for batches of up to mb rows and the widest
            # tensor of the three networks; zeroed, as its ticket counters must start at 0
            widest = max(max(n.g.widths) for n in self.nets.values())
            self.reduce_ws = torch.zeros(ops.reduce_ws_floats(mb, max(widest, self.Gn, Z)),
                                         dtype=torch.float32, device=dev)
            self.reduce_kw = {"ws": self.reduce_ws}
            for n in self.nets.values():
                n.reduce_kw = self.reduce_kw

    # ------------------------------------------------------------------ helpers
    def _drop_args(self, substep, net, masks):
        if masks is not None:
            return {"dropout": "masks", "masks": masks[substep][net]}
        base = self._rank_stream + substep * 16 + {"G": 0, "E": 4, "D": 8}[net]
        return {"dropout": "rng", "rng": (self.rng_seed, self.rng_counter, base)}

    def set_latents(self, encodings, noise, rows):
        """Stage the step's prior samples (host or device, fp32) as fp32 + bf16 device views."""
        self.reserve(rows)
        z32, r32 = self.z32[:rows], self.r32[:rows]
        z32.copy_(torch.as_tensor(encodings, dtype=torch.float32), non_blocking=True)
        r32.copy_(torch.as_tensor(noise, dtype=torch.float32), non_blocking=True)
        ops.cast_f32_to_bf16(z32, self.z16[:rows])
        ops.cast_f32_to_bf16(r32, self.r16[:rows])

    def draw_latents(self, rows):
        """tf.random.uniform priors on the device (src/bigan_basic.py:36-37, bigan_cont.py:52-53)."""
        self.reserve(rows)
        ops.uniform(out32=self.z32[:rows], out16=self.z16[:rows], seed=self.rng_seed,
                    counter=self.rng_counter, stream_id=self._rank_stream + 1000)
        ops.uniform(out32=self.r32[:rows], out16=self.r16[:rows], seed=self.rng_seed,
                    counter=self.rng_counter, stream_id=self._rank_stream + 1001)

    # ------------------------------------------------------------------ the step
    def train_step(self, x16, masks=None):
        """One `trainings_step` on the batch x16 ([B, gene_size] bf16 view).  The priors must
        have been staged with set_latents()/draw_latents().  Returns (g, e, d) LossScalars."""
        B = x16.shape[0]
        if B > self.max_batch:
            raise ValueError(f"batch of {B} rows: stage the priors (set_latents/draw_latents) first")
        ops.fill_f32(self.loss_buf, 0.0)
        for k in (1, 2, 3, 4, 5, 6, 7, 8):
            self.substep(k, x16, masks)
        return self.finish_step(masks)

    def substep(self, k, x16, masks=None):
        """Sub-step k (1..8) of `trainings_step`, src/bigan_classify.py:126-155 (numbering of
        SURVEY.md 3.2).  Exposed separately so the parity tests can compare every update
        against the oracle from identical weights."""
        B = x16.shape[0]
        z, r = self.z32[:B], self.r32[:B]          # latents stay fp32 (hi/lo in the GEMMs)
        G, E, D = self.G, self.E, self.D
        n_total = B * self.dist.world_size
        L = self.loss_buf
        if self.gen_cells is None:
            self.gen_cells = ops.alloc2d(self.max_batch, self.Gn, device=self.device)
        cells = self.gen_cells[:B]
        if k == 1:
            # _train_gen_w_discr.train_on_batch((encodings, noise), y_ones)          :145
            gen = G.forward({"z": z, "r": r}, B, bn_train=True, **self._drop_args(1, "G", masks))
            logit = D.forward({"z": z, "cell": gen}, B, bn_train=False, pre_activation=True,
                              **self._drop_args(1, "D", masks))
            dz1 = D.output_grad(B)
            ops.bce_fwd_bwd(logit, REAL_LABEL, n_total, L[0:1], dz1)
            dcell = D.backward(dz1, train=False, want=("cell",))["cell"]
            G.backward(dcell, train=True)
            G.apply_rmsprop()
        elif k == 2:
            # _train_gen_w_enc.train_on_batch((cell_data, noise), cell_data)         :146
            enc = E.forward({"cell": x16}, B, bn_train=False, **self._drop_args(2, "E", masks))
            gen = G.forward({"z": enc, "r": r}, B, bn_train=True, **self._drop_args(2, "G", masks))
            dgen = G.output_grad(B)
            ops.mse_fwd_bwd(gen, n_total, L[1:2], target=x16, dpred=dgen, **self._reduce_args())
            G.backward(dgen, train=True)
            G.apply_rmsprop()
        elif k == 3:
            # _train_enc_w_discr.train_on_batch(cell_data, y_zeros)                  :150
            enc = E.forward({"cell": x16}, B, bn_train=True, **self._drop_args(3, "E", masks))
            logit = D.forward({"z": enc, "cell": x16}, B, bn_train=False, pre_activation=True,
                              **self._drop_args(3, "D", masks))
            dz1 = D.output_grad(B)
            ops.bce_fwd_bwd(logit, 0.0, n_total, L[2:3], dz1)
            dzin = D.backward(dz1, train=False, want=("z",))["z"]
            E.backward(dzin, train=True)
            E.apply_rmsprop()
        elif k == 4:
            # _train_enc_w_gen.train_on_batch((encodings, noise), encodings)         :151
            gen = G.forward({"z": z, "r": r}, B, bn_train=False, **self._drop_args(4, "G", masks))
            enc = E.forward({"cell": gen}, B, bn_train=True, **self._drop_args(4, "E", masks))
            denc = E.output_grad(B)
            ops.mse_fwd_bwd(enc, n_total, L[3:4], target=self.z32[:B], dpred=denc,
                            **self._reduce_args())
            E.backward(denc, train=True)
            E.apply_rmsprop()
        elif k == 5:
            # generated_cells = generate_cells(encodings, noise)                    :136
            gen = G.forward({"z": z, "r": r}, B, bn_train=False, dropout="off")
            ops.round_half_even(gen, out16=cells)
        elif k == 6:
            # _discriminator.train_on_batch((encodings, generated_cells), y_zeros)   :137
            self.train_discriminator(z, cells, 0.0, 4, self._drop_args(6, "D", masks))
        elif k == 7:
            # generated_encodings = trainings_encoding_prediction(batch)            :138
            self.encode(x16, out32=self.gen_enc32[:B])
            if self.variant == "classify":
                ops.argmax_onehot(self.gen_enc32[:B], out32=self.gen_enc32[:B])
        elif k == 8:
            # _discriminator.train_on_batch((generated_encodings, batch), y_ones)    :139
            self.train_discriminator(self.gen_enc32[:B], x16, REAL_LABEL, 5,
                                     self._drop_args(8, "D", masks))
        else:
            raise ValueError(f"no sub-step {k}")

    def train_discriminator(self, z, cells, label, loss_slot, drop_args):
        """One `_discriminator.train_on_batch((z, cells), label * ones)`: BCE on D's sigmoid
        output against a constant label vector, backward, RMSprop on D
        (src/bigan_classify.py:112-115,154-155).  z: [B, Z] fp32, cells: [B, genes] bf16."""
        B = cells.shape[0]
        D = self.D
        logit = D.forward({"z": z, "cell": cells}, B, bn_train=True, pre_activation=True,
                          **drop_args)
        dz1 = D.output_grad(B)
        ops.bce_fwd_bwd(logit, float(label), B * self.dist.world_size,
                        self.loss_buf[loss_slot:loss_slot + 1], dz1)
        D.backward(dz1, train=True)
        D.apply_rmsprop()

    def snapshot_state(self):
        """Device copies of everything a training step mutates (weights, bf16 copies, RMSprop
        slots, BN moving statistics, RNG counter)."""
        self.join()
        snap = {"rng": self.rng_counter.clone()}
        for k, n in self.nets.items():
            snap[k] = {"p32": n.p32.clone(), "p16": n.p16.clone(), "ms": n.ms.clone(),
                       "mom": n.mom.clone(), "state_blocked": n.state_blocked,
                       "p16lo": None if n.p16lo is None else n.p16lo.clone(),
                       "bn": [(L["moving_mean"].clone(), L["moving_var"].clone())
                              for L in n.layers if L["kind"] == "bn"]}
        return snap

    def restore_state(self, snap):
        self.join()
        self.rng_counter.copy_(snap["rng"])
        for k, n in self.nets.items():
            s = snap[k]
            n.p32.copy_(s["p32"])
            n.p16.copy_(s["p16"])
            n.ms.copy_(s["ms"])
            n.mom.copy_(s["mom"])
            n.state_blocked = s["state_blocked"]       # raw copies: the layout they were taken in
            if n.p16lo is not None:
                n.p16lo.copy_(s["p16lo"])
            for L, (mm, mv) in zip([L for L in n.layers if L["kind"] == "bn"], s["bn"]):
                L["moving_mean"].copy_(mm)
                L["moving_var"].copy_(mv)

    # ------------------------------------------------------------------ checkpoint / resume
    def state_dict(self):
        """Everything a resumed run needs, as host numpy arrays in Keras layout: per network the
        weights in creation order (Dense kernel[in,out], bias; BatchNormalization gamma, beta,
        moving_mean, moving_variance), the RMSprop slots (rms, momentum) of every trainable
        tensor, plus the dropout / prior RNG stream position.  The reference has no
        checkpointing at all (SURVEY.md 5); the layout is the one `Model.get_weights()` and
        `optimizer.get_weights()` would give, so a Keras-side tool can consume it."""
        self.join()
        out = {"meta/variant": self.variant, "meta/encoding_size": self.Z,
               "meta/gene_size": self.Gn, "meta/rng_seed": self.rng_seed,
               "meta/rng_counter": int(self.rng_counter.item())}
        for name, net in self.nets.items():
            for i, w in enumerate(net.get_weights()):
                out[f"{name}/w{i}"] = w
            for i, (ms, mom) in enumerate(net.get_slots()):
                out[f"{name}/rms{i}"] = ms
                out[f"{name}/mom{i}"] = mom
        return out

    def load_state_dict(self, state):
        for key, want in (("meta/variant", self.variant), ("meta/encoding_size", self.Z),
                          ("meta/gene_size", self.Gn)):
            got = state[key]
            got = got.item() if hasattr(got, "item") else got
            if str(got) != str(want):
                raise ValueError(f"checkpoint {key} = {got}, this model has {want}")
        for name, net in self.nets.items():
            n_w = len([k for k in state if k.startswith(f"{name}/w")])
            net.set_weights([state[f"{name}/w{i}"] for i in range(n_w)])   # zeroes the slots
            n_s = len([k for k in state if k.startswith(f"{name}/rms")])
            net.set_slots([(state[f"{name}/rms{i}"], state[f"{name}/mom{i}"]) for i in range(n_s)])
        self.rng_seed = int(state["meta/rng_seed"])
        self.rng_counter.fill_(int(state["meta/rng_counter"]))
        self._graphs.clear()          # captured steps baked the old RNG seed in

    def write_checkpoint(self, path, state):
        """rank 0 writes `state` (a state_dict(), possibly with extra meta entries) atomically."""
        import numpy as np
        if self.dist.rank == 0:
            tmp = path + ".tmp.npz"
            np.savez(tmp, **state)
            os.replace(tmp, path)

    def save_checkpoint(self, path):
        """One .npz file (written atomically).  Data-parallel runs: call on every rank (the
        sharded fp32 master weights and RMSprop slots are gathered collectively); rank 0 writes."""
        self.write_checkpoint(path, self.state_dict())

    def load_checkpoint(self, path):
        """-> the loaded state (callers read their own `meta/*` entries from it)."""
        import numpy as np
        with np.load(path, allow_pickle=False) as f:
            state = {k: f[k] for k in f.files}
        self.load_state_dict(state)
        return state

    def join(self):
        """Order the current stream after every pending side-stream optimiser update (call
        before timing / reading weights; does not block the host)."""
        for n in self.nets.values():
            n._wait_optimizer()

    def finish_step(self, masks=None):
        L = self.loss_buf
        if masks is None:
            ops.counter_add(self.rng_counter, 1)
        self.dist.all_reduce(L)
        Lc = L.clone()
        g = LossScalar(Lc[0] + Lc[1])
        e = LossScalar(Lc[2] + Lc[3])
        d = LossScalar((Lc[4] + Lc[5]) * 0.5)       # np.mean([d_loss_1, d_loss_2])    :140
        self.last_losses = Lc
        return g, e, d

    def peer_graphable(self):
        """Data-parallel step without any NCCL call inside (gradient exchange, optimiser and the
        small all-reduces all run as peer-memory kernels with device-resident epochs), so
        capture_step() may record it.  CELLCOMM_B200_DP_GRAPH=0 keeps data parallel eager."""
        if self.dist.world_size == 1:
            return True
        if os.environ.get("CELLCOMM_B200_DP_GRAPH", "1") == "0":
            return False
        probe = getattr(self.dist, "_peer_allreduce_state", None)
        return (all(n.peer is not None for n in self.nets.values()) and probe is not None
                and probe(self.device) is not None)

    # ------------------------------------------------------------------ CUDA graph of a step
    def capture_step(self, csr, n_cols, batch, latents="device"):
        """Capture gather -> (priors) -> trainings_step for a fixed batch size into ONE CUDA
        graph (~850 kernel launches become one graph launch; at the reference's batch of 128 the
        eager step is bound by host launch overhead, not by the GPU).

        csr = (rowptr, colidx, values) on the device.  latents = "device": tf.random.uniform
        priors are drawn inside the graph from the Philox streams; "host": the caller writes
        self.z32 / self.r32 before every replay.  Returns GraphedStep; .idx is the static row
        index buffer to fill before .replay()."""
        if self.device.type != "cuda":
            raise RuntimeError("CUDA graphs need a CUDA device")
        if self.dist.world_size > 1 and not self.peer_graphable():
            raise RuntimeError("graph capture needs the peer-memory data-parallel path (NCCL "
                               "collectives are not captured)")
        self.reserve(batch)
        key = (int(batch), latents, csr[0].data_ptr(), csr[1].data_ptr(), csr[2].data_ptr())
        gs = self._graphs.get(key)
        if gs is None:
            gs = GraphedStep(self, csr, n_cols, batch, latents)
            self._graphs[key] = gs
        return gs

    # ------------------------------------------------------------------ inference
    PREDICT_TILE = 4096       # rows per tile of every pass over cells (see _generated_tiles)

    def _tiling(self, name, tile_rows, cuda=True):
        """Rows per tile of the pass `name`: tile_rows, or PREDICT_TILE when None."""
        if cuda and self.device.type != "cuda":
            raise RuntimeError(f"{name} needs a CUDA device (no host fallback)")
        tile_rows = self.PREDICT_TILE if tile_rows is None else int(tile_rows)
        if tile_rows < 1:
            raise ValueError(f"{name}: tile_rows must be >= 1")
        return tile_rows

    def _latents(self, name, z32, r32, n=None):
        """z32 / r32 ([n, Z] fp32, host or device; n = z32's rows when None) on the device."""
        z32 = torch.as_tensor(z32, dtype=torch.float32).to(self.device)
        r32 = torch.as_tensor(r32, dtype=torch.float32).to(self.device)
        n = z32.shape[0] if n is None else n
        if tuple(z32.shape) != (n, self.Z) or tuple(r32.shape) != (n, self.Z):
            raise ValueError(f"{name}: z32 / r32 must both be [{n}, {self.Z}]")
        return z32, r32

    def _cells(self, name, csr, order, z32, r32, n=None):
        """The cells of a pass over real or generated ones: the rows `order` (host or device
        int64) of the device CSR `csr`, or the generator's output for z32 / r32.  Exactly one
        of the two must be given, with n cells when n is given -> (n, order, z32, r32), the
        given pair on the device and the other None."""
        if (csr is None) == (z32 is None):
            raise ValueError(f"{name}: give either csr and order (real cells) or z32 and r32 "
                             "(generated cells)")
        if csr is None:
            z32, r32 = self._latents(name, z32, r32, n)
            return z32.shape[0], None, z32, r32
        order = torch.as_tensor(order, dtype=torch.int64).to(self.device)
        if order.dim() != 1 or n not in (None, order.numel()):
            raise ValueError(f"{name}: order must be a vector of row numbers"
                             + ("" if n is None else f", {n} of them"))
        return order.numel(), order, None, None

    def _generated_tiles(self, z32, r32, tile_rows, out):
        """Generated cells tile by tile: for rows [s, s + m) of z32 / r32 ([n, Z] fp32 on the
        device), from row 0 in tiles of tile_rows rows, set_latents + generate() into
        x = out[s:s + m] when out ([n, gene_size] fp32) holds every row, else into x = out[:m]
        of one fp32 tile buffer; yields (s, m, x).

        This is G.predict's tiling, and the only one that reproduces generate_cells bit for
        bit: the generator's GEMMs choose their split-K from the row count.  Every pass over
        generated cells takes its tiles from here."""
        n = z32.shape[0]
        for s in range(0, n, tile_rows):
            m = min(tile_rows, n - s)
            x = out[s:s + m] if out.shape[0] == n else out[:m]
            self.set_latents(z32[s:s + m], r32[s:s + m], m)
            self.generate(m, out32=x)
            yield s, m, x

    def _real_tiles(self, csr, rows, tile):
        """Real cells tile by tile: for cells [s, s + m) of `rows` of the device CSR
        csr = (rowptr, colidx, values) with gene_size columns, in tiles of tile's rows,
        cc_gather_rows into x = tile[:m] (bf16 or fp32); yields (s, m, x).  rows: a row range
        (row_begin, row_end), gathered by row_start / n_rows, or an int64 device vector of row
        numbers, gathered by row_idx."""
        T, key = tile.shape[0], "out16" if tile.dtype == ops.COMPUTE_DTYPE else "out32"
        ranged = isinstance(rows, tuple)
        n = rows[1] - rows[0] if ranged else rows.numel()
        for s in range(0, n, T):
            m = min(T, n - s)
            x = tile[:m]
            if ranged:
                ops.gather_rows(*csr, self.Gn, row_start=rows[0] + s, n_rows=m, **{key: x})
            else:
                ops.gather_rows(*csr, self.Gn, row_idx=rows[s:s + m], **{key: x})
            yield s, m, x

    def encode(self, x16, out32=None):
        """E.predict on a [rows, gene_size] bf16 tile; fp32 result in out32 when given."""
        return self.E.forward({"cell": x16}, x16.shape[0], bn_train=False, dropout="off",
                              out32=out32)

    def encode_plan(self, tile_rows=None):
        """cc_encode_plan for this engine's encoder: the op list Net.forward(bn_train=False,
        dropout="off") would launch for one tile (same kernels, same precision policy), over
        scratch slots.  None when a layer has width 0 (the 5-gene fixture's Dense(0))."""
        from . import _lib
        tile_rows = int(tile_rows or self.PREDICT_TILE)
        cached = getattr(self, "_enc_plan", None)
        if cached is not None and cached[0] == tile_rows:
            return cached[1]
        net, g = self.E, self.E.g
        if any(w == 0 for w in g.widths):
            return None
        plan = _lib.EncodePlan()
        slots = []                      # (width, fp32)

        def new_slot(width, fp32):
            slots.append((int(width), int(bool(fp32))))
            return len(slots) - 1

        cell = g.inputs["cell"]
        val = {cell: new_slot(g.widths[cell], False)}      # tensor id -> slot
        operands = {}                                       # tensor id -> [bf16 slots]
        ops_ = []

        def emit(**kw):
            op = plan.ops[len(ops_)]
            for k, v in kw.items():
                setattr(op, k, v)
            ops_.append(op)
            return op

        def gemm_operands(t):
            if t not in operands:
                s_ = val[t]
                if not slots[s_][1]:
                    operands[t] = [s_]
                elif t in net.split:
                    hi, lo = new_slot(g.widths[t], False), new_slot(g.widths[t], False)
                    op = emit(kind=_lib.ENC_SPLIT, n_in=1, out=hi, out2=lo)
                    op.in_[0] = s_
                    operands[t] = [hi, lo]
                else:
                    sh = new_slot(g.widths[t], False)
                    op = emit(kind=_lib.ENC_COPY, n_in=1, out=sh)
                    op.in_[0] = s_
                    operands[t] = [sh]
            return operands[t]

        last = g.nodes[-1]
        for node in g.nodes:
            kind, out = node["kind"], node["out"]
            if kind == "dense":
                L = net.layers[node["layer"]]
                if "w16lo" in L:
                    return None                          # hi + lo kernels: not expressible
                segs, ro = [], 0
                for i in node["ins"]:
                    for term in gemm_operands(i):
                        segs.append((term, ro))
                    ro += g.widths[i]
                if len(segs) > 4:
                    return None
                is_last = node is last
                fp32 = out in net.hp
                dst = -1 if (is_last and fp32) else new_slot(g.widths[out], fp32)
                op = emit(kind=_lib.ENC_DENSE, n_in=len(segs), out=dst, width=L["N"],
                          act=_ACT[node["act"]], w16=L["w16"].data_ptr(), ldw=L["ld"],
                          bias=L["b32"].data_ptr())
                for j, (sl, r_) in enumerate(segs):
                    op.in_[j], op.w_row[j] = sl, r_
                if is_last and not fp32:
                    op2 = emit(kind=_lib.ENC_COPY, n_in=1, out=-1)
                    op2.in_[0] = dst
                val[out] = dst
            elif kind == "bn":
                L = net.layers[node["layer"]]
                dst = new_slot(g.widths[out], out in net.hp)
                op = emit(kind=_lib.ENC_BN_INFER, n_in=1, out=dst, gamma=L["gamma"].data_ptr(),
                          beta=L["beta"].data_ptr(), mean=L["moving_mean"].data_ptr(),
                          var=L["moving_var"].data_ptr(), eps=BN_EPS)
                op.in_[0] = val[node["ins"][0]]
                val[out] = dst
            elif kind == "dropout":
                val[out] = val[node["ins"][0]]           # predict: Dropout is the identity
            elif kind == "softmax":
                dst = new_slot(g.widths[out], out in net.hp)
                op = emit(kind=_lib.ENC_SOFTMAX, n_in=1, out=dst)
                op.in_[0] = val[node["ins"][0]]
                val[out] = dst
            else:                                        # the encoders have no Concatenate node
                return None
            if len(ops_) > _lib.ENC_MAX_OPS - 2 or len(slots) > _lib.ENC_MAX_SLOTS - 3:
                return None
        plan.n_cols, plan.tile_rows = self.Gn, tile_rows
        plan.n_slots, plan.n_ops = len(slots), len(ops_)
        for i, (w, f) in enumerate(slots):
            plan.slot_width[i], plan.slot_fp32[i] = w, f
        nbytes = ops.encode_scratch_bytes(plan)
        scratch = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        ws = ops.workspace(self.device)
        plan.scratch, plan.scratch_bytes = scratch.data_ptr(), nbytes
        plan.workspace, plan.workspace_elems = ws.data_ptr(), ws.numel()
        self._enc_plan = (tile_rows, plan, scratch)
        return plan

    def encode_stream(self, rowptr, colidx, values, row_begin, row_end, out32, tile_rows=None):
        """encoding_prediction for rows [row_begin, row_end) of a device CSR in ONE C call
        (cc_encode_stream): gather + encoder forward per tile, no Python between tiles.  Falls
        back to the tile loop over encode() off CUDA and for encoders the plan cannot express."""
        self.E._wait_optimizer()
        tile_rows = self._tiling("encode_stream", tile_rows, cuda=False)
        plan = self.encode_plan(tile_rows) if self.device.type == "cuda" else None
        if plan is not None:
            ops.encode_stream(rowptr, colidx, values, row_begin, row_end, plan, out32)
            return
        tile = ops.alloc2d(min(tile_rows, max(1, row_end - row_begin)), self.Gn,
                           device=self.device)
        for s, m, x in self._real_tiles((rowptr, colidx, values), (row_begin, row_end), tile):
            self.encode(x, out32=out32[s:s + m])

    def generate(self, rows, out32=None):
        """G.predict on the staged latents (first `rows`)."""
        return self.G.forward({"z": self.z32[:rows], "r": self.r32[:rows]}, rows, bn_train=False,
                              dropout="off", out32=out32)

    def generate_csr(self, z32, r32, tile_rows=None, consume=None):
        """rint(G.predict(z, r)) for every row of z32 / r32 ([n, Z] fp32, host or device) as a
        CSR, without ever holding the dense (n, genes) output.  Per generated tile
        (_generated_tiles, into one fp32 tile): cc_round_csr_count, a read-back of the tile's
        nnz, cc_round_csr_fill, and cudaMemcpyAsync of the entries into pinned host staging on
        a side stream, so that the copy of tile i overlaps the forward of tile i+1 (two staging
        sets, events).
        Device memory: the fp32 tile plus the largest tile's entries.

        Engine state (weights, BN statistics, RNG counter, loss_buf) is not touched; like
        generate(), the pass orders itself after pending side-stream optimiser updates, and it
        issues no collective.

        consume(row0, rowptr, colidx, values) receives each finished tile (rowptr: the tile's
        m + 1 offsets from 0, numpy; colidx / values: pinned torch views valid until the call
        returns).  consume=None: accumulate and return the host CSR
        (rowptr int64 [n + 1], colidx int32 [nnz], values float32 [nnz]) as numpy arrays."""
        import numpy as np
        dev = self.device
        tile_rows = self._tiling("generate_csr", tile_rows)
        z32, r32 = self._latents("generate_csr", z32, r32)
        n = z32.shape[0]
        parts = None
        if consume is None:
            rowptr_out = np.zeros(n + 1, dtype=np.int64)
            parts = []

            def consume(row0, rp, col, val):
                rowptr_out[row0 + 1:row0 + len(rp)] = rowptr_out[row0] + rp[1:]
                # pageable copies out of the staging (torch copies on host threads)
                parts.append((torch.empty_like(col, pin_memory=False).copy_(col),
                              torch.empty_like(val, pin_memory=False).copy_(val)))

        T = max(1, min(tile_rows, n))
        main = torch.cuda.current_stream(dev)
        side = getattr(self, "_gen_side", None)
        if side is None:
            side = self._gen_side = torch.cuda.Stream(device=dev)
        tile = ops.alloc2d(T, self.Gn, dtype=torch.float32, device=dev, zero=False)
        rowptr_d = torch.zeros(T + 1, dtype=torch.int64, device=dev)   # [0] stays 0: tile-local
        rowptr_h = torch.empty(T + 1, dtype=torch.int64, pin_memory=True)
        ent_d = None                   # (colidx, values) on the device, the largest tile's size
        stage = [None, None]           # pinned (colidx, values), alternating between tiles
        copied = [None, None]
        pending = None

        def finish(p):
            slot, row0, rp, nnz = p
            copied[slot].synchronize()
            consume(row0, rp, stage[slot][0][:nnz], stage[slot][1][:nnz])

        for i, (s, m, x) in enumerate(self._generated_tiles(z32, r32, T, tile)):
            slot = i % 2
            ops.round_csr_count(x, rowptr_d[:m + 1])
            rowptr_h[:m + 1].copy_(rowptr_d[:m + 1], non_blocking=True)
            counted = torch.cuda.Event()
            counted.record(main)
            if pending is not None:      # the host takes tile i-1 while the GPU runs tile i
                finish(pending)
                main.wait_event(copied[pending[0]])   # its entries buffer is free again
            counted.synchronize()
            rp = rowptr_h[:m + 1].numpy().copy()
            nnz = int(rp[m])
            if ent_d is None or ent_d[0].numel() < nnz:
                ent_d = None
                cap = max(nnz, 1)
                ent_d = (torch.empty(cap, dtype=torch.int32, device=dev),
                         torch.empty(cap, dtype=torch.float32, device=dev))
            ops.round_csr_fill(x, rowptr_d[:m + 1], ent_d[0][:nnz], ent_d[1][:nnz])
            filled = torch.cuda.Event()
            filled.record(main)
            if stage[slot] is None or stage[slot][0].numel() < nnz:
                cap = max(nnz, 1)
                stage[slot] = (torch.empty(cap, dtype=torch.int32, pin_memory=True),
                               torch.empty(cap, dtype=torch.float32, pin_memory=True))
            side.wait_event(filled)
            with torch.cuda.stream(side):
                stage[slot][0][:nnz].copy_(ent_d[0][:nnz], non_blocking=True)
                stage[slot][1][:nnz].copy_(ent_d[1][:nnz], non_blocking=True)
                copied[slot] = torch.cuda.Event()
                copied[slot].record(side)
            pending = (slot, s, rp, nnz)
        if pending is not None:
            finish(pending)
            main.wait_event(copied[pending[0]])
        if parts is None:
            return None
        if parts:
            colidx = torch.cat([c for c, _ in parts]).numpy()
            values = torch.cat([v for _, v in parts]).numpy()
        else:
            colidx, values = np.zeros(0, np.int32), np.zeros(0, np.float32)
        return rowptr_out, colidx, values

    def score_stream(self, rowptr, colidx, values, row_begin, row_end, r32, enc_out, mse_out,
                     d_out, tile_rows=None):
        """Per-cell scores of rows [row_begin, row_end) of a device CSR with gene_size columns:
            enc_out[i] = E.predict(x)                      ([n, Z] fp32, device)
            mse_out[i] = mean_c (G.predict(z, r) - x)^2    ([n] fp32, device; G's fp32 output
                                                            against the exact fp32 counts)
            d_out[i]   = D.predict(z, x)                   ([n] or [n, 1] fp32, device)
        with z = enc_out[i] and r = r32[i] ([n, Z] fp32, host or device).  Per tile of
        `tile_rows` rows from row_begin (the tiling of E / G / D.predict, so the bits match;
        see _generated_tiles): encode_stream into z, set_latents(z, r) + generate() into one
        fp32 tile, cc_recon_sqerr with scale 1 / gene_size, cc_gather_rows into one bf16 cell
        tile (_real_tiles), and discriminate(z, x).  Device memory: those two tiles and the
        nets' activations for tile_rows rows; nothing of size (n, genes).

        Engine state (weights, BN statistics, RNG counter, loss_buf) is not touched; every
        forward orders itself after pending side-stream optimiser updates of its net, and the
        pass issues no collective."""
        dev = self.device
        tile_rows = self._tiling("score_stream", tile_rows)
        row_begin, row_end = int(row_begin), int(row_end)
        n = row_end - row_begin
        if row_begin < 0 or n < 0 or row_end > rowptr.shape[0] - 1:
            raise ValueError(f"score_stream: rows [{row_begin}, {row_end}) outside the CSR's "
                             f"{rowptr.shape[0] - 1} rows")
        r32 = torch.as_tensor(r32, dtype=torch.float32).to(dev)
        if tuple(r32.shape) != (n, self.Z) or tuple(enc_out.shape) != (n, self.Z):
            raise ValueError(f"score_stream: r32 and enc_out must be [{n}, {self.Z}]")
        if mse_out.numel() != n or d_out.numel() != n:
            raise ValueError(f"score_stream: mse_out and d_out must hold {n} values")
        if n == 0:
            return
        T = min(tile_rows, n)
        pred = ops.alloc2d(T, self.Gn, dtype=torch.float32, device=dev, zero=False)
        cells = self._real_tiles((rowptr, colidx, values), (row_begin, row_end),
                                 ops.alloc2d(T, self.Gn, device=dev))   # zero padding
        mse, d = mse_out.view(n), d_out.view(n, 1)
        for s in range(0, n, T):
            m, row = min(T, n - s), row_begin + s
            z = enc_out[s:s + m]
            self.encode_stream(rowptr, colidx, values, row, row + m, z)
            self.set_latents(z, r32[s:s + m], m)
            self.generate(m, out32=pred[:m])
            ops.recon_sqerr(pred[:m], rowptr, colidx, values, row, mse[s:s + m],
                            scale=1.0 / self.Gn)
            _, _, x = next(cells)           # the gather of these rows, after the generator
            self.discriminate(z, x, d[s:s + m])

    def moments_stream(self, bounds, *, csr=None, order=None, z32=None, r32=None,
                       tile_rows=None):
        """Per-group column moments of real or generated cells, for K groups given by `bounds`
        (K + 1 non-decreasing host ints from 0) -> device tensors
            sum     [K, gene_size] fp64   sum over the group's cells of v
            sumsq   [K, gene_size] fp64   sum of v^2
            nonzero [K, gene_size] int64  number of cells with v != 0
        Real cells: csr = (rowptr, colidx, values) of a device CSR with gene_size columns and
        `order` (host or device int64) its row numbers sorted by group; group k is the rows
        order[bounds[k]:bounds[k + 1]] and v the exact fp32 count.  Per tile of at most
        tile_rows positions of one group (_real_tiles into the fp32 tile): cc_col_moments into
        that group's accumulators.
        Generated cells: z32 / r32 ([n, Z] fp32, host or device, n = bounds[-1]) sorted by
        group; group k is rows [bounds[k], bounds[k + 1]) and v = rint(G.predict(z, r)).  Per
        generated tile (_generated_tiles into the fp32 tile, so the cells are generate_cells'
        bit for bit): one cc_col_moments(round_half_even=1) per group segment inside the tile.
        Device memory: the fp32 tile, the accumulators and the cc_col_moments workspace;
        nothing of size (n, genes).  Engine state (weights, BN statistics, RNG counter,
        loss_buf) is not touched; the generator forward orders itself after pending side-stream
        optimiser updates, and the pass issues no collective."""
        dev = self.device
        tile_rows = self._tiling("moments_stream", tile_rows)
        bounds = [int(b) for b in bounds]
        K = len(bounds) - 1
        if K < 1 or bounds[0] != 0 or any(b > e for b, e in zip(bounds, bounds[1:])):
            raise ValueError("moments_stream: bounds must be K + 1 >= 2 non-decreasing "
                             "offsets from 0")
        n, order, z32, r32 = self._cells("moments_stream", csr, order, z32, r32, bounds[-1])
        Gn = self.Gn
        sums = torch.zeros((K, Gn), dtype=torch.float64, device=dev)
        sumsq = torch.zeros((K, Gn), dtype=torch.float64, device=dev)
        nonzero = torch.zeros((K, Gn), dtype=torch.int64, device=dev)
        if n == 0:
            return sums, sumsq, nonzero
        T = min(tile_rows, n if csr is None else max(e - b for b, e in zip(bounds, bounds[1:])))
        tile = ops.alloc2d(T, Gn, dtype=torch.float32, device=dev, zero=False)
        ws_bytes = ops.col_moments_ws_bytes(T, Gn)
        ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        if csr is not None:
            for k in range(K):
                for _, _, x in self._real_tiles(csr, order[bounds[k]:bounds[k + 1]], tile):
                    ops.col_moments(x, sums[k], sumsq[k], nonzero[k], ws=ws)
            return sums, sumsq, nonzero
        for s, m, x in self._generated_tiles(z32, r32, tile_rows, tile):
            for k in range(K):
                lo, hi = max(bounds[k], s), min(bounds[k + 1], s + m)
                if lo < hi:
                    ops.col_moments(x[lo - s:hi - s], sums[k], sumsq[k], nonzero[k],
                                    round=True, ws=ws)
        return sums, sumsq, nonzero

    def features_stream(self, *, csr=None, order=None, z32=None, r32=None, tile_rows=None):
        """log1p features of real or generated cells -> device tensors
            features       [n, gene_size] bf16  view of a [n, pad_ld(gene_size)] buffer whose
                                                padding columns are zero (a GEMM operand)
            library_size   [n] fp64             sum over genes of v
            genes_detected [n] int32            #{genes : v != 0}
        with features = bf16(float(log1p(double(v)))) (cc_log1p_features).  The two modes of
        moments_stream: real cells are the rows `order` (host or device int64) of the device CSR
        `csr` (_real_tiles), v the exact fp32 count; generated cells are the rows of z32 / r32
        ([n, Z] fp32), v = rint(G.predict(z, r)) (_generated_tiles, so they are generate_cells'
        cells bit for bit).  Device memory: one fp32 tile and the outputs.  Engine state is not
        touched and no collective is issued."""
        dev = self.device
        tile_rows = self._tiling("features_stream", tile_rows)
        n, order, z32, r32 = self._cells("features_stream", csr, order, z32, r32)
        feats = ops.alloc2d(n, self.Gn, dtype=torch.bfloat16, device=dev, zero=False)
        lib = torch.zeros(n, dtype=torch.float64, device=dev)
        det = torch.zeros(n, dtype=torch.int32, device=dev)
        if n == 0:
            return feats, lib, det
        tile = ops.alloc2d(min(tile_rows, n), self.Gn, dtype=torch.float32, device=dev,
                           zero=False)
        tiles = (self._real_tiles(csr, order, tile) if csr is not None
                 else self._generated_tiles(z32, r32, tile_rows, tile))
        for s, m, x in tiles:
            ops.log1p_features(x, feats[s:s + m], lib[s:s + m], det[s:s + m], round=csr is None)
        return feats, lib, det

    MEDIAN_ROWS = 1024        # rows of d^2 formed at a time for the median

    def mmd_sums(self, fx, fy, scales, masks):
        """Kernel sums of an MMD permutation test on two device feature blocks fx, fy ([n, K]
        bf16, rows of features_stream) -> (median, sums):
            median  the lower median of d2_ij = max((G_ii + G_jj) - 2 G_ij, 0), i < j, over the
                    pooled cells (fx rows first), G their fp32 Gram matrix
            sums    host fp64 [L, len(scales), 3]: XX, YY, XY of k = exp(-d2 / (s * median)) per
                    labelling (cc_mmd_sums; XX, YY, XY as in mmd_from_sums)
        masks: uint32 [L, ceil(2n / 32)] (host), bit i = pooled cell i is in X.  The Gram
        matrix is three cc_gemm calls (XX, XY and YY quadrants; the YX quadrant is never read),
        the median a torch kthvalue over the upper triangle formed with the kernel's fp32
        expression.  Device memory: the [2n, 2n] fp32 Gram matrix, the upper triangle of d2 and
        the workspace; nothing of size (n, genes) in fp32.  Rank-local, no collective.
        A zero median (most pairs identical) gives median 0 and NaN sums."""
        import numpy as np
        dev = self.device
        n, K = fx.shape
        if tuple(fy.shape) != (n, K):
            raise ValueError("mmd_sums: fx and fy must have the same shape")
        N = 2 * n
        masks = np.ascontiguousarray(masks, dtype=np.uint32)
        L = masks.shape[0]
        if masks.ndim != 2 or masks.shape[1] != (N + 31) // 32:
            raise ValueError(f"mmd_sums: masks must be [L, {(N + 31) // 32}]")
        if not 1 <= len(scales) <= 4:
            raise ValueError("mmd_sums: 1 to 4 bandwidth scales")
        if n < 1:
            raise ValueError("mmd_sums: needs at least one cell per block")
        G = ops.alloc2d(N, N, dtype=torch.float32, device=dev, zero=False)
        ops.gemm(n, n, [fx], [fx], [K], 0, 0, out32=G[:n, :n])
        ops.gemm(n, n, [fx], [fy], [K], 0, 0, out32=G[:n, n:])
        ops.gemm(n, n, [fy], [fy], [K], 0, 0, out32=G[n:, n:])
        diag = torch.diagonal(G).clone()
        upper = []
        cols = torch.arange(N, device=dev)
        for s in range(0, N - 1, self.MEDIAN_ROWS):
            e = min(N - 1, s + self.MEDIAN_ROWS)
            d2 = torch.clamp_min((diag[s:e, None] + diag[None, :]) - 2.0 * G[s:e], 0.0)
            upper.append(d2[cols[None, :] > torch.arange(s, e, device=dev)[:, None]])
            del d2
        upper = torch.cat(upper)
        m = upper.numel()
        median = float(torch.kthvalue(upper, (m - 1) // 2 + 1).values) if m else float("nan")
        del upper
        out = np.full((L, len(scales), 3), np.nan)
        if not median > 0:
            return median, out
        inv = [1.0 / (float(s) * median) for s in scales]
        sums = torch.empty((L, len(scales), 3), dtype=torch.float64, device=dev)
        ws = torch.empty(ops.mmd_sums_ws_bytes(N, len(scales), L), dtype=torch.uint8, device=dev)
        ops.mmd_sums(G, inv, torch.from_numpy(masks.view(np.int32)).to(dev), sums, ws=ws)
        return median, sums.cpu().numpy()

    def discriminate(self, z16, x16, out32):
        """D.predict -> probabilities (fp32 [rows,1])."""
        return self.D.forward({"z": z16, "cell": x16}, x16.shape[0], bn_train=False, dropout="off",
                              out32=out32)
