// Data-parallel optimiser step over NVLink peer memory (one process per GPU, one node):
// ONE kernel per gradient bucket does what "NCCL reduce-scatter -> RMSprop on the shard ->
// NCCL all-gather of the bf16 weights" does in three, with no staging buffers and no NCCL
// CTAs competing with the GEMMs for SMs:
//
//   for every element i of this rank's shard of the bucket:
//       g      = sum_q  grad_q[i]              (P2P loads from every rank's gradient buffer,
//                                               fixed rank order -> bit-identical everywhere)
//       ms,mom,w = Keras RMSprop(momentum)     (local fp32 master + slots)
//       p16_q[i] = bf16(w)  for every rank q   (P2P stores: the all-gather)
//
// Replaces the gradient exchange that `optimizer.apply_gradients` would need under data
// parallelism; the reference itself is single-process (src/bigan_classify.py:88,144-155).
// Hand-shake: each rank publishes "bucket b of update e is complete" / "... is consumed and
// my shard is written" by storing the epoch into every peer's flag array (st.release.sys
// after a system fence); consumers poll their LOCAL flags with ld.acquire.sys.
#include "common.cuh"

namespace cc {

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// spin until *flag >= value (epochs only grow); a lost peer must trap, not hang the box
__device__ __forceinline__ void wait_flag(const uint32_t* flag, uint32_t value, int tag) {
  long long t0 = 0;
  uint32_t spins = 0;
  while ((int32_t)(ld_acquire_sys(flag) - value) < 0) {
    if (++spins == 1024u) t0 = clock64();
    if (spins > 1024u && (spins & 255u) == 0) {
      __nanosleep(200);
      if (clock64() - t0 > 20000000000LL) {   // ~10 s
        printf("cc_peer: flag timeout tag=%d block=%d want=%u have=%u\n", tag, blockIdx.x, value,
               ld_acquire_sys(flag));
        __trap();
      }
    }
  }
}

struct PeerPtrs {
  const float* g[CC_PEER_MAX];
  bf16* p16[CC_PEER_MAX];
};
// low-order terms of the kernels kept as hi + lo: only inside [begin, end) x 2
struct PeerLo {
  bf16* p16lo[CC_PEER_MAX];
  bf16* mc;
  long long begin[2], end[2];
};

__global__ void __launch_bounds__(256)
peer_rmsprop_kernel(const PeerPtrs pp, const int world, float* __restrict__ p32,
                    float* __restrict__ ms, float* __restrict__ mom, const long long start,
                    const long long count, const int broadcast, const float lr, const float rho,
                    const float momentum, const float eps, const uint32_t* ready,
                    const uint32_t epoch_rel, const uint32_t* __restrict__ epoch_ctr,
                    bf16* __restrict__ p16_mc, const PeerLo lo) {
  // epochs: host value, or (CUDA-graph friendly) a device counter plus a constant
  const uint32_t epoch = epoch_rel + (epoch_ctr ? *epoch_ctr : 0u);
  // every rank's gradient for this bucket must be complete (and, because the flags are only
  // raised after the producing wgrad GEMMs, every rank has finished READING the old weights)
  if (threadIdx.x < world) wait_flag(ready + threadIdx.x, epoch, 1);
  __syncthreads();
  const long long n8 = count >> 3;   // count is a multiple of 8 (buckets are multiples of 64)
  const float omr = 1.f - rho;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8;
       i += (long long)gridDim.x * blockDim.x) {
    const long long off = start + (i << 3);
    float g[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) g[k] = 0.f;
    for (int q = 0; q < world; ++q) {
      // .cv: never served from a stale L1 line of an earlier update
      const float4 a = __ldcv(reinterpret_cast<const float4*>(pp.g[q] + off));
      const float4 b = __ldcv(reinterpret_cast<const float4*>(pp.g[q] + off + 4));
      g[0] += a.x; g[1] += a.y; g[2] += a.z; g[3] += a.w;
      g[4] += b.x; g[5] += b.y; g[6] += b.z; g[7] += b.w;
    }
    float w[8], s[8], m[8];
    {
      const float4 a = *reinterpret_cast<const float4*>(p32 + off);
      const float4 b = *reinterpret_cast<const float4*>(p32 + off + 4);
      w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
      const float4 c = *reinterpret_cast<const float4*>(ms + off);
      const float4 d = *reinterpret_cast<const float4*>(ms + off + 4);
      s[0] = c.x; s[1] = c.y; s[2] = c.z; s[3] = c.w; s[4] = d.x; s[5] = d.y; s[6] = d.z; s[7] = d.w;
      const float4 e = *reinterpret_cast<const float4*>(mom + off);
      const float4 f = *reinterpret_cast<const float4*>(mom + off + 4);
      m[0] = e.x; m[1] = e.y; m[2] = e.z; m[3] = e.w; m[4] = f.x; m[5] = f.y; m[6] = f.z; m[7] = f.w;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      s[k] = rho * s[k] + omr * g[k] * g[k];
      m[k] = momentum * m[k] + lr * g[k] * rsqrtf(s[k] + eps);
      w[k] -= m[k];
    }
    *reinterpret_cast<float4*>(p32 + off) = make_float4(w[0], w[1], w[2], w[3]);
    *reinterpret_cast<float4*>(p32 + off + 4) = make_float4(w[4], w[5], w[6], w[7]);
    *reinterpret_cast<float4*>(ms + off) = make_float4(s[0], s[1], s[2], s[3]);
    *reinterpret_cast<float4*>(ms + off + 4) = make_float4(s[4], s[5], s[6], s[7]);
    *reinterpret_cast<float4*>(mom + off) = make_float4(m[0], m[1], m[2], m[3]);
    *reinterpret_cast<float4*>(mom + off + 4) = make_float4(m[4], m[5], m[6], m[7]);
    uint4 u;
    {
      __nv_bfloat162 h0 = __floats2bfloat162_rn(w[0], w[1]), h1 = __floats2bfloat162_rn(w[2], w[3]);
      __nv_bfloat162 h2 = __floats2bfloat162_rn(w[4], w[5]), h3 = __floats2bfloat162_rn(w[6], w[7]);
      u.x = *reinterpret_cast<uint32_t*>(&h0);
      u.y = *reinterpret_cast<uint32_t*>(&h1);
      u.z = *reinterpret_cast<uint32_t*>(&h2);
      u.w = *reinterpret_cast<uint32_t*>(&h3);
    }
    if (broadcast && p16_mc != nullptr) {
      // NVLS: one store to the multicast mapping, the switch replicates it to every rank
      asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p16_mc + off),
                   "f"(__uint_as_float(u.x)), "f"(__uint_as_float(u.y)), "f"(__uint_as_float(u.z)),
                   "f"(__uint_as_float(u.w))
                   : "memory");
    } else if (broadcast) {
      for (int q = 0; q < world; ++q) *reinterpret_cast<uint4*>(pp.p16[q] + off) = u;
    } else {
      *reinterpret_cast<uint4*>(pp.p16[0] + off) = u;   // replicated update: local copy only
    }
    if (lo.p16lo[0] != nullptr &&
        ((off >= lo.begin[0] && off < lo.end[0]) || (off >= lo.begin[1] && off < lo.end[1]))) {
      // hi + lo kernels: the low-order term travels the same way
      uint4 v;
      {
        const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&u);
        float r[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 h = __bfloat1622float2(hp[k]);
          r[2 * k] = w[2 * k] - h.x;
          r[2 * k + 1] = w[2 * k + 1] - h.y;
        }
        __nv_bfloat162 l0 = __floats2bfloat162_rn(r[0], r[1]), l1 = __floats2bfloat162_rn(r[2], r[3]);
        __nv_bfloat162 l2 = __floats2bfloat162_rn(r[4], r[5]), l3 = __floats2bfloat162_rn(r[6], r[7]);
        v.x = *reinterpret_cast<uint32_t*>(&l0);
        v.y = *reinterpret_cast<uint32_t*>(&l1);
        v.z = *reinterpret_cast<uint32_t*>(&l2);
        v.w = *reinterpret_cast<uint32_t*>(&l3);
      }
      if (broadcast && lo.mc != nullptr) {
        asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(lo.mc + off),
                     "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)),
                     "f"(__uint_as_float(v.w))
                     : "memory");
      } else if (broadcast) {
        for (int q = 0; q < world; ++q) *reinterpret_cast<uint4*>(lo.p16lo[q] + off) = v;
      } else {
        *reinterpret_cast<uint4*>(lo.p16lo[0] + off) = v;
      }
    }
  }
}

struct FlagPtrs {
  uint32_t* t[CC_PEER_MAX];
};

// after everything this stream has written so far: *targets[q] = value for every q
__global__ void peer_signal_kernel(const FlagPtrs f, const int n, const uint32_t value_rel,
                                   const uint32_t* __restrict__ epoch_ctr) {
  const uint32_t value = value_rel + (epoch_ctr ? *epoch_ctr : 0u);
  __threadfence_system();
  if (threadIdx.x < n) st_release_sys(f.t[threadIdx.x], value);
}

// bump != 0: the counter advances to the awaited epoch once every flag has arrived (the last
// kernel of an update on its stream; the next update's kernels then see the new base)
__global__ void peer_wait_kernel(const uint32_t* flags, const int n, const uint32_t value_rel,
                                 uint32_t* epoch_ctr, const int bump) {
  const uint32_t value = value_rel + (epoch_ctr ? *epoch_ctr : 0u);
  for (int i = threadIdx.x; i < n; i += blockDim.x) wait_flag(flags + i, value, 2);
  __syncthreads();
  if (bump && epoch_ctr != nullptr && threadIdx.x == 0) *epoch_ctr = value;
}

}  // namespace cc

using namespace cc;

// the kernel moves 8 elements per thread as 16-byte vectors (fp32 float4 pairs, one bf16 uint4)
static bool vec16_at(const void* base, long long start, int elem_bytes) {
  return base == nullptr || (((uintptr_t)base + (uintptr_t)(start * elem_bytes)) & 15) == 0;
}

extern "C" int cc_peer_rmsprop(const cc_peer_rmsprop_desc* d, cc_stream_t stream) {
  CC_REQUIRE(d != nullptr, "cc_peer_rmsprop: null descriptor");
  CC_REQUIRE(d->world >= 1 && d->world <= CC_PEER_MAX, "cc_peer_rmsprop: world=%d", d->world);
  CC_REQUIRE(d->rank >= 0 && d->rank < d->world, "cc_peer_rmsprop: rank=%d of world=%d", d->rank,
             d->world);
  CC_REQUIRE(d->count >= 0 && (d->count & 7) == 0 && (d->start & 7) == 0,
             "cc_peer_rmsprop: range [%lld, +%lld) must be 8-element granular",
             (long long)d->start, (long long)d->count);
  if (d->count == 0) return 0;
  const long long st = d->start;
  CC_REQUIRE(d->p32 && d->ms && d->mom && d->ready, "cc_peer_rmsprop: null p32/ms/mom/ready");
  CC_REQUIRE(vec16_at(d->p32, st, 4) && vec16_at(d->ms, st, 4) && vec16_at(d->mom, st, 4),
             "cc_peer_rmsprop: p32/ms/mom must be 16-byte aligned at start=%lld", st);
  CC_REQUIRE(vec16_at(d->p16_multicast, st, 2) && vec16_at(d->p16lo_multicast, st, 2),
             "cc_peer_rmsprop: multicast pointers must be 16-byte aligned at start=%lld", st);
  const bool has_lo = d->p16lo[0] != nullptr;
  PeerPtrs pp;
  for (int q = 0; q < CC_PEER_MAX; ++q) {
    pp.g[q] = q < d->world ? d->grad[q] : nullptr;
    pp.p16[q] = q < d->world ? (bf16*)d->p16[q] : nullptr;
    CC_REQUIRE(q >= d->world || (pp.g[q] != nullptr && pp.p16[q] != nullptr &&
                                 (!has_lo || d->p16lo[q] != nullptr)),
               "cc_peer_rmsprop: missing peer pointer %d", q);
    CC_REQUIRE(q >= d->world || (vec16_at(pp.g[q], st, 4) && vec16_at(pp.p16[q], st, 2) &&
                                 vec16_at(d->p16lo[q], st, 2)),
               "cc_peer_rmsprop: grad/p16/p16lo of rank %d must be 16-byte aligned at start=%lld",
               q, st);
  }
  if (!d->broadcast) pp.p16[0] = (bf16*)d->p16[d->rank];
  PeerLo lo;
  for (int q = 0; q < CC_PEER_MAX; ++q) lo.p16lo[q] = q < d->world ? (bf16*)d->p16lo[q] : nullptr;
  if (has_lo && !d->broadcast) lo.p16lo[0] = (bf16*)d->p16lo[d->rank];
  lo.mc = (bf16*)d->p16lo_multicast;
  for (int k = 0; k < 2; ++k) {
    lo.begin[k] = d->lo_begin[k];
    lo.end[k] = d->lo_end[k];
    CC_REQUIRE((lo.begin[k] & 7) == 0 && (lo.end[k] & 7) == 0,
               "cc_peer_rmsprop: hi+lo range %d must be 8-element granular", k);
  }
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    CC_CHECK_CUDA(cudaGetDevice(&dev));
    CC_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  // a modest grid: the kernel is bound by NVLink / HBM, and it runs NEXT TO the backward GEMMs
  long long blocks = ((d->count >> 3) + 255) / 256;
  static int per_sm = 0;
  if (per_sm == 0) {
    const char* v = getenv("CC_PEER_BLOCKS_PER_SM");
    per_sm = v ? atoi(v) : 2;
    if (per_sm < 1 || per_sm > 8) per_sm = 2;
  }
  const long long cap = (long long)sms * per_sm;
  if (blocks > cap) blocks = cap;
  peer_rmsprop_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      pp, d->world, d->p32, d->ms, d->mom, d->start, d->count, d->broadcast, d->lr, d->rho,
      d->momentum, d->eps, d->ready, d->epoch, d->epoch_ctr, (bf16*)d->p16_multicast, lo);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_peer_signal(uint32_t* const* targets, int32_t n, uint32_t value,
                              const uint32_t* epoch_ctr, cc_stream_t stream) {
  CC_REQUIRE(n >= 1 && n <= CC_PEER_MAX, "cc_peer_signal: n=%d", n);
  FlagPtrs f;
  for (int q = 0; q < CC_PEER_MAX; ++q) f.t[q] = q < n ? targets[q] : nullptr;
  peer_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(f, n, value, epoch_ctr);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_peer_wait(const uint32_t* flags, int32_t n, uint32_t value, uint32_t* epoch_ctr,
                            int32_t bump, cc_stream_t stream) {
  if (n <= 0) return 0;
  peer_wait_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(flags, n, value, epoch_ctr, bump);
  CC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Small sum all-reduce over peer memory (BatchNorm batch statistics, BN-backward sums, the loss
// buffer: a few KB, ~25 times per training step).  One CTA: push my values into my slot on
// every rank, raise my flag on every rank, wait for everybody's flag, sum the slots in rank
// order (bit-identical result everywhere).  Replaces NCCL's all-reduce for these latency-bound
// reductions: one ~10 us kernel, no host-side collective call, no NCCL CTAs.
//   slots : per rank a [2][world][cap] fp32 array (double-buffered by epoch parity: a rank can
//           run at most one all-reduce ahead of the slowest reader)
//   flags : per rank [world] uint32
namespace cc {

struct ArPtrs {
  float* slots[CC_PEER_MAX];
  uint32_t* flags[CC_PEER_MAX];
};

__global__ void __launch_bounds__(1024)
peer_allreduce_kernel(const ArPtrs ap, const int world, const int rank, float* __restrict__ data,
                      const int n, const long long cap, const uint32_t epoch_rel,
                      uint32_t* epoch_ctr) {
  const uint32_t epoch = epoch_rel + (epoch_ctr ? *epoch_ctr : 0u);
  const long long par = (long long)(epoch & 1u) * world * cap;
  // 1. my contribution into slot [parity][rank] of every rank (own copy included)
  for (int q = 0; q < world; ++q) {
    float* dst = ap.slots[q] + par + (long long)rank * cap;
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = data[i];
  }
  __threadfence_system();
  __syncthreads();
  // 2. publish, 3. wait for everybody
  if (threadIdx.x < world) {
    st_release_sys(ap.flags[threadIdx.x] + rank, epoch);
    wait_flag(ap.flags[rank] + threadIdx.x, epoch, 3);
  }
  __syncthreads();
  // 4. sum in rank order
  const float* mine = ap.slots[rank] + par;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < world; ++q) s += __ldcv(mine + (long long)q * cap + i);
    data[i] = s;
  }
  // (every thread read the counter before the first barrier above)
  if (epoch_ctr != nullptr && threadIdx.x == 0) *epoch_ctr = epoch;
}

}  // namespace cc

extern "C" int cc_peer_allreduce(float* data, int32_t n, int32_t world, int32_t rank,
                                 float* const* slots, uint32_t* const* flags, int64_t cap,
                                 uint32_t epoch, uint32_t* epoch_ctr, cc_stream_t stream) {
  CC_REQUIRE(world >= 1 && world <= CC_PEER_MAX && rank >= 0 && rank < world,
             "cc_peer_allreduce: world=%d rank=%d", world, rank);
  CC_REQUIRE(n >= 0 && n <= cap, "cc_peer_allreduce: n=%d exceeds the slot capacity %lld", n,
             (long long)cap);
  if (n == 0) return 0;
  ArPtrs ap;
  for (int q = 0; q < CC_PEER_MAX; ++q) {
    ap.slots[q] = q < world ? slots[q] : nullptr;
    ap.flags[q] = q < world ? flags[q] : nullptr;
  }
  const int threads = n >= 1024 ? 1024 : ((n + 31) / 32 * 32 < 32 ? 32 : (n + 31) / 32 * 32);
  peer_allreduce_kernel<<<1, threads, 0, (cudaStream_t)stream>>>(ap, world, rank, data, n, cap,
                                                                  epoch, epoch_ctr);
  CC_CHECK_LAUNCH();
  return 0;
}
