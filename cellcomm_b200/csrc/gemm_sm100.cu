// tcgen05 / TMEM / TMA bf16 GEMM with fused epilogue for sm_100a.
//
// D[M,N] = epi( sum_s A_s[M,K_s] * B_s[K_s,N] )         (see include/cellcomm_b200.h)
//
// Replaces the Dense matmuls TensorFlow's CPU runtime executes for
// Model.train_on_batch / Model.predict in the reference
// (src/bigan_classify.py:10-75,144-155, src/bigan_cont.py:7-41).
//
// Structure (one 128 x BN output tile per CTA, 128 threads, 2 CTAs per SM so one
// CTA's epilogue overlaps the other's main loop):
//   warp 0 : TMA producer   (cp.async.bulk.tensor.2d, 128B swizzle, mbarrier tx)
//   warp 1 : tcgen05.mma issuer (single elected lane), owns TMEM alloc/dealloc
//   warps 0-3 : epilogue    (tcgen05.ld 32x32b -> registers -> global)
// Operands can be K-major or MN-major (UMMA "major" bits), so forward
// (A K-major, B MN-major), dgrad (K,K) and wgrad (MN,MN) all read the same
// row-major tensors with no transposes.
// Split-K: gridDim.z CTAs each accumulate a k-block range and write fp32
// partials; splitk_finalize applies the epilogue.
#include <cuda.h>

#include <mutex>
#include <unordered_map>

#include "common.cuh"

namespace cc {

constexpr int BM = 128;     // tile rows  (UMMA M, cta_group::1)
constexpr int BK = 64;      // k-block: 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;  // fixed for 16-bit inputs
constexpr int MAX_SEG = CC_GEMM_MAX_SEG;

struct EpiParams {
  int M, N;
  float alpha;
  const float* bias;
  int act;
  const bf16* dact_y;
  long long ld_dact;
  int dact;
  bf16* out16;
  long long ld16;
  int beta16;
  bf16* out16_lo;      // low-order term of a two-term bf16 expansion (out16 = the high-order one)
  long long ld16_lo;
  float* out32;
  long long ld32;
  int beta32;
  // fused Keras RMSprop(momentum) on the tile (wgrad epilogue): the accumulator IS the gradient
  float* rms_p32;
  float* rms_ms;
  float* rms_mom;
  bf16* rms_p16;
  long long rms_ld;
  float rms_lr, rms_rho, rms_momentum, rms_eps;
  // blocked optimiser-state layout (cc_gemm_desc.rms_blocked): rms_p32 / rms_ms / rms_mom are
  // the LAYER's blocked arrays, this GEMM's rows start at layer row rms_row0
  int rms_blocked;
  int rms_row0;
  bf16* rms_p16lo;  // blocked path: low-order bf16 term of the updated weight (hi + lo kernels)
  // routed fp32 output (data-parallel wgrad): element `rel` of the bucket goes to the rank that
  // owns it, route_base[owner] + rel (peer-mapped staging slot; own share: local memory)
  int route_world;
  unsigned int route_shard;
  long long route_off0;
  float* route_base[CC_PEER_MAX];
};

struct GemmParams {
  EpiParams epi;
  int nseg;
  int kblocks[MAX_SEG];  // k-blocks per segment
  int total_kblocks;
  int kb_per_split;      // k-blocks handled by one blockIdx.z
  int psplits;           // persistent kernel: k-ranges per tile (work unit = tile x k-range)
  float* partial;        // split-K partials [splits][Mpad][Npad] or nullptr
  long long partial_ld;      // Npad
  long long partial_stride;  // Mpad*Npad
  // smem matrix descriptor templates (everything except the start address)
  unsigned long long adesc_hi, bdesc_hi;
  unsigned int a_kstep, b_kstep;  // bytes to advance the start address per UMMA_K
  unsigned int idesc;
  // persistent kernel: effective tile width (multiple of 32, <= BN).  The smem / TMEM layout
  // stays BN wide; a narrower MMA N trades a little per-tile efficiency for a tile count that
  // fills the last wave (N = 3369 at BN 256 is 1.51 waves, at 192 it is 1.95).
  int bn_eff;
  int b_boxes;            // MN-major B: 64-column TMA boxes per stage
  int b_half_rows;        // K-major B in a 2-CTA cluster: rows of the tile each CTA loads
  int cluster;            // 1 or 2 CTAs per cluster (persistent kernel)
  unsigned int stage_tx;  // bytes TMA delivers per stage
};

struct TmaMaps {
  CUtensorMap a[MAX_SEG];
  CUtensorMap b[MAX_SEG];
};

// ----------------------------------------------------------------------- PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must trap (recoverable) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag) {
  long long t0 = 0;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins == 4096u) t0 = clock64();
    if (spins > 4096u && (spins & 1023u) == 0 && clock64() - t0 > 4000000000LL) {
      printf("cc_gemm: mbarrier timeout tag=%d block=(%d,%d,%d) thread=%d parity=%u\n", tag,
             blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
      "{%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// One lane of a converged warp (elect.sync): ptxas then issues the uniform-datapath TMA / MMA
// instructions under a plain predicate instead of a per-lane ELECT/BRA.U.ANY retry loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// --------------------------------------------------------------- epilogue math
// One thread owns 32 consecutive columns [c0, c0+32) of row r.
__device__ __forceinline__ void epilogue_store32(const EpiParams& e, int r, int c0, float (&v)[32]) {
  if (r >= e.M) return;
  const int ncols = min(32, e.N - c0);
  if (ncols <= 0) return;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    // fmaf(v, alpha, bias), one rounding: epilogue_chunk (persistent kernel) and
    // splitk_finalize_kernel compute the same expression, so the bits do not depend on the path
    float x = fmaf(v[j], e.alpha, (e.bias != nullptr && j < ncols) ? __ldg(e.bias + c0 + j) : 0.f);
    if (e.act == CC_ACT_SIGMOID) x = sigmoidf_(x);
    else if (e.act == CC_ACT_RELU) x = fmaxf(x, 0.f);
    v[j] = x;
  }
  if (e.dact != 0) {
    const bf16* yrow = e.dact_y + (long long)r * e.ld_dact + c0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (j < ncols) {
        float y = bf2f(yrow[j]);
        v[j] *= (e.dact == CC_ACT_SIGMOID) ? y * (1.f - y) : (y > 0.f ? 1.f : 0.f);
      }
    }
  }
  if (e.out32 != nullptr) {
    float* o = e.out32 + (long long)r * e.ld32 + c0;
    if (ncols == 32 && (((uintptr_t)o) & 15) == 0 && !e.beta32) {
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < ncols) o[j] = e.beta32 ? o[j] + v[j] : v[j];
    }
  }
  if (e.out16 != nullptr) {
    bf16* o = e.out16 + (long long)r * e.ld16 + c0;
    if (ncols == 32 && (((uintptr_t)o) & 15) == 0 && !e.beta16) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        __nv_bfloat162 p0 = __floats2bfloat162_rn(v[j], v[j + 1]);
        __nv_bfloat162 p1 = __floats2bfloat162_rn(v[j + 2], v[j + 3]);
        __nv_bfloat162 p2 = __floats2bfloat162_rn(v[j + 4], v[j + 5]);
        __nv_bfloat162 p3 = __floats2bfloat162_rn(v[j + 6], v[j + 7]);
        uint4 u;
        u.x = *reinterpret_cast<uint32_t*>(&p0);
        u.y = *reinterpret_cast<uint32_t*>(&p1);
        u.z = *reinterpret_cast<uint32_t*>(&p2);
        u.w = *reinterpret_cast<uint32_t*>(&p3);
        *reinterpret_cast<uint4*>(o + j) = u;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < ncols) o[j] = f2bf(e.beta16 ? bf2f(o[j]) + v[j] : v[j]);
    }
    if (e.out16_lo != nullptr) {
      bf16* l = e.out16_lo + (long long)r * e.ld16_lo + c0;
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < ncols) l[j] = f2bf(v[j] - bf2f(f2bf(v[j])));
    }
  }
}

// Persistent-kernel epilogue for one 32 x 32 block of a warp (thread `lane` holds the raw fp32
// accumulators of row r0+lane, columns c0..c0+31).  The block is transposed through a padded
// smem tile (row stride 36 floats: the 16-byte row writes and the 16-byte reads are both
// bank-conflict free); afterwards lane (rs = lane/8, cg = lane%8) owns columns c0+4cg..+3 of
// rows rs, rs+4, ..., rs+28, so every global instruction of the warp touches 4 rows x 128
// contiguous bytes (fp32) and bias / act' operands are loaded once per lane, vectorised.
// MATH = false strips alpha / bias / activation / act' (wgrad and dgrad tiles).
constexpr int EPI_LD = 36;

__device__ __forceinline__ float4 act4(float4 v, int act) {
  if (act == CC_ACT_SIGMOID) {
    v.x = sigmoidf_(v.x); v.y = sigmoidf_(v.y); v.z = sigmoidf_(v.z); v.w = sigmoidf_(v.w);
  } else if (act == CC_ACT_RELU) {
    v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
  }
  return v;
}

template <int K>
__device__ __forceinline__ float f4c(const float4& v) {
  return K == 0 ? v.x : (K == 1 ? v.y : (K == 2 ? v.z : v.w));
}
template <int K>
__device__ __forceinline__ void f4set(float4& v, float x) {
  if (K == 0) v.x = x; else if (K == 1) v.y = x; else if (K == 2) v.z = x; else v.w = x;
}
// apply f(t, k, value&) to every valid (row t, column k) of the lane's 8 x 4 block, fully
// unrolled (no dynamically indexed local arrays -> no stack traffic)
template <typename F>
__device__ __forceinline__ void for_each_valid(float4 (&g)[8], int nrow, int ncol, F f) {
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    if (t < nrow) {
      if (0 < ncol) f(t, 0, g[t].x);
      if (1 < ncol) f(t, 1, g[t].y);
      if (2 < ncol) f(t, 2, g[t].z);
      if (3 < ncol) f(t, 3, g[t].w);
    }
  }
}

template <bool MATH>
__device__ __forceinline__ void epilogue_chunk(const EpiParams& e, float* stage /*32x36*/, int lane,
                                               int r0, int c0, const uint32_t (&raw)[32],
                                               long long out32_off = 0) {
#pragma unroll
  for (int j = 0; j < 32; j += 4)
    *reinterpret_cast<uint4*>(stage + lane * EPI_LD + j) =
        make_uint4(raw[j], raw[j + 1], raw[j + 2], raw[j + 3]);
  __syncwarp();
  const int rs = lane >> 3, cg = lane & 7;
  const int c = c0 + 4 * cg;
  const int ncol = min(4, e.N - c);  // valid columns of this lane's float4 (<= 0: none)
  float4 g[8];
#pragma unroll
  for (int t = 0; t < 8; ++t)
    g[t] = *reinterpret_cast<const float4*>(stage + (t * 4 + rs) * EPI_LD + 4 * cg);
  __syncwarp();  // the tile may be overwritten by the next chunk from here on
  if (ncol <= 0) return;
  const int rbase = r0 + rs;               // rows rbase + 4t
  const int nrow = (e.M - rbase + 3) >> 2;  // number of valid t (may be <= 0 or > 8)

  if (MATH) {
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (e.bias != nullptr) {
      if (ncol == 4 && ((((uintptr_t)(e.bias + c)) & 15) == 0)) {
        b4 = __ldg(reinterpret_cast<const float4*>(e.bias + c));
      } else {
        b4.x = __ldg(e.bias + c);
        if (ncol > 1) b4.y = __ldg(e.bias + c + 1);
        if (ncol > 2) b4.z = __ldg(e.bias + c + 2);
        if (ncol > 3) b4.w = __ldg(e.bias + c + 3);
      }
    }
    const float al = e.alpha;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      g[t].x = fmaf(g[t].x, al, b4.x);
      g[t].y = fmaf(g[t].y, al, b4.y);
      g[t].z = fmaf(g[t].z, al, b4.z);
      g[t].w = fmaf(g[t].w, al, b4.w);
      g[t] = act4(g[t], e.act);
    }
    if (e.dact != 0) {
      const bf16* y0 = e.dact_y + (long long)rbase * e.ld_dact + c;
      const long long ystep = 4 * e.ld_dact;
      const int dact = e.dact;
      for_each_valid(g, nrow, ncol, [&](int t, int k, float& x) {
        const float yy = bf2f(y0[t * ystep + k]);
        x *= (dact == CC_ACT_SIGMOID) ? yy * (1.f - yy) : (yy > 0.f ? 1.f : 0.f);
      });
    }
  }

  if (e.rms_p32 != nullptr) {
    // fused Keras RMSprop(momentum): ms = rho*ms + (1-rho) g^2 ; mom = momentum*mom +
    // lr*g/sqrt(ms+eps) ; w -= mom ; bf16 copy.  All loads are issued before the first use;
    // the state is streamed with evict-first (.cs) hints.
    const bool vec = ncol == 4 && (e.rms_ld & 3) == 0 && ((c & 3) == 0) &&
                     ((((uintptr_t)e.rms_p32) & 15) == 0) && ((((uintptr_t)e.rms_ms) & 15) == 0) &&
                     ((((uintptr_t)e.rms_mom) & 15) == 0) &&
                     (e.rms_p16 == nullptr || (((uintptr_t)e.rms_p16) & 7) == 0);
    const long long off0 = (long long)rbase * e.rms_ld + c;
    const long long step = 4 * e.rms_ld;
    if (vec) {
      float4 w[8], s[8], m[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (t < nrow) {
          const long long off = off0 + t * step;
          w[t] = __ldcs(reinterpret_cast<const float4*>(e.rms_p32 + off));
          s[t] = __ldcs(reinterpret_cast<const float4*>(e.rms_ms + off));
          m[t] = __ldcs(reinterpret_cast<const float4*>(e.rms_mom + off));
        }
      }
      const float rho = e.rms_rho, omr = 1.f - e.rms_rho, mu = e.rms_momentum, lr = e.rms_lr,
                  eps = e.rms_eps;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (t < nrow) {
          const long long off = off0 + t * step;
          float4 ss, mm, ww;
          ss.x = rho * s[t].x + omr * g[t].x * g[t].x;
          ss.y = rho * s[t].y + omr * g[t].y * g[t].y;
          ss.z = rho * s[t].z + omr * g[t].z * g[t].z;
          ss.w = rho * s[t].w + omr * g[t].w * g[t].w;
          mm.x = mu * m[t].x + lr * g[t].x * rsqrtf(ss.x + eps);
          mm.y = mu * m[t].y + lr * g[t].y * rsqrtf(ss.y + eps);
          mm.z = mu * m[t].z + lr * g[t].z * rsqrtf(ss.z + eps);
          mm.w = mu * m[t].w + lr * g[t].w * rsqrtf(ss.w + eps);
          ww.x = w[t].x - mm.x;
          ww.y = w[t].y - mm.y;
          ww.z = w[t].z - mm.z;
          ww.w = w[t].w - mm.w;
          __stcs(reinterpret_cast<float4*>(e.rms_ms + off), ss);
          __stcs(reinterpret_cast<float4*>(e.rms_mom + off), mm);
          __stcs(reinterpret_cast<float4*>(e.rms_p32 + off), ww);
          if (e.rms_p16 != nullptr) {
            __nv_bfloat162 lo = __floats2bfloat162_rn(ww.x, ww.y);
            __nv_bfloat162 hi = __floats2bfloat162_rn(ww.z, ww.w);
            uint2 u;
            u.x = *reinterpret_cast<uint32_t*>(&lo);
            u.y = *reinterpret_cast<uint32_t*>(&hi);
            *reinterpret_cast<uint2*>(e.rms_p16 + off) = u;
          }
        }
      }
    } else {
      for_each_valid(g, nrow, ncol, [&](int t, int k, float& gv) {
        const long long off = off0 + t * step + k;
        const float ms = e.rms_rho * e.rms_ms[off] + (1.f - e.rms_rho) * gv * gv;
        const float mo = e.rms_momentum * e.rms_mom[off] + e.rms_lr * gv * rsqrtf(ms + e.rms_eps);
        const float w = e.rms_p32[off] - mo;
        e.rms_ms[off] = ms;
        e.rms_mom[off] = mo;
        e.rms_p32[off] = w;
        if (e.rms_p16 != nullptr) e.rms_p16[off] = f2bf(w);
      });
    }
  }
  if (e.route_world > 0) {
    // the reduce-scatter's data movement, done by the GEMM: store each row segment to its owner
    const long long rel0 = e.route_off0 + (long long)rbase * e.ld32 + c;
    const long long step = 4 * e.ld32;
    const unsigned last = (unsigned)e.route_world - 1u;
    const bool vec = ncol == 4 && (e.ld32 & 3) == 0 && ((c & 3) == 0);
    auto owner_of = [&](long long rel) {
      return min((unsigned)((unsigned long long)rel / e.route_shard), last);
    };
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      if (t < nrow) {
        const long long rel = rel0 + t * step;
        if (vec) {
          // rel % 4 == 0 and route_shard % 8 == 0: the four elements have one owner
          *reinterpret_cast<float4*>(e.route_base[owner_of(rel)] + rel) = g[t];
        } else {
          // rel % 4 != 0 when ld32 % 4 != 0: a shard boundary may fall inside the four
          // columns, so every element finds its own owner
          e.route_base[owner_of(rel)][rel] = g[t].x;
          if (ncol > 1) e.route_base[owner_of(rel + 1)][rel + 1] = g[t].y;
          if (ncol > 2) e.route_base[owner_of(rel + 2)][rel + 2] = g[t].z;
          if (ncol > 3) e.route_base[owner_of(rel + 3)][rel + 3] = g[t].w;
        }
      }
    }
  } else if (e.out32 != nullptr) {
    float* o = e.out32 + out32_off + (long long)rbase * e.ld32 + c;   // (+ the split's partial)
    const long long step = 4 * e.ld32;
    if (ncol == 4 && !e.beta32 && (e.ld32 & 3) == 0 && ((c & 3) == 0) &&
        ((((uintptr_t)e.out32) & 15) == 0)) {
#pragma unroll
      for (int t = 0; t < 8; ++t)
        if (t < nrow) *reinterpret_cast<float4*>(o + t * step) = g[t];
    } else {
      const int beta = e.beta32;
      for_each_valid(g, nrow, ncol, [&](int t, int k, float& gv) {
        float* ot = o + t * step + k;
        *ot = beta ? *ot + gv : gv;
      });
    }
  }
  if (e.out16 != nullptr) {
    bf16* o = e.out16 + (long long)rbase * e.ld16 + c;
    const long long step = 4 * e.ld16;
    if (ncol == 4 && !e.beta16 && (e.ld16 & 3) == 0 && ((c & 3) == 0) &&
        ((((uintptr_t)e.out16) & 7) == 0)) {
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (t < nrow) {
          __nv_bfloat162 lo = __floats2bfloat162_rn(g[t].x, g[t].y);
          __nv_bfloat162 hi = __floats2bfloat162_rn(g[t].z, g[t].w);
          uint2 u;
          u.x = *reinterpret_cast<uint32_t*>(&lo);
          u.y = *reinterpret_cast<uint32_t*>(&hi);
          *reinterpret_cast<uint2*>(o + t * step) = u;
        }
      }
    } else {
      const int beta = e.beta16;
      for_each_valid(g, nrow, ncol, [&](int t, int k, float& gv) {
        bf16* ot = o + t * step + k;
        *ot = f2bf(beta ? bf2f(*ot) + gv : gv);
      });
    }
    if (e.out16_lo != nullptr) {
      bf16* l = e.out16_lo + (long long)rbase * e.ld16_lo + c;
      const long long lstep = 4 * e.ld16_lo;
      if (ncol == 4 && (e.ld16_lo & 3) == 0 && ((c & 3) == 0) && ((((uintptr_t)e.out16_lo) & 7) == 0)) {
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          if (t < nrow) {
            const float4 v = g[t];
            __nv_bfloat162 lo = __floats2bfloat162_rn(v.x - bf2f(f2bf(v.x)), v.y - bf2f(f2bf(v.y)));
            __nv_bfloat162 hi = __floats2bfloat162_rn(v.z - bf2f(f2bf(v.z)), v.w - bf2f(f2bf(v.w)));
            uint2 u;
            u.x = *reinterpret_cast<uint32_t*>(&lo);
            u.y = *reinterpret_cast<uint32_t*>(&hi);
            *reinterpret_cast<uint2*>(l + t * lstep) = u;
          }
        }
      } else {
        for_each_valid(g, nrow, ncol, [&](int t, int k, float& gv) {
          l[t * lstep + k] = f2bf(gv - bf2f(f2bf(gv)));
        });
      }
    }
  }
}

// ------------------------------------------------------------------- kernel
template <int BN, int STAGES, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(128, 2)
gemm_tcgen05_kernel(const __grid_constant__ TmaMaps maps, const GemmParams p) {
  constexpr uint32_t A_BYTES = BM * BK * 2;
  constexpr uint32_t B_BYTES = BN * BK * 2;
  constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = BN;  // fp32 accumulator: one column per N

  extern __shared__ uint8_t smem_raw[];
  // 128B swizzle atoms need 1024B-aligned tiles
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
  // barriers: full[STAGES], empty[STAGES], tmem_full, then tmem ptr slot
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * STAGES);
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 1);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_gen + STAGES * STAGE_BYTES + 8u * (2 * STAGES + 1));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * BM;
  const int n0 = blockIdx.x * BN;
  const int kb_begin = blockIdx.z * p.kb_per_split;
  const int kb_end = min(p.total_kblocks, kb_begin + p.kb_per_split);
  const int nkb = kb_end - kb_begin;

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    int seg = 0, kb_in_seg = kb_begin;
    while (seg < p.nseg - 1 && kb_in_seg >= p.kblocks[seg]) {
      kb_in_seg -= p.kblocks[seg];
      ++seg;
    }
    for (int i = 0; i < nkb; ++i) {
      const int s = i % STAGES;
      const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
      mbar_wait(empty_bar(s), ph ^ 1u, 1);
      if (elect_one()) {
        const uint32_t a_dst = smem_base + s * STAGE_BYTES;
        const uint32_t b_dst = a_dst + A_BYTES;
        const int k0 = kb_in_seg * BK;
        mbar_expect_tx(full_bar(s), STAGE_BYTES);
        if (A_MN) {
          // A stored [K, M]: inner = M.  Two 64-wide boxes of BK rows each.
#pragma unroll
          for (int j = 0; j < BM / 64; ++j)
            tma_load_2d(a_dst + j * (64 * BK * 2), &maps.a[seg], full_bar(s), m0 + 64 * j, k0);
        } else {
          // A stored [M, K]: inner = K.  One box 64(K) x 128(M).
          tma_load_2d(a_dst, &maps.a[seg], full_bar(s), k0, m0);
        }
        if (B_MN) {
#pragma unroll
          for (int j = 0; j < BN / 64; ++j)
            tma_load_2d(b_dst + j * (64 * BK * 2), &maps.b[seg], full_bar(s), n0 + 64 * j, k0);
        } else {
          tma_load_2d(b_dst, &maps.b[seg], full_bar(s), k0, n0);
        }
      }
      __syncwarp();
      if (++kb_in_seg >= p.kblocks[seg] && seg < p.nseg - 1) {
        kb_in_seg = 0;
        ++seg;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    for (int i = 0; i < nkb; ++i) {
      const int s = i % STAGES;
      const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
      mbar_wait(full_bar(s), ph, 2);
      tcgen05_fence_after();
      if (elect_one()) {
        const uint32_t a_src = smem_base + s * STAGE_BYTES;
        const uint32_t b_src = a_src + A_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint64_t adesc = p.adesc_hi | (uint64_t)(((a_src + k * p.a_kstep) & 0x3FFFFu) >> 4);
          const uint64_t bdesc = p.bdesc_hi | (uint64_t)(((b_src + k * p.b_kstep) & 0x3FFFFu) >> 4);
          umma_bf16(tmem_acc, adesc, bdesc, p.idesc, (i > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(empty_bar(s));  // frees this smem stage when the MMAs retire
        if (i == nkb - 1) umma_commit(tmem_full_bar);
      }
      __syncwarp();
    }
  }

  // ===================== epilogue (all 4 warps) =====================
  mbar_wait(tmem_full_bar, 0, 3);
  tcgen05_fence_after();
  {
    const int r = m0 + warp * 32 + lane;
    const uint32_t t_row = tmem_acc + ((uint32_t)(warp * 32) << 16);
    const bool split = (p.partial != nullptr);
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      if (n0 + c >= p.epi.N) break;  // warp-uniform
      uint32_t raw[32];
      tmem_ld32(t_row + (uint32_t)c, raw);
      tmem_ld_wait();
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(raw[j]);
      if (split) {
        if (r < p.epi.M) {
          float* o = p.partial + (long long)blockIdx.z * p.partial_stride +
                     (long long)r * p.partial_ld + n0 + c;
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      } else {
        epilogue_store32(p.epi, r, n0 + c, v);
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc),
                 "r"(TMEM_COLS)
                 : "memory");
  }
}

// ------------------------------------------------------- persistent warp-specialised kernel
// One CTA per SM loops over output tiles (m fastest, so concurrently running CTAs share the
// same B / weight tile through L2).  Warp 0 = TMA producer, warp 1 = MMA issuer, warps 2.. =
// epilogue.  The fp32 accumulator is double-buffered in TMEM (2 x BN columns), so the epilogue
// of tile i overlaps the main loop of tile i+1, and the smem ring has STAGES k-blocks in
// flight across tile boundaries.
//
// CLUSTER = 2: two CTAs (an SM pair) work on vertically adjacent tiles (same n-tile, m-tiles
// 2j and 2j+1).  Each CTA loads its own A tile and HALF of the shared B tile, multicast into
// both CTAs' smem (cp.async.bulk.tensor ... .multicast::cluster), so the L2 -> SM operand
// traffic per k-block drops from 48 KB to 32 KB per CTA -- the big GEMMs are bound by that
// traffic (ncu: ~15.7 TB/s xbar reads at 74 % tensor-pipe activity), not by the tensor pipe.
// A stage may only be refilled once BOTH CTAs' MMAs have consumed it: the empty barriers
// count two arrivals and every tcgen05.commit is multicast to both CTAs.
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                               int c0, int c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      ".multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(bar),
      "h"(mask)
      : "memory");
}

// Fused RMSprop on one 32 x 32 accumulator chunk with the optimiser state in the BLOCKED layout
// (include/cellcomm_b200.h, cc_gemm_desc.rms_blocked): the three fp32 arrays of a layer are
// stored as 32-row x 32-column blocks of 4 KB, block (rb, cb) at ((rb * ld/32) + cb) * 1024
// floats, and inside a block element (r, c) at (c/4) * 128 + r * 4 + c % 4 -- the order in which
// tcgen05.ld 32x32b hands a warp its accumulators (lane = row, registers = columns).  Each of the
// eight float4 accesses per array then covers 512 contiguous bytes and the chunk one 4 KB block
// per array, with no shared-memory transpose (the smem it used buys a fourth operand stage)
// and row-major 128-byte pieces ld * 4 bytes apart replaced by whole DRAM pages.  A GEMM whose
// first row is not a multiple of 32 in the layer (second Concatenate segment) simply has its
// lanes wrap into the next block row.  The bf16 compute copy (a TMA operand of the forward
// GEMMs) and the optional gradient output stay row-major: 64 / 128 bytes per lane.
__device__ __forceinline__ void rms_blocked_chunk(const EpiParams& e, int lane, int r0, int c0,
                                                  const uint32_t (&raw)[32]) {
  const int r = r0 + lane;  // row of this GEMM's output
  if (r >= e.M) return;
  const int row = e.rms_row0 + r;  // row of the layer's kernel
  const long long sb =
      ((long long)(row >> 5) * (e.rms_ld >> 5) + (c0 >> 5)) * 1024 + (long long)(row & 31) * 4;
  float* pw = e.rms_p32 + sb;
  float* ps = e.rms_ms + sb;
  float* pm = e.rms_mom + sb;
  float4 w[8], s[8], m[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    w[t] = __ldcs(reinterpret_cast<const float4*>(pw + t * 128));
    s[t] = __ldcs(reinterpret_cast<const float4*>(ps + t * 128));
    m[t] = __ldcs(reinterpret_cast<const float4*>(pm + t * 128));
  }
  const float rho = e.rms_rho, omr = 1.f - e.rms_rho, mu = e.rms_momentum, lr = e.rms_lr,
              eps = e.rms_eps;
  const int nvalid = e.N - c0;  // columns of this chunk inside the matrix (padding: gradient 0)
  uint32_t h[16], hl[16];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    float g0 = (4 * t + 0 < nvalid) ? __uint_as_float(raw[4 * t + 0]) : 0.f;
    float g1 = (4 * t + 1 < nvalid) ? __uint_as_float(raw[4 * t + 1]) : 0.f;
    float g2 = (4 * t + 2 < nvalid) ? __uint_as_float(raw[4 * t + 2]) : 0.f;
    float g3 = (4 * t + 3 < nvalid) ? __uint_as_float(raw[4 * t + 3]) : 0.f;
    float4 ss, mm, ww;
    ss.x = rho * s[t].x + omr * g0 * g0;
    ss.y = rho * s[t].y + omr * g1 * g1;
    ss.z = rho * s[t].z + omr * g2 * g2;
    ss.w = rho * s[t].w + omr * g3 * g3;
    mm.x = mu * m[t].x + lr * g0 * rsqrtf(ss.x + eps);
    mm.y = mu * m[t].y + lr * g1 * rsqrtf(ss.y + eps);
    mm.z = mu * m[t].z + lr * g2 * rsqrtf(ss.z + eps);
    mm.w = mu * m[t].w + lr * g3 * rsqrtf(ss.w + eps);
    ww.x = w[t].x - mm.x;
    ww.y = w[t].y - mm.y;
    ww.z = w[t].z - mm.z;
    ww.w = w[t].w - mm.w;
    __stcs(reinterpret_cast<float4*>(ps + t * 128), ss);
    __stcs(reinterpret_cast<float4*>(pm + t * 128), mm);
    __stcs(reinterpret_cast<float4*>(pw + t * 128), ww);
    __nv_bfloat162 lo = __floats2bfloat162_rn(ww.x, ww.y);
    __nv_bfloat162 hi = __floats2bfloat162_rn(ww.z, ww.w);
    h[2 * t] = *reinterpret_cast<uint32_t*>(&lo);
    h[2 * t + 1] = *reinterpret_cast<uint32_t*>(&hi);
    if (e.rms_p16lo != nullptr) {  // hi + lo kernels: lo = bf16(w - float(bf16(w)))
      __nv_bfloat162 l0 = __floats2bfloat162_rn(ww.x - __uint_as_float(h[2 * t] << 16),
                                                ww.y - __uint_as_float(h[2 * t] & 0xFFFF0000u));
      __nv_bfloat162 l1 = __floats2bfloat162_rn(ww.z - __uint_as_float(h[2 * t + 1] << 16),
                                                ww.w - __uint_as_float(h[2 * t + 1] & 0xFFFF0000u));
      hl[2 * t] = *reinterpret_cast<uint32_t*>(&l0);
      hl[2 * t + 1] = *reinterpret_cast<uint32_t*>(&l1);
    }
    if (e.out32 != nullptr)  // the gradient itself (parity tests); row-major, padding stays 0
      *reinterpret_cast<float4*>(e.out32 + (long long)r * e.ld32 + c0 + 4 * t) =
          make_float4(g0, g1, g2, g3);
  }
  if (e.rms_p16 != nullptr) {
    uint4* dst = reinterpret_cast<uint4*>(e.rms_p16 + (long long)r * e.rms_ld + c0);
#pragma unroll
    for (int t = 0; t < 4; ++t) dst[t] = make_uint4(h[4 * t], h[4 * t + 1], h[4 * t + 2], h[4 * t + 3]);
  }
  if (e.rms_p16lo != nullptr) {
    uint4* dst = reinterpret_cast<uint4*>(e.rms_p16lo + (long long)r * e.rms_ld + c0);
#pragma unroll
    for (int t = 0; t < 4; ++t)
      dst[t] = make_uint4(hl[4 * t], hl[4 * t + 1], hl[4 * t + 2], hl[4 * t + 3]);
  }
}

// N_FAST: consecutive tiles walk along N (the contiguous direction of the output / parameter
// matrix), so the CTAs of one wave cover whole output rows: used by the fused-optimiser wgrad,
// whose epilogue streams 26 B per element and wants DRAM-page-local bursts.
template <int BN, int STAGES, bool A_MN, bool B_MN, bool MATH, int EPI_WARPS, bool N_FAST = false,
          int CLUSTER = 1, bool RMS_DIRECT = false>
__global__ void __launch_bounds__(64 + 32 * EPI_WARPS, 1)
gemm_tcgen05_persistent_kernel(const __grid_constant__ TmaMaps maps,
                               const __grid_constant__ GemmParams p,
                               const int tiles_m, const int tiles_n) {
  constexpr uint32_t A_BYTES = BM * BK * 2;
  constexpr uint32_t B_BYTES = BN * BK * 2;
  constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = 2 * BN;  // two accumulator stages
  static_assert(TMEM_COLS <= 512, "TMEM has 512 columns");
  static_assert(CLUSTER == 1 || CLUSTER == 2, "cluster of 1 or 2 CTAs");

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_gen + STAGES * STAGE_BYTES + 8u * (2 * STAGES + 4));
  // per-epilogue-warp 32x36 fp32 transpose tiles, after the barrier block
  float* epi_stage = reinterpret_cast<float*>(smem_gen + STAGES * STAGE_BYTES + 8u * (2 * STAGES + 6));  // 16-B aligned: 2*STAGES+6 is even

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // work units: one tile (CLUSTER 1) or a vertical pair of tiles (CLUSTER 2)
  const int rank = (CLUSTER == 2) ? (int)cluster_ctarank() : 0;
  const int tiles_mu = (tiles_m + CLUSTER - 1) / CLUSTER;
  // split-K (weight-streaming regime): a work unit is a tile x one of `psplits` k-ranges; the
  // tile index varies fastest, so the CTAs running side by side share the same k-slab of A
  // through L2, and the operand ring / TMEM double buffering run across units like across tiles
  const int num_tiles = tiles_mu * tiles_n;
  const int psplits = p.psplits > 1 ? p.psplits : 1;
  const int num_units = num_tiles * psplits;
  const int unit0 = (int)blockIdx.x / CLUSTER, unit_step = (int)gridDim.x / CLUSTER;
  auto unit_tile = [&](int u) { return psplits > 1 ? u % num_tiles : u; };
  auto unit_split = [&](int u) { return psplits > 1 ? u / num_tiles : 0; };
  auto unit_m0 = [&](int u) {
    const int t = unit_tile(u);
    return ((N_FAST ? t / tiles_n : t % tiles_mu) * CLUSTER + rank) * BM;
  };
  auto unit_n0 = [&](int u) {
    const int t = unit_tile(u);
    return (N_FAST ? t % tiles_n : t / tiles_mu) * p.bn_eff;
  };
  // k-blocks [kb0, kb0 + count) of a unit
  auto unit_kb0 = [&](int u) { return unit_split(u) * p.kb_per_split; };
  auto unit_nkb = [&](int u) {
    return psplits > 1 ? min(p.kb_per_split, p.total_kblocks - unit_kb0(u)) : p.total_kblocks;
  };

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), CLUSTER);  // one commit from every CTA of the cluster
    }
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), EPI_WARPS);  // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  if (CLUSTER == 2) cluster_sync_all();  // the peer's barriers exist before anything is sent to them
  tcgen05_fence_after();
  const uint32_t tmem_acc = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    uint32_t it = 0;
    for (int u = unit0; u < num_units; u += unit_step) {
      const int m0 = unit_m0(u), n0 = unit_n0(u);
      const int nkb_u = unit_nkb(u);
      int seg = 0, kb_in_seg = unit_kb0(u);   // first k-block of the unit's range -> (segment, offset)
      while (seg < p.nseg - 1 && kb_in_seg >= p.kblocks[seg]) {
        kb_in_seg -= p.kblocks[seg];
        ++seg;
      }
      for (int i = 0; i < nkb_u; ++i, ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (it / STAGES) & 1u;
        mbar_wait(empty_bar(s), ph ^ 1u, 11);
        if (elect_one()) {
          const uint32_t a_dst = smem_base + s * STAGE_BYTES;
          const uint32_t b_dst = a_dst + A_BYTES;
          const int k0 = kb_in_seg * BK;
          mbar_expect_tx(full_bar(s), p.stage_tx);
          if (A_MN) {
#pragma unroll
            for (int j = 0; j < BM / 64; ++j)
              tma_load_2d(a_dst + j * (64 * BK * 2), &maps.a[seg], full_bar(s), m0 + 64 * j, k0);
          } else {
            tma_load_2d(a_dst, &maps.a[seg], full_bar(s), k0, m0);
          }
          if (CLUSTER == 2) {
            // this CTA's half of the B tile, delivered to both CTAs
            if (B_MN) {
#pragma unroll
              for (int j = 0; j < BN / 64; ++j)
                if (j < p.b_boxes && (j & 1) == rank)
                  tma_load_2d_mc(b_dst + j * (64 * BK * 2), &maps.b[seg], full_bar(s), n0 + 64 * j,
                                 k0, (uint16_t)3);
            } else {
              tma_load_2d_mc(b_dst + rank * p.b_half_rows * (BK * 2), &maps.b[seg], full_bar(s), k0,
                             n0 + rank * p.b_half_rows, (uint16_t)3);
            }
          } else if (B_MN) {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              if (j < p.b_boxes)
                tma_load_2d(b_dst + j * (64 * BK * 2), &maps.b[seg], full_bar(s), n0 + 64 * j, k0);
          } else {
            tma_load_2d(b_dst, &maps.b[seg], full_bar(s), k0, n0);
          }
        }
        __syncwarp();
        if (++kb_in_seg >= p.kblocks[seg] && seg < p.nseg - 1) {
          kb_in_seg = 0;
          ++seg;
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    uint32_t it = 0, tl = 0;
    for (int u = unit0; u < num_units; u += unit_step, ++tl) {
      const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
      mbar_wait(tempty_bar(acc), aph ^ 1u, 12);  // epilogue has drained this accumulator
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_acc + acc * BN;
      const int nkb = unit_nkb(u);
      for (int i = 0; i < nkb; ++i, ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (it / STAGES) & 1u;
        mbar_wait(full_bar(s), ph, 13);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint32_t a_src = smem_base + s * STAGE_BYTES;
          const uint32_t b_src = a_src + A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t adesc = p.adesc_hi | (uint64_t)(((a_src + k * p.a_kstep) & 0x3FFFFu) >> 4);
            const uint64_t bdesc = p.bdesc_hi | (uint64_t)(((b_src + k * p.b_kstep) & 0x3FFFFu) >> 4);
            umma_bf16(d_tmem, adesc, bdesc, p.idesc, (i > 0 || k > 0) ? 1u : 0u);
          }
          if (CLUSTER == 2) umma_commit_mc(empty_bar(s), (uint16_t)3);
          else umma_commit(empty_bar(s));
          if (i == nkb - 1) umma_commit(tfull_bar(acc));
        }
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue warps 2.. =====================
    // TMEM lane quarter = warp id mod 4 (hardware rule); with 8 epilogue warps the two warps of
    // a quarter split the tile's columns (more loads in flight for the fused optimiser)
    const int q = warp & 3;
    const int ew = warp - 2;
    constexpr int COLS_PER_WARP = BN / (EPI_WARPS / 4);
    const int col_lo = (ew >> 2) * COLS_PER_WARP;
    uint32_t tl = 0;
    for (int u = unit0; u < num_units; u += unit_step, ++tl) {
      const int m0 = unit_m0(u), n0 = unit_n0(u);
      const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
      mbar_wait(tfull_bar(acc), aph, 14);
      tcgen05_fence_after();
      const uint32_t t_row = tmem_acc + ((uint32_t)(q * 32) << 16) + acc * BN;
      if (m0 < p.epi.M) {  // (the odd row tile of a pair may lie wholly below the matrix)
#pragma unroll 1
        for (int c = col_lo; c < col_lo + COLS_PER_WARP; c += 32) {
          if (c >= p.bn_eff || n0 + c >= p.epi.N) break;  // warp-uniform
          uint32_t raw[32];
          tmem_ld32(t_row + (uint32_t)c, raw);
          tmem_ld_wait();
          if constexpr (RMS_DIRECT) rms_blocked_chunk(p.epi, lane, m0 + q * 32, n0 + c, raw);
          else epilogue_chunk<MATH>(p.epi, epi_stage + ew * (32 * EPI_LD), lane, m0 + q * 32, n0 + c, raw,
                                    (long long)unit_split(u) * p.partial_stride);
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  // no CTA may leave while its peer can still multicast into its smem / arrive on its barriers
  if (CLUSTER == 2) cluster_sync_all();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc),
                   "r"(TMEM_COLS)
                   : "memory");
  }
}

// Sum split-K partials and apply the epilogue.  One thread per (row, 32-col chunk).
// One thread per (row, 4 columns): consecutive lanes read consecutive float4 of a partial row
// (coalesced) and a 256 x 256 output still spreads over 128 CTAs -- with one thread per 32
// columns the narrow layers' 24-way split-K sums ran on 16 CTAs and cost more than their GEMMs.
__global__ void splitk_finalize_kernel(const EpiParams e, const float* __restrict__ partial,
                                       long long partial_ld, long long partial_stride, int splits) {
  const int groups = (e.N + 3) / 4;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)e.M * groups) return;
  const int r = (int)(idx / groups);
  const int c0 = (int)(idx % groups) * 4;
  const float* src = partial + (long long)r * partial_ld + c0;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  // eight partials' loads in flight, summed in split order (bit-reproducible): with one load
  // per iteration a 24-way sum was 24 dependent L2 round trips, ~12 us whatever the size
  for (int s0 = 0; s0 < splits; s0 += 8) {
    float4 q[8];
#pragma unroll
    for (int u = 0; u < 8; ++u)
      q[u] = (s0 + u < splits)
                 ? __ldcs(reinterpret_cast<const float4*>(src + (long long)(s0 + u) * partial_stride))
                 : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (s0 + u < splits) {
        a.x += q[u].x;
        a.y += q[u].y;
        a.z += q[u].z;
        a.w += q[u].w;
      }
    }
  }
  float v[4] = {a.x, a.y, a.z, a.w};
  const int ncols = min(4, e.N - c0);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float x = fmaf(v[j], e.alpha, (e.bias != nullptr && j < ncols) ? __ldg(e.bias + c0 + j) : 0.f);
    if (e.act == CC_ACT_SIGMOID) x = sigmoidf_(x);
    else if (e.act == CC_ACT_RELU) x = fmaxf(x, 0.f);
    v[j] = x;
  }
  if (e.dact != 0) {
    const bf16* yrow = e.dact_y + (long long)r * e.ld_dact + c0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j < ncols) {
        const float y = bf2f(yrow[j]);
        v[j] *= (e.dact == CC_ACT_SIGMOID) ? y * (1.f - y) : (y > 0.f ? 1.f : 0.f);
      }
    }
  }
  if (e.out32 != nullptr) {
    float* o = e.out32 + (long long)r * e.ld32 + c0;
    if (ncols == 4 && (((uintptr_t)o) & 15) == 0 && !e.beta32) {
      *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < ncols) o[j] = e.beta32 ? o[j] + v[j] : v[j];
    }
  }
  if (e.out16 != nullptr) {
    bf16* o = e.out16 + (long long)r * e.ld16 + c0;
    if (ncols == 4 && (((uintptr_t)o) & 7) == 0 && !e.beta16) {
      __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]);
      __nv_bfloat162 p1 = __floats2bfloat162_rn(v[2], v[3]);
      uint2 u;
      u.x = *reinterpret_cast<uint32_t*>(&p0);
      u.y = *reinterpret_cast<uint32_t*>(&p1);
      *reinterpret_cast<uint2*>(o) = u;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < ncols) o[j] = f2bf(e.beta16 ? bf2f(o[j]) + v[j] : v[j]);
    }
    if (e.out16_lo != nullptr) {
      bf16* l = e.out16_lo + (long long)r * e.ld16_lo + c0;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < ncols) l[j] = f2bf(v[j] - bf2f(f2bf(v[j])));
    }
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) ==
            cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)ptr;
  });
  return fn;
}

struct MapKey {
  const void* ptr;
  uint64_t inner, outer, ld;
  uint32_t box_inner, box_outer;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && inner == o.inner && outer == o.outer && ld == o.ld &&
           box_inner == o.box_inner && box_outer == o.box_outer;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = (uint64_t)(uintptr_t)k.ptr * 0x9E3779B97F4A7C15ull;
    h ^= k.inner + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    h ^= k.outer + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    h ^= k.ld + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    h ^= ((uint64_t)k.box_inner << 32 | k.box_outer) + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    return (size_t)h;
  }
};

// bf16 GEMM operand: row-major [outer, inner] tensor with leading dimension ld (elements),
// 128-byte swizzle
static int make_map(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t outer, uint64_t ld,
                    uint32_t box_inner, uint32_t box_outer) {
  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  MapKey key{ptr, inner, outer, ld, box_inner, box_outer};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return 0;
    }
  }
  PFN_encodeTiled enc = get_encode_fn();
  CC_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is unavailable (no CUDA driver?)");
  CC_REQUIRE(((uintptr_t)ptr & 15) == 0, "cc_gemm: operand base %p is not 16-byte aligned", ptr);
  CC_REQUIRE((ld * 2) % 16 == 0, "cc_gemm: operand ld=%llu is not a multiple of 16 bytes",
             (unsigned long long)ld);
  CC_REQUIRE(inner > 0 && outer > 0, "cc_gemm: empty operand");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CC_REQUIRE(r == CUDA_SUCCESS,
             "cuTensorMapEncodeTiled failed (%d) ptr=%p inner=%llu outer=%llu ld=%llu box=%ux%u",
             (int)r, ptr, (unsigned long long)inner, (unsigned long long)outer,
             (unsigned long long)ld, box_inner, box_outer);
  {
    std::lock_guard<std::mutex> g(mu);
    if (cache.size() > (1u << 16)) cache.clear();
    cache.emplace(key, *out);
  }
  return 0;
}

// smem matrix descriptor without the start address (cute::UMMA::SmemDescriptor):
//   [16,30) leading byte offset >>4, [32,46) stride byte offset >>4,
//   [46,48) version = 1, [61,64) layout type (2 = SWIZZLE_128B)
static uint64_t desc_hi(uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

// Test knobs, read from the environment ONCE (a GEMM launch should not cost getenv calls);
// cc_reload_env() re-reads them (tests change them at run time).  The first two force a choice
// the dispatcher otherwise makes from the shape, so that small shapes cover every choice; the
// third selects the reference that persistent split-K is compared with.
struct GemmEnv {
  int bn_eff;             // CC_GEMM_BN_EFF: effective tile width of the persistent kernel
  int rms_nfast;          // CC_GEMM_RMS_NFAST: raster of the fused-optimiser wgrad
  int persistent_splitk;  // CC_GEMM_PERSISTENT_SPLITK=0: split-K in the one-tile-per-CTA kernel
};
static GemmEnv g_env;
static std::atomic<int> g_env_state{0};   // 0: not loaded
static std::mutex g_env_mu;
static int g_num_sms = 0;

static const GemmEnv& gemm_env() {
  if (g_env_state.load(std::memory_order_acquire) == 0) {
    std::lock_guard<std::mutex> lock(g_env_mu);
    GemmEnv e;
    e.bn_eff = env_int("CC_GEMM_BN_EFF", 0);
    e.rms_nfast = env_int("CC_GEMM_RMS_NFAST", -1);
    e.persistent_splitk = env_int("CC_GEMM_PERSISTENT_SPLITK", 1);
    g_env = e;
    g_env_state.store(1, std::memory_order_release);
  }
  return g_env;
}

template <int BN, int STAGES>
static constexpr size_t smem_bytes() {
  return (size_t)STAGES * (BM * BK * 2 + BN * BK * 2) + 8 * (2 * STAGES + 2) + 1024;
}

template <int BN, int STAGES, bool A_MN, bool B_MN>
static int launch_cfg(const TmaMaps& maps, const GemmParams& p, dim3 grid, cudaStream_t st) {
  auto kern = gemm_tcgen05_kernel<BN, STAGES, A_MN, B_MN>;
  static bool attr_set = false;
  constexpr size_t smem = smem_bytes<BN, STAGES>();
  if (!attr_set) {
    CC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  kern<<<grid, 128, smem, st>>>(maps, p);
  CC_CHECK_LAUNCH();
  return 0;
}

template <int BN, int STAGES>
static int launch_major(const TmaMaps& maps, const GemmParams& p, dim3 grid, bool a_mn, bool b_mn,
                        cudaStream_t st) {
  if (!a_mn && b_mn) return launch_cfg<BN, STAGES, false, true>(maps, p, grid, st);
  if (!a_mn && !b_mn) return launch_cfg<BN, STAGES, false, false>(maps, p, grid, st);
  if (a_mn && b_mn) return launch_cfg<BN, STAGES, true, true>(maps, p, grid, st);
  return launch_cfg<BN, STAGES, true, false>(maps, p, grid, st);
}

template <int BN, int STAGES, int EPI_WARPS, bool RMS_DIRECT = false>
static constexpr size_t smem_bytes_persistent() {
  return (size_t)STAGES * (BM * BK * 2 + BN * BK * 2) + 8 * (2 * STAGES + 6) + 16 +
         (RMS_DIRECT ? 0 : EPI_WARPS * 32 * EPI_LD * 4) + 1024;   // no transpose tiles
}

template <int BN, int STAGES, bool A_MN, bool B_MN, bool MATH, int EPI_WARPS, bool N_FAST, int CLUSTER,
          bool RMS_DIRECT = false>
static int launch_persistent_one(const TmaMaps& maps, const GemmParams& p, int mt, int nt,
                                 int num_sms, cudaStream_t st) {
  auto kern = gemm_tcgen05_persistent_kernel<BN, STAGES, A_MN, B_MN, MATH, EPI_WARPS, N_FAST, CLUSTER,
                                             RMS_DIRECT>;
  static bool attr_set = false;
  static int max_ctas = 0;
  constexpr size_t smem = smem_bytes_persistent<BN, STAGES, EPI_WARPS, RMS_DIRECT>();
  static_assert(smem <= 232448, "shared memory per CTA");
  constexpr int threads = 64 + 32 * EPI_WARPS;
  if (!attr_set) {
    CC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    max_ctas = num_sms;
    if (CLUSTER > 1) {
      // co-resident clusters (an SM pair each); the persistent loop strides by the grid size
      cudaLaunchConfig_t q{};
      q.gridDim = dim3((unsigned)(num_sms / CLUSTER * CLUSTER));
      q.blockDim = dim3(threads);
      q.dynamicSmemBytes = smem;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = CLUSTER;
      qa[0].val.clusterDim.y = 1;
      qa[0].val.clusterDim.z = 1;
      q.attrs = qa;
      q.numAttrs = 1;
      int nclusters = 0;
      CC_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&nclusters, kern, &q));
      CC_REQUIRE(nclusters >= 1, "cc_gemm: no %d-CTA cluster fits on this device", CLUSTER);
      if (nclusters * CLUSTER < max_ctas) max_ctas = nclusters * CLUSTER;
    }
    attr_set = true;
  }
  const int units = ((mt + CLUSTER - 1) / CLUSTER) * nt * (p.psplits > 1 ? p.psplits : 1);
  int grid = units * CLUSTER < max_ctas ? units * CLUSTER : max_ctas / CLUSTER * CLUSTER;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CLUSTER;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p, mt, nt));
  count_launch();
  return 0;
}

template <int BN, int STAGES, bool A_MN, bool B_MN, bool MATH, int EPI_WARPS = 4, bool N_FAST = false>
static int launch_persistent_cfg(const TmaMaps& maps, const GemmParams& p, int mt, int nt,
                                 int num_sms, cudaStream_t st) {
  if (p.cluster == 2)
    return launch_persistent_one<BN, STAGES, A_MN, B_MN, MATH, EPI_WARPS, N_FAST, 2>(maps, p, mt, nt, num_sms, st);
  return launch_persistent_one<BN, STAGES, A_MN, B_MN, MATH, EPI_WARPS, N_FAST, 1>(maps, p, mt, nt, num_sms, st);
}

template <int BN, int STAGES, bool MATH>
static int launch_persistent_m(const TmaMaps& maps, const GemmParams& p, int mt, int nt,
                               int num_sms, bool a_mn, bool b_mn, cudaStream_t st) {
  if (!a_mn && b_mn) return launch_persistent_cfg<BN, STAGES, false, true, MATH>(maps, p, mt, nt, num_sms, st);
  if (!a_mn && !b_mn) return launch_persistent_cfg<BN, STAGES, false, false, MATH>(maps, p, mt, nt, num_sms, st);
  if (a_mn && b_mn) return launch_persistent_cfg<BN, STAGES, true, true, MATH>(maps, p, mt, nt, num_sms, st);
  return launch_persistent_cfg<BN, STAGES, true, false, MATH>(maps, p, mt, nt, num_sms, st);
}

template <int BN, int STAGES>
static int launch_persistent(const TmaMaps& maps, const GemmParams& p, int mt, int nt, int num_sms,
                             bool a_mn, bool b_mn, cudaStream_t st) {
  const EpiParams& e = p.epi;
  const bool math = e.alpha != 1.f || e.bias != nullptr || e.act != 0 || e.dact != 0;
  if (math) return launch_persistent_m<BN, STAGES, true>(maps, p, mt, nt, num_sms, a_mn, b_mn, st);
  return launch_persistent_m<BN, STAGES, false>(maps, p, mt, nt, num_sms, a_mn, b_mn, st);
}

int gemm_impl(const cc_gemm_desc* d, cudaStream_t st) {
  const GemmEnv& ENV = gemm_env();
  CC_REQUIRE(d != nullptr, "cc_gemm: null descriptor");
  CC_REQUIRE(d->M > 0 && d->N > 0, "cc_gemm: empty output %dx%d", d->M, d->N);
  CC_REQUIRE(d->nseg >= 1 && d->nseg <= MAX_SEG, "cc_gemm: nseg=%d out of range", d->nseg);
  CC_REQUIRE(d->out16 != nullptr || d->out32 != nullptr || d->rms_p32 != nullptr,
             "cc_gemm: no output");
  CC_REQUIRE(d->rms_p32 == nullptr || (d->rms_ms != nullptr && d->rms_mom != nullptr),
             "cc_gemm: fused RMSprop needs ms and mom");
  CC_REQUIRE(d->route_world >= 0 && d->route_world <= CC_PEER_MAX, "cc_gemm: route_world=%d",
             d->route_world);
  CC_REQUIRE(d->out16_lo == nullptr || (d->out16 != nullptr && d->beta16 == 0),
             "cc_gemm: out16_lo needs a plain out16 (the high-order term)");
  if (d->rms_blocked) {
    CC_REQUIRE(d->rms_p32 != nullptr && d->a_mn_major && d->b_mn_major && d->N > 128 &&
                   d->alpha == 1.f && d->bias == nullptr && d->act == 0 && d->dact_y == nullptr &&
                   d->out16 == nullptr && d->beta32 == 0 && d->route_world == 0 &&
                   d->force_splits <= 1 && (d->force_bn == 0 || d->force_bn == 256),
               "cc_gemm: rms_blocked is for plain weight-gradient GEMMs (X^T dZ, N > 128)");
    // the bf16 copies and out32 are written in whole 32-column chunks (zeros past N), so their
    // rows must be at least round_up(N, 32) long or a chunk spills into the next row
    const long long n32 = ((long long)d->N + 31) / 32 * 32;
    CC_REQUIRE(d->rms_row0 >= 0 && (d->rms_ld & 31) == 0 && d->rms_ld >= n32 &&
                   ((((uintptr_t)d->rms_p32) | ((uintptr_t)d->rms_ms) | ((uintptr_t)d->rms_mom) |
                     ((uintptr_t)d->rms_p16) | ((uintptr_t)d->rms_p16_lo) | ((uintptr_t)d->out32)) & 15) == 0 &&
                   (d->out32 == nullptr || ((d->ld32 & 3) == 0 && d->ld32 >= n32)),
               "cc_gemm: rms_blocked needs 16-byte aligned blocks, rms_ld %% 32 == 0 and rms_ld, "
               "ld32 >= round_up(N, 32) (N=%d rms_ld=%lld ld32=%lld)",
               d->N, (long long)d->rms_ld, (long long)d->ld32);
  }
  CC_REQUIRE(d->rms_p16_lo == nullptr || d->rms_blocked,
             "cc_gemm: rms_p16_lo is written by the blocked fused-optimiser epilogue only");
  if (d->route_world > 0) {
    CC_REQUIRE(d->out32 != nullptr && d->beta32 == 0 && d->workspace == nullptr &&
                   d->rms_p32 == nullptr,
               "cc_gemm: a routed output needs a plain fp32 output without split-K");
    CC_REQUIRE(d->route_shard > 0 && (d->route_shard & 7) == 0 && d->route_shard < (1ll << 32) &&
                   d->route_off0 >= 0 && (d->route_off0 & 3) == 0,
               "cc_gemm: route_shard=%lld route_off0=%lld", (long long)d->route_shard,
               (long long)d->route_off0);
    for (int q = 0; q < d->route_world; ++q)
      CC_REQUIRE(d->route_base[q] != nullptr && ((uintptr_t)d->route_base[q] & 15) == 0,
                 "cc_gemm: route_base[%d]=%p is null or not 16-byte aligned", q,
                 (const void*)d->route_base[q]);
  }
  if (g_num_sms == 0) {
    int dev = 0;
    CC_CHECK_CUDA(cudaGetDevice(&dev));
    CC_CHECK_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const bool a_mn = d->a_mn_major != 0, b_mn = d->b_mn_major != 0;

  const int bn = d->force_bn ? d->force_bn : (d->N > 128 ? 256 : 128);
  CC_REQUIRE(bn == 128 || bn == 256, "cc_gemm: BN=%d unsupported", bn);

  GemmParams p{};
  TmaMaps maps;
  memset(&maps, 0, sizeof(maps));
  p.nseg = d->nseg;
  int total = 0;
  for (int s = 0; s < d->nseg; ++s) {
    CC_REQUIRE(d->k[s] > 0, "cc_gemm: segment %d has k=%d", s, d->k[s]);
    p.kblocks[s] = (d->k[s] + BK - 1) / BK;
    total += p.kblocks[s];
  }
  p.total_kblocks = total;

  const int mt = (d->M + BM - 1) / BM;
  int nt = (d->N + bn - 1) / bn;
  // split-K when the tile grid cannot fill the machine and the reduction is long
  int splits = 1;
  const long long Mpad = (long long)mt * BM, Npad = (long long)nt * bn;
  if (d->workspace != nullptr && d->rms_p32 == nullptr) {
    int want = d->force_splits;
    if (want == 0) {
      // split-K only when the tile grid leaves more than half of the SMs idle (small batch,
      // long reduction: the weight-streaming regime of the reference's batch 128); otherwise
      // the persistent kernel runs the tiles unsplit
      const int tiles = mt * nt;
      if (2 * tiles <= g_num_sms && total >= 8) {
        // as many splits as keep every CTA in ONE co-resident wave (2 CTAs per SM): rounding up
        // here put 4-8 % of the CTAs into a second wave and nearly doubled the launch time of
        // the weight-streaming GEMMs (Dx1 forward at batch 128: 40 tiles x 8 splits = 320 CTAs
        // on 296 slots)
        want = (2 * g_num_sms) / tiles;
        if (want < 1) want = 1;
        if (want > total / 4) want = total / 4;
      } else {
        want = 1;
      }
    }
    if (want > total) want = total;
    const long long cap = d->workspace_elems / (Mpad * Npad);
    if (want > cap) want = (int)cap;
    if (want >= 2) splits = want;
  }
  p.kb_per_split = (total + splits - 1) / splits;
  splits = (total + p.kb_per_split - 1) / p.kb_per_split;  // no empty split
  if (splits >= 2) {
    p.partial = d->workspace;
    p.partial_ld = Npad;
    p.partial_stride = Mpad * Npad;
  } else {
    p.partial = nullptr;
    p.kb_per_split = total;
    splits = 1;
  }
  // split-K inside the persistent kernel (work unit = tile x k-range): the operand ring and the
  // TMEM double buffer keep running across units, where the one-tile-per-CTA kernel runs one
  // wave of short-lived CTAs whose prologues and partial-tile stores all coincide.  The
  // one-tile-per-CTA kernel stays as the reference it is tested against.
  const bool persistent = splits == 1 || ENV.persistent_splitk != 0;

  // 2-CTA clusters (B tile multicast) whenever there are at least two row tiles
  // (fused optimiser: only when the batch reduction is long enough for the shared B tile to
  // matter -- at the reference's batch 128 the epilogue is everything and coupling two CTAs'
  // operand rings only costs, profiles/r02_fused_rmsprop_blocked_state.jsonl)
  p.cluster = (persistent && mt >= 2 && (d->rms_p32 == nullptr || total > 8)) ? 2 : 1;
  // effective tile width of the persistent kernel: the candidate that minimises
  // waves x (per-tile cost); e.g. N = 3369 at batch 2048 is 224 tiles of 256 (1.51 waves on 148
  // SMs -> 2) but 288 tiles of 192 (1.95 waves -> 2, each shorter).  The per-tile cost model is
  // operand bytes (A is fixed, B scales with the width): the kernels are L2->SM bound.
  int bn_eff = bn;
  if (persistent && bn == 256 && d->rms_p32 == nullptr && splits == 1) {
    const int forced = ENV.bn_eff;
    if (forced >= 32 && forced <= 256 && forced % 32 == 0) {
      bn_eff = forced;
    } else {
      long long best = -1;
      const int mu = (mt + p.cluster - 1) / p.cluster, slots = g_num_sms / p.cluster;
      for (int cand = 256; cand >= 128; cand -= 64) {
        const long long units = (long long)mu * ((d->N + cand - 1) / cand);
        const long long cost = ((units + slots - 1) / slots) * (cand + 128);
        if (best < 0 || cost < best) {
          best = cost;
          bn_eff = cand;
        }
      }
    }
    nt = (d->N + bn_eff - 1) / bn_eff;
  }
  p.bn_eff = bn_eff;
  p.b_boxes = (bn_eff + 63) / 64;
  p.b_half_rows = bn_eff / 2;
  p.stage_tx = (unsigned)(BM * BK * 2 + (b_mn ? p.b_boxes * 64 * BK * 2 : bn_eff * BK * 2));

  for (int s = 0; s < d->nseg; ++s) {
    int rc;
    if (a_mn)  // stored [K, M]
      rc = make_map(&maps.a[s], d->a[s], (uint64_t)d->M, (uint64_t)d->k[s], (uint64_t)d->lda[s], 64, BK);
    else  // stored [M, K]
      rc = make_map(&maps.a[s], d->a[s], (uint64_t)d->k[s], (uint64_t)d->M, (uint64_t)d->lda[s], BK, BM);
    if (rc) return rc;
    if (b_mn)  // stored [K, N]
      rc = make_map(&maps.b[s], d->b[s], (uint64_t)d->N, (uint64_t)d->k[s], (uint64_t)d->ldb[s], 64, BK);
    else  // stored [N, K]
      rc = make_map(&maps.b[s], d->b[s], (uint64_t)d->k[s], (uint64_t)d->N, (uint64_t)d->ldb[s], BK,
                    (uint32_t)(persistent ? (p.cluster == 2 ? bn_eff / 2 : bn_eff) : bn));
    if (rc) return rc;
  }

  // UMMA descriptors.  K-major, 128B swizzle: 8-row groups 1024 B apart (SBO), LBO unused (=16B),
  // K advance = 32 B inside the swizzle row.  MN-major, 128B swizzle: 64-element MN atoms are
  // separate TMA boxes 64*BK*2 = 8192 B apart (LBO), 8-k groups 1024 B apart (SBO), K advance =
  // 16 rows * 128 B.
  const uint64_t mn_desc = desc_hi(64 * BK * 2, 1024), k_desc = desc_hi(16, 1024);
  const uint32_t mn_kstep = UMMA_K * 128, k_kstep = UMMA_K * 2;
  p.adesc_hi = a_mn ? mn_desc : k_desc;
  p.bdesc_hi = b_mn ? mn_desc : k_desc;
  p.a_kstep = a_mn ? mn_kstep : k_kstep;
  p.b_kstep = b_mn ? mn_kstep : k_kstep;
  // cute::UMMA::InstrDescriptor: c_format F32 (1<<4), a/b format BF16 (1<<7, 1<<10),
  // a_major bit 15, b_major bit 16, N>>3 at [17,23), M>>4 at [24,29)
  p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) |
            ((b_mn ? 1u : 0u) << 16) | ((uint32_t)((persistent ? bn_eff : bn) >> 3) << 17) |
            ((uint32_t)(BM >> 4) << 24);

  EpiParams& e = p.epi;
  e.M = d->M;
  e.N = d->N;
  e.alpha = d->alpha;
  e.bias = d->bias;
  e.act = d->act;
  e.dact_y = (const bf16*)d->dact_y;
  e.ld_dact = d->ld_dact;
  e.dact = d->dact_y ? d->dact : 0;
  e.out16 = (bf16*)d->out16;
  e.ld16 = d->ld16;
  e.beta16 = d->beta16;
  e.out16_lo = (bf16*)d->out16_lo;
  e.ld16_lo = d->ld16_lo;
  e.out32 = d->out32;
  e.ld32 = d->ld32;
  e.beta32 = d->beta32;
  e.rms_p32 = d->rms_p32;
  e.rms_ms = d->rms_ms;
  e.rms_mom = d->rms_mom;
  e.rms_p16 = (bf16*)d->rms_p16;
  e.rms_ld = d->rms_ld;
  e.rms_lr = d->rms_lr;
  e.rms_rho = d->rms_rho;
  e.rms_momentum = d->rms_momentum;
  e.rms_eps = d->rms_eps;
  e.rms_blocked = d->rms_blocked;
  e.rms_row0 = d->rms_row0;
  e.rms_p16lo = d->rms_blocked ? (bf16*)d->rms_p16_lo : nullptr;
  e.route_world = d->route_world;
  e.route_shard = (unsigned)d->route_shard;
  e.route_off0 = d->route_off0;
  for (int q = 0; q < CC_PEER_MAX; ++q)
    e.route_base[q] = q < d->route_world ? d->route_base[q] : nullptr;

  if (persistent) {
    // fused optimiser on weight gradients (both operands MN-major, no epilogue math): the
    // epilogue streams 26 B per element, so it gets 8 warps (twice the loads in flight) and
    // the main loop one stage less
    if (bn == 256 && d->rms_p32 != nullptr && a_mn && b_mn && d->alpha == 1.f &&
        d->bias == nullptr && d->act == 0 && e.dact == 0) {
      // raster: walk along N (DRAM-page-local optimiser stream) when the whole B operand
      // (dZ, batch x N) stays L2-resident across row blocks; otherwise keep m fastest so the
      // CTAs of a wave share one B tile and A (X^T) is the L2-resident operand
      int nfast = ENV.rms_nfast;
      if (nfast < 0) nfast = ((long long)total * BK * d->N * 2 <= (48ll << 20)) ? 1 : 0;
      if (d->rms_blocked) {
        // blocked optimiser state: accumulators go straight from TMEM registers to 4 KB state
        // blocks (rms_blocked_chunk), no transpose tiles -> four operand stages
        if (p.cluster == 2)
          return nfast ? launch_persistent_one<256, 4, true, true, false, 8, true, 2, true>(
                             maps, p, mt, nt, g_num_sms, st)
                       : launch_persistent_one<256, 4, true, true, false, 8, false, 2, true>(
                             maps, p, mt, nt, g_num_sms, st);
        return nfast ? launch_persistent_one<256, 4, true, true, false, 8, true, 1, true>(
                           maps, p, mt, nt, g_num_sms, st)
                     : launch_persistent_one<256, 4, true, true, false, 8, false, 1, true>(
                           maps, p, mt, nt, g_num_sms, st);
      }
      if (nfast != 0)
        return launch_persistent_cfg<256, 3, true, true, false, 8, true>(maps, p, mt, nt, g_num_sms, st);
      return launch_persistent_cfg<256, 3, true, true, false, 8>(maps, p, mt, nt, g_num_sms, st);
    }
    if (splits >= 2) {
      // k-ranges of a tile go to fp32 partials (raw accumulators, no epilogue math); the
      // finalize kernel sums them in split order and applies the real epilogue
      CC_REQUIRE(d->rms_p32 == nullptr, "cc_gemm: fused RMSprop is not available with split-K");
      GemmParams pp = p;
      pp.psplits = splits;
      EpiParams pe{};
      pe.M = d->M;
      pe.N = d->N;
      pe.alpha = 1.f;
      pe.out32 = p.partial;
      pe.ld32 = p.partial_ld;
      pp.epi = pe;
      int rc = bn == 256
                   ? launch_persistent_m<256, 4, false>(maps, pp, mt, nt, g_num_sms, a_mn, b_mn, st)
                   : launch_persistent_m<128, 6, false>(maps, pp, mt, nt, g_num_sms, a_mn, b_mn, st);
      if (rc) return rc;
      const long long work = (long long)d->M * ((d->N + 3) / 4);
      const int threads = 256;
      splitk_finalize_kernel<<<(unsigned)((work + threads - 1) / threads), threads, 0, st>>>(
          p.epi, p.partial, p.partial_ld, p.partial_stride, splits);
      CC_CHECK_LAUNCH();
      return 0;
    }
    if (bn == 256) return launch_persistent<256, 4>(maps, p, mt, nt, g_num_sms, a_mn, b_mn, st);
    return launch_persistent<128, 6>(maps, p, mt, nt, g_num_sms, a_mn, b_mn, st);
  }
  CC_REQUIRE(d->rms_p32 == nullptr, "cc_gemm: fused RMSprop is not available with split-K");

  dim3 grid((unsigned)nt, (unsigned)mt, (unsigned)splits);
  int rc;
  if (bn == 256)
    rc = launch_major<256, 2>(maps, p, grid, a_mn, b_mn, st);
  else
    rc = launch_major<128, 3>(maps, p, grid, a_mn, b_mn, st);
  if (rc) return rc;
  if (splits >= 2) {
    const long long work = (long long)d->M * ((d->N + 3) / 4);
    const int threads = 256;
    splitk_finalize_kernel<<<(unsigned)((work + threads - 1) / threads), threads, 0, st>>>(
        p.epi, p.partial, p.partial_ld, p.partial_stride, splits);
    CC_CHECK_LAUNCH();
  }
  return 0;
}

}  // namespace cc

extern "C" void cc_reload_env(void) {
  std::lock_guard<std::mutex> lock(cc::g_env_mu);
  cc::g_env_state.store(0, std::memory_order_release);
  cc::g_num_sms = 0;
}

extern "C" int cc_gemm(const cc_gemm_desc* desc, cc_stream_t stream) {
  return cc::gemm_impl(desc, (cudaStream_t)stream);
}

extern "C" int64_t cc_gemm_workspace_elems(int32_t M, int32_t N) {
  // room for up to 2*148 CTAs' worth of 128x256 fp32 partial tiles, or 8 splits of the padded
  // output, whichever is larger
  const long long Mpad = ((long long)M + 127) / 128 * 128, Npad = ((long long)N + 255) / 256 * 256;
  long long a = 296LL * 128 * 256 * 2;
  long long b = 8 * Mpad * Npad;
  return a > b ? a : b;
}
