// The two-sample pass (ClassifyCellBiGan.two_sample_test): log1p features of cells and the
// kernel sums of an MMD permutation test.
//
// cc_log1p_features: per row of a dense fp32 tile, f(v) = bf16_rn(float(log1p(double(v)))) per
// gene (v optionally rint first), written row-major with the padding up to the next multiple of
// 64 columns zeroed, so the output is a ready GEMM operand; plus the row's library size sum v
// (fp64) and genes detected #{v != 0}.  One CTA of 256 threads per row, float4 loads where the
// layout allows; nothing at or past `cols` is read.  Most counts are 0 (the bits of v itself, so
// -0.0 stays -0.0) or small integers (a 256-entry shared table built with the same formula), so
// fp64 log1p runs only for the rest.  The row sums combine in a fixed tree: identical bits every
// run, and exact on integer counts.
//
// cc_mmd_sums: for the fp32 Gram matrix G of N cells, every inverse bandwidth g_b and every
// labelling p (a bitmask over the cells, bit set = the cell is in X), the sums over ordered pairs
// i != j of k_b(i, j) = exp(-d2 g_b), d2 = max((G_ii + G_jj) - 2 G_ij, 0) (no FMA contraction):
//   XX (both in X), YY (both in Y), XY (i in X, j in Y).
// Only upper-triangle 64 x 64 tiles of G are read, and only elements i < j.  A thread holds 32
// elements of one tile row (one mask word of columns) times the bandwidths in registers and loops
// over all labellings: x_b = sum over set column bits of k_b, then per tile
//   X_b += b_i x_b          (= sum_{i<j} k b_i b_j)
//   A_b += x_b + b_i r_b    (= sum_{i<j} k (b_i + b_j), r_b the thread's row sum)
// and a labelling-independent total S_b = sum_{i<j} k.  With R = A, XX = 2X, XY = R - XX and
// YY = 2S - 2R + XX.  Thread partials are fp32 (32 terms), everything above them fp64.
// Deterministic: a fixed grid of CTAs (a function of N alone) walks the tiles in a fixed order,
// each CTA owns one row of the workspace, and a second launch sums the rows in CTA order.  No
// float atomics.
#include "common.cuh"

namespace cc {

// ------------------------------------------------------------------ log1p features
__device__ __forceinline__ uint16_t bf16_bits_rn(float f) {
  const uint32_t u = __float_as_uint(f);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40u);  // quiet NaN
  return (uint16_t)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);                 // round half even
}

__device__ __forceinline__ uint16_t log1p_bf16(double v) { return bf16_bits_rn((float)log1p(v)); }

constexpr int kFeatThreads = 256;
constexpr int kFeatUnroll = 4;   // float4 loads in flight per thread

template <bool VEC, bool ROUND>
__global__ void __launch_bounds__(kFeatThreads)
log1p_features_kernel(const float* __restrict__ x, long long ldx, long long cols,
                      uint16_t* __restrict__ f, long long ldf, double* __restrict__ lib,
                      int* __restrict__ det) {
  __shared__ uint16_t table[256];
  __shared__ double slib[kFeatThreads];
  __shared__ int sdet[kFeatThreads];
  const int t = threadIdx.x;
  table[t] = log1p_bf16((double)t);
  __syncthreads();
  const long long row = blockIdx.x;
  const float* xr = x + row * ldx;
  uint16_t* fr = f + row * ldf;
  const long long pad = (cols + 63) / 64 * 64;
  double s = 0.0;
  int n = 0;
  auto load = [&](long long c) {
    if (VEC && c + 3 < cols) return *reinterpret_cast<const float4*>(xr + c);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c + 0 < cols) v.x = xr[c + 0];
    if (c + 1 < cols) v.y = xr[c + 1];
    if (c + 2 < cols) v.z = xr[c + 2];
    if (c + 3 < cols) v.w = xr[c + 3];
    return v;
  };
  auto consume = [&](long long c, float4 v4) {
    const float in[4] = {v4.x, v4.y, v4.z, v4.w};
    uint16_t o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      o[e] = 0;
      if (c + e < cols) {
        const float y = ROUND ? rintf(in[e]) : in[e];
        s += (double)y;
        n += y != 0.f;
        if (y == 0.f) o[e] = (uint16_t)(__float_as_uint(y) >> 16);      // +-0 -> +-0
        else if (y > 0.f && y < 256.f && y == truncf(y)) o[e] = table[(int)y];
        else o[e] = log1p_bf16((double)y);
      }
    }
    *reinterpret_cast<uint2*>(fr + c) =
        make_uint2((uint32_t)o[0] | ((uint32_t)o[1] << 16), (uint32_t)o[2] | ((uint32_t)o[3] << 16));
  };
  constexpr long long kStep = 4ll * kFeatThreads;
  long long c = 4ll * t;
  for (; c + kStep * (kFeatUnroll - 1) < pad; c += kStep * kFeatUnroll) {
    float4 v[kFeatUnroll];
#pragma unroll
    for (int u = 0; u < kFeatUnroll; ++u) v[u] = load(c + kStep * u);
#pragma unroll
    for (int u = 0; u < kFeatUnroll; ++u) consume(c + kStep * u, v[u]);
  }
  for (; c < pad; c += kStep) consume(c, load(c));
  slib[t] = s;
  sdet[t] = n;
  __syncthreads();
  for (int w = kFeatThreads / 2; w > 0; w >>= 1) {   // fixed tree
    if (t < w) {
      slib[t] += slib[t + w];
      sdet[t] += sdet[t + w];
    }
    __syncthreads();
  }
  if (t == 0) {
    lib[row] = slib[0];
    det[row] = sdet[0];
  }
}

// ------------------------------------------------------------------ MMD sums
constexpr int kMmdTile = 64;
constexpr int kMmdThreads = 128;   // two threads per tile row, 32 columns (one mask word) each
constexpr int kMmdChunk = 8;       // labellings per shared-memory reduction
constexpr int kMmdMaxCtas = 592;   // fixed, not the device's SM count: the bits depend on N only
constexpr int kMmdMaxBw = 4;

struct MmdBw {
  float g[kMmdMaxBw];
};

static long long mmd_tiles(long long n) {
  const long long T = (n + kMmdTile - 1) / kMmdTile;
  return T * (T + 1) / 2;
}

static long long mmd_ctas(long long n) { return std::min<long long>(kMmdMaxCtas, mmd_tiles(n)); }

template <int NB>
__global__ void __launch_bounds__(kMmdThreads)
mmd_tiles_kernel(const float* __restrict__ G, long long ld, long long N, MmdBw bw,
                 const uint32_t* __restrict__ masks, long long W, long long L,
                 double* __restrict__ part, long long part_ld) {
  __shared__ float sdr[kMmdTile], sdc[kMmdTile];
  __shared__ float red[kMmdChunk][2 * NB][kMmdThreads];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int r = t >> 1, h = t & 1;
  double* my = part + (long long)blockIdx.x * part_ld;
  for (long long v = t; v < part_ld; v += kMmdThreads) my[v] = 0.0;
  double s_acc[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) s_acc[b] = 0.0;
  const long long T = (N + kMmdTile - 1) / kMmdTile;
  const long long ntiles = T * (T + 1) / 2;
  long long ti = 0, rem = blockIdx.x;      // tile index -> (ti, tj = ti + rem), row-major
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, rem += gridDim.x) {
    while (rem >= T - ti) {
      rem -= T - ti;
      ++ti;
    }
    const long long tj = ti + rem;
    __syncthreads();   // the previous tile is done with sdr / sdc / red, `my` is zeroed
    if (t < kMmdTile) {
      const long long i = ti * kMmdTile + t;
      sdr[t] = i < N ? G[i * ld + i] : 0.f;
    } else {
      const long long j = tj * kMmdTile + t - kMmdTile;
      sdc[t - kMmdTile] = j < N ? G[j * ld + j] : 0.f;
    }
    __syncthreads();
    const long long i = ti * kMmdTile + r;
    const long long j0 = tj * kMmdTile + 32 * h;
    const bool live = i < N && j0 < N;
    float k[NB][32];
    float rs[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) rs[b] = 0.f;
    {
      float g[32];
      const float* gr = G + (live ? i * ld + j0 : 0);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live && j0 + 4 * q + 3 < N) {
          v = *reinterpret_cast<const float4*>(gr + 4 * q);
        } else if (live) {
          if (j0 + 4 * q + 0 < N) v.x = gr[4 * q + 0];
          if (j0 + 4 * q + 1 < N) v.y = gr[4 * q + 1];
          if (j0 + 4 * q + 2 < N) v.z = gr[4 * q + 2];
        }
        g[4 * q + 0] = v.x;
        g[4 * q + 1] = v.y;
        g[4 * q + 2] = v.z;
        g[4 * q + 3] = v.w;
      }
      const float gi = sdr[r];
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const long long j = j0 + e;
        const bool valid = live && j < N && j > i;
        const float d2 =
            fmaxf(__fsub_rn(__fadd_rn(gi, sdc[32 * h + e]), __fmul_rn(2.f, g[e])), 0.f);
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          k[b][e] = valid ? expf(-__fmul_rn(d2, bw.g[b])) : 0.f;
          rs[b] += k[b][e];
        }
      }
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) s_acc[b] += (double)rs[b];
    const uint32_t* mrow = masks + (live ? (i >> 5) : 0);
    const uint32_t* mcol = masks + (live ? (j0 >> 5) : 0);
    const int ibit = (int)(i & 31);
    for (long long p0 = 0; p0 < L; p0 += kMmdChunk) {
#pragma unroll 1
      for (int c = 0; c < kMmdChunk; ++c) {
        const long long p = p0 + c;
        float x[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) x[b] = 0.f;
        bool bi = false;
        if (live && p < L) {
          const uint32_t w = __ldg(mcol + p * W);
          bi = (__ldg(mrow + p * W) >> ibit) & 1u;
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            if (w & (1u << e)) {
#pragma unroll
              for (int b = 0; b < NB; ++b) x[b] += k[b][e];
            }
          }
        }
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          red[c][b][t] = bi ? x[b] : 0.f;
          red[c][NB + b][t] = bi ? x[b] + rs[b] : x[b];
        }
      }
      __syncthreads();
      for (int row = warp; row < kMmdChunk * 2 * NB; row += kMmdThreads / 32) {
        const int c = row / (2 * NB), v = row % (2 * NB);
        double a = (double)red[c][v][lane] + (double)red[c][v][lane + 32];
        a += (double)red[c][v][lane + 64] + (double)red[c][v][lane + 96];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0 && p0 + c < L) my[(p0 + c) * 2 * NB + v] += a;
      }
      __syncthreads();
    }
  }
  // the labelling-independent total: fixed-order block reduction of the per-thread sums
  __shared__ double ss[NB][kMmdThreads];
#pragma unroll
  for (int b = 0; b < NB; ++b) ss[b][t] = s_acc[b];
  __syncthreads();
  for (int w = kMmdThreads / 2; w > 0; w >>= 1) {
    if (t < w) {
#pragma unroll
      for (int b = 0; b < NB; ++b) ss[b][t] += ss[b][t + w];
    }
    __syncthreads();
  }
  if (t < NB) my[L * 2 * NB + t] = ss[t][0];
}

__global__ void mmd_finish_kernel(const double* __restrict__ part, long long part_ld, int ctas,
                                  int nb, long long L, double* __restrict__ out) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= L * nb) return;
  const long long p = q / nb;
  const int b = (int)(q % nb);
  double X = 0.0, A = 0.0, S = 0.0;
  for (int c = 0; c < ctas; ++c) {   // CTA order: fixed
    const double* row = part + (long long)c * part_ld;
    X += row[p * 2 * nb + b];
    A += row[p * 2 * nb + nb + b];
    S += row[L * 2 * nb + b];
  }
  const double xx = 2.0 * X;
  out[q * 3 + 0] = xx;
  out[q * 3 + 1] = 2.0 * S - 2.0 * A + xx;
  out[q * 3 + 2] = A - xx;
}

}  // namespace cc

extern "C" int cc_log1p_features(const float* x, int64_t ldx, int64_t rows, int64_t cols,
                                 int32_t round_half_even, void* features, int64_t ldf,
                                 double* library_size, int32_t* genes_detected,
                                 cc_stream_t stream) {
  using namespace cc;
  CC_REQUIRE(rows >= 0 && cols >= 0, "cc_log1p_features: rows %lld / cols %lld < 0",
             (long long)rows, (long long)cols);
  CC_REQUIRE(ldx >= cols, "cc_log1p_features: ldx %lld < cols %lld", (long long)ldx,
             (long long)cols);
  const long long pad = (cols + 63) / 64 * 64;
  CC_REQUIRE(ldf >= pad && ldf % 8 == 0, "cc_log1p_features: ldf %lld must be a multiple of 8 "
             "and at least %lld (cols rounded up to 64)", (long long)ldf, pad);
  CC_REQUIRE(rows <= 0x7fffffffll, "cc_log1p_features: %lld rows", (long long)rows);
  if (rows == 0) return 0;
  CC_REQUIRE(x != nullptr && features != nullptr && library_size != nullptr &&
             genes_detected != nullptr, "cc_log1p_features: null pointer");
  CC_REQUIRE((((uintptr_t)features) & 15) == 0,
             "cc_log1p_features: features must be 16-byte aligned");
  if (cols == 0) {
    CC_CHECK_CUDA(cudaMemsetAsync(library_size, 0, rows * sizeof(double), (cudaStream_t)stream));
    CC_CHECK_CUDA(cudaMemsetAsync(genes_detected, 0, rows * sizeof(int32_t),
                                  (cudaStream_t)stream));
    return 0;
  }
  const bool vec = ldx % 4 == 0 && (((uintptr_t)x) & 15) == 0;
  uint16_t* f = static_cast<uint16_t*>(features);
  int* det = reinterpret_cast<int*>(genes_detected);
  cudaStream_t st = (cudaStream_t)stream;
#define CC_FEAT_LAUNCH(V, R)                                                                  \
  log1p_features_kernel<V, R><<<(unsigned)rows, kFeatThreads, 0, st>>>(x, ldx, cols, f, ldf, \
                                                                       library_size, det)
  if (vec && round_half_even) CC_FEAT_LAUNCH(true, true);
  else if (vec) CC_FEAT_LAUNCH(true, false);
  else if (round_half_even) CC_FEAT_LAUNCH(false, true);
  else CC_FEAT_LAUNCH(false, false);
#undef CC_FEAT_LAUNCH
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int64_t cc_mmd_sums_ws_bytes(int64_t n_cells, int32_t n_bandwidths,
                                        int64_t labellings) {
  using namespace cc;
  if (n_cells < 2 || n_bandwidths < 1 || labellings < 1) return 0;
  const long long part_ld = labellings * 2 * n_bandwidths + n_bandwidths;
  return mmd_ctas(n_cells) * part_ld * (long long)sizeof(double);
}

extern "C" int cc_mmd_sums(const float* gram, int64_t ldg, int64_t n_cells,
                           const float* inv_bandwidths, int32_t n_bandwidths,
                           const uint32_t* masks, int64_t labellings, double* sums, void* ws,
                           int64_t ws_bytes, cc_stream_t stream) {
  using namespace cc;
  CC_REQUIRE(n_cells >= 0 && labellings >= 0, "cc_mmd_sums: n_cells %lld / labellings %lld < 0",
             (long long)n_cells, (long long)labellings);
  CC_REQUIRE(n_bandwidths >= 1 && n_bandwidths <= kMmdMaxBw,
             "cc_mmd_sums: %d bandwidths (1 to %d)", (int)n_bandwidths, kMmdMaxBw);
  CC_REQUIRE(ldg >= n_cells && ldg % 4 == 0, "cc_mmd_sums: ldg %lld must be a multiple of 4 and "
             "at least n_cells %lld", (long long)ldg, (long long)n_cells);
  if (labellings == 0) return 0;
  CC_REQUIRE(sums != nullptr && inv_bandwidths != nullptr, "cc_mmd_sums: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_cells < 2) {   // no pairs
    CC_CHECK_CUDA(cudaMemsetAsync(sums, 0, labellings * n_bandwidths * 3 * sizeof(double), st));
    return 0;
  }
  CC_REQUIRE(gram != nullptr && masks != nullptr, "cc_mmd_sums: null pointer");
  CC_REQUIRE((((uintptr_t)gram) & 15) == 0, "cc_mmd_sums: gram must be 16-byte aligned");
  const long long need = cc_mmd_sums_ws_bytes(n_cells, n_bandwidths, labellings);
  CC_REQUIRE(ws_bytes >= need && ws != nullptr,
             "cc_mmd_sums of %lld cells, %lld labellings: workspace of %lld bytes, needs %lld "
             "(cc_mmd_sums_ws_bytes)", (long long)n_cells, (long long)labellings,
             (long long)(ws == nullptr ? 0 : ws_bytes), need);
  MmdBw bw{};
  for (int b = 0; b < n_bandwidths; ++b) bw.g[b] = inv_bandwidths[b];
  const long long W = (n_cells + 31) / 32;
  const long long part_ld = labellings * 2 * n_bandwidths + n_bandwidths;
  const int ctas = (int)mmd_ctas(n_cells);
  double* part = static_cast<double*>(ws);
#define CC_MMD_LAUNCH(NB)                                                                     \
  mmd_tiles_kernel<NB><<<ctas, kMmdThreads, 0, st>>>(gram, ldg, n_cells, bw, masks, W,       \
                                                      labellings, part, part_ld)
  switch (n_bandwidths) {
    case 1: CC_MMD_LAUNCH(1); break;
    case 2: CC_MMD_LAUNCH(2); break;
    case 3: CC_MMD_LAUNCH(3); break;
    default: CC_MMD_LAUNCH(4); break;
  }
#undef CC_MMD_LAUNCH
  CC_CHECK_LAUNCH();
  const long long q = labellings * n_bandwidths;
  mmd_finish_kernel<<<(unsigned)((q + 255) / 256), 256, 0, st>>>(part, part_ld, ctas,
                                                                 n_bandwidths, labellings, sums);
  CC_CHECK_LAUNCH();
  return 0;
}
