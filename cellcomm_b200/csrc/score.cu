// Per-cell reconstruction error of a dense fp32 prediction tile against CSR count rows.
//
// The score pass (BiGanEngine.score_stream) needs, for every cell x, the squared error of the
// generator's fp32 output G(E(x), r) against x's exact counts.  The training MSE kernel sums
// over the whole batch and compares against the bf16 gather (counts above 256 are rounded
// there), so this is its own kernel: out[r] = scale * sum_c (pred[r, c] - x[row0 + r, c])^2.
//
// One CTA per row, no atomics on the output, so the result is a pure function of the inputs:
//   1. a bitmap of the row's stored columns in shared memory (atomicOr on shared words only)
//   2. stream the dense row with float4 loads, adding p^2 where the bit is clear
//   3. add (p - x)^2 over the row's stored entries (the row was just read: L2 hits)
//   4. block reduction in a fixed order (warp shuffles, then warp 0 over the warp sums)
// Every term is non-negative; the expanded form sum p^2 - 2 sum p x + sum x^2 would cancel
// catastrophically in fp32 when large counts are reconstructed closely.  Columns [cols, ld)
// are never counted.  Stored entries must have unique columns within a row (the loader's
// CSR); an explicit zero is counted once, as (p - 0)^2.
#include "common.cuh"

namespace cc {

// bitmap capacity: 32 KB of shared memory (262,144 columns), inside the default 48 KB limit
constexpr long long kScoreMaxCols = 1ll << 18;

template <bool VEC>
__global__ void __launch_bounds__(512, 4)
recon_sqerr_kernel(const float* __restrict__ pred, long long ld, long long cols,
                   const long long* __restrict__ rowptr, const int* __restrict__ colidx,
                   const float* __restrict__ values, long long row0, float scale,
                   float* __restrict__ out) {
  extern __shared__ unsigned bits[];
  __shared__ float warp_sum[32];
  const long long r = blockIdx.x;
  const float* row = pred + r * ld;
  const long long beg = rowptr[row0 + r], end = rowptr[row0 + r + 1];
  const long long words = (cols + 31) >> 5;
  for (long long w = threadIdx.x; w < words; w += blockDim.x) bits[w] = 0u;
  __syncthreads();
  for (long long e = beg + threadIdx.x; e < end; e += blockDim.x) {
    const long long c = colidx[e];
    if (c >= 0 && c < cols) atomicOr(&bits[c >> 5], 1u << (c & 31));
  }
  __syncthreads();

  float acc = 0.f;
  for (long long c = 4ll * threadIdx.x; c < cols; c += 4ll * blockDim.x) {
    float p[4];
    if (VEC) {
      const float4 v = *reinterpret_cast<const float4*>(row + c);
      p[0] = v.x, p[1] = v.y, p[2] = v.z, p[3] = v.w;
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) p[k] = c + k < cols ? row[c + k] : 0.f;
    }
    const unsigned m = bits[c >> 5] >> (c & 31);   // c % 4 == 0: one word holds all four bits
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (c + k < cols && !((m >> k) & 1u)) acc += p[k] * p[k];
  }
  for (long long e = beg + threadIdx.x; e < end; e += blockDim.x) {
    const long long c = colidx[e];
    if (c >= 0 && c < cols) {
      const float d = row[c] - values[e];
      acc += d * d;
    }
  }

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) warp_sum[warp] = acc;
  __syncthreads();
  if (warp == 0) {
    float s = lane < nwarps ? warp_sum[lane] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[r] = scale * s;
  }
}

}  // namespace cc

extern "C" int cc_recon_sqerr(const float* pred, int64_t ld, int64_t rows, int64_t cols,
                              const int64_t* rowptr, const int32_t* colidx, const float* values,
                              int64_t row0, float scale, float* out, cc_stream_t stream) {
  using namespace cc;
  CC_REQUIRE(rows >= 0 && cols >= 0 && row0 >= 0, "cc_recon_sqerr: rows %lld / cols %lld / "
             "row0 %lld < 0", (long long)rows, (long long)cols, (long long)row0);
  CC_REQUIRE(ld >= cols, "cc_recon_sqerr: ld %lld < cols %lld", (long long)ld, (long long)cols);
  CC_REQUIRE(cols <= kScoreMaxCols, "cc_recon_sqerr: %lld columns exceed the %lld the "
             "shared-memory bitmap holds", (long long)cols, kScoreMaxCols);
  CC_REQUIRE(rows <= INT32_MAX, "cc_recon_sqerr: %lld rows: launch one tile at a time",
             (long long)rows);
  if (rows == 0) return 0;
  CC_REQUIRE((cols == 0 || pred != nullptr) && rowptr != nullptr && out != nullptr,
             "cc_recon_sqerr: null pointer");
  // threads: enough that four float4 loads per thread cover the row, 32..512
  int threads = 32;
  while (threads < 512 && (long long)threads * 16 < cols) threads <<= 1;
  const size_t smem = (size_t)((cols + 31) >> 5) * sizeof(unsigned);
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = ld % 4 == 0 && (((uintptr_t)pred) & 15) == 0;
  if (vec)
    recon_sqerr_kernel<true><<<(unsigned)rows, threads, smem, st>>>(
        pred, ld, cols, (const long long*)rowptr, colidx, values, row0, scale, out);
  else
    recon_sqerr_kernel<false><<<(unsigned)rows, threads, smem, st>>>(
        pred, ld, cols, (const long long*)rowptr, colidx, values, row0, scale, out);
  CC_CHECK_LAUNCH();
  return 0;
}
