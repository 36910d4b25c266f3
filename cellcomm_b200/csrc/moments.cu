// Per-gene moments of a dense fp32 tile: column sums, sums of squares and non-zero counts.
//
// The compare pass (BiGanEngine.moments_stream) reduces real cells (gathered to fp32) and
// generated cells (the generator's fp32 output, rounded half to even) per cell class into
//   sum[c] += sum_r v,   sumsq[c] += sum_r v^2,   nonzero[c] += #{r : v != 0}
// from which mean, variance and detection rate follow on the host.
//
// Geometry: a CTA of 32 x 8 threads owns 128 columns (four adjacent columns per thread, float4
// loads where the layout allows) and one slab of kMomentsSlabRows rows; the grid is column
// blocks x row slabs, so a 4096-row tile of 33,694 genes is 264 x 16 CTAs with several KB of
// loads in flight each.  Every thread accumulates in fp64, so for integer data (counts, rounded
// counts) every partial and total is an exact integer below 2^53 and the result does not
// depend on the order, the tiling or the slab count at all.
//
// Combine, fixed order and no float atomics (the ticket scheme of colreduce_kernel in
// tail_kernels.cu): with one slab the CTA adds its column totals straight into the outputs;
// with more, every CTA stores its per-column partials to the workspace and takes a ticket from
// its column block's counter, and the CTA that draws the last ticket sums the partials in slab
// order 0, 1, ..., adds them once to the outputs and re-zeroes the counter.  No CTA waits for
// another.  The geometry depends on (rows, cols) alone, so the workspace size is a host-side
// function and identical inputs give identical bits on any GPU.
#include "common.cuh"

namespace cc {

constexpr long long kMomentsSlabRows = 256;
constexpr long long kMomentsMaxCols = 1ll << 18;             // column blocks <= 2048 tickets
constexpr long long kMomentsTicketBytes = (kMomentsMaxCols / 128) * sizeof(unsigned);
constexpr int kMomentsUnroll = 8;                            // row loads in flight per thread

template <bool VEC>
__device__ __forceinline__ float4 moments_load(const float* __restrict__ row, long long c,
                                               long long cols) {
  if (VEC) return *reinterpret_cast<const float4*>(row + c);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c + 0 < cols) v.x = row[c + 0];
  if (c + 1 < cols) v.y = row[c + 1];
  if (c + 2 < cols) v.z = row[c + 2];
  if (c + 3 < cols) v.w = row[c + 3];
  return v;
}

template <bool VEC, bool ROUND>
__global__ void __launch_bounds__(256, 3)
col_moments_kernel(const float* __restrict__ x, long long ld, long long rows, long long cols,
                   double* __restrict__ sum, double* __restrict__ sumsq,
                   long long* __restrict__ nonzero, double* __restrict__ part,
                   unsigned* __restrict__ tickets) {
  __shared__ double s1[8][128], s2[8][128];
  __shared__ int sn[8][128];
  __shared__ bool last;
  const int tx = threadIdx.x, ty = threadIdx.y;
  const long long c = (long long)blockIdx.x * 128 + tx * 4;
  const long long r_begin = (long long)blockIdx.y * kMomentsSlabRows;
  const long long r_end = min(rows, r_begin + kMomentsSlabRows);
  double a1[4] = {0.0, 0.0, 0.0, 0.0}, a2[4] = {0.0, 0.0, 0.0, 0.0};
  int an[4] = {0, 0, 0, 0};
  // columns at or past `cols` (the padding [cols, ld) may hold anything) are never added
  const int nv = (int)max(0ll, min(4ll, cols - c));
  auto consume = [&](const float4 v) {
    const float f[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (k < nv) {
        const float y = ROUND ? rintf(f[k]) : f[k];     // rintf: round half to even
        const double d = (double)y;
        a1[k] += d;
        a2[k] = fma(d, d, a2[k]);
        an[k] += y != 0.f;                              // -0.0f counts as zero
      }
    }
  };
  if (nv > 0) {
    long long r = r_begin + ty;
    for (; r + 8 * (kMomentsUnroll - 1) < r_end; r += 8 * kMomentsUnroll) {
      float4 v[kMomentsUnroll];
#pragma unroll
      for (int u = 0; u < kMomentsUnroll; ++u)
        v[u] = moments_load<VEC>(x + (r + 8 * u) * ld, c, cols);
#pragma unroll
      for (int u = 0; u < kMomentsUnroll; ++u) consume(v[u]);
    }
    for (; r < r_end; r += 8) consume(moments_load<VEC>(x + r * ld, c, cols));
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    s1[ty][tx * 4 + k] = a1[k];
    s2[ty][tx * 4 + k] = a2[k];
    sn[ty][tx * 4 + k] = an[k];
  }
  __syncthreads();
  const int j = ty * 32 + tx;                  // ty < 4: one column of the block per thread
  const long long col = (long long)blockIdx.x * 128 + j;
  const bool mine = ty < 4 && col < cols;
  double t1 = 0.0, t2 = 0.0;
  long long tn = 0;
  if (mine) {
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      t1 += s1[y][j];
      t2 += s2[y][j];
      tn += sn[y][j];
    }
  }
  if (gridDim.y == 1) {                        // the only writer of these columns
    if (mine) {
      sum[col] += t1;
      sumsq[col] += t2;
      nonzero[col] += tn;
    }
    return;
  }
  double* p1 = part;
  double* p2 = part + (long long)gridDim.y * cols;
  long long* pn = reinterpret_cast<long long*>(part + 2ll * gridDim.y * cols);
  if (mine) {
    const long long at = (long long)blockIdx.y * cols + col;
    p1[at] = t1;
    p2[at] = t2;
    pn[at] = tn;
  }
  __threadfence();  // partials visible device-wide before the ticket is taken
  __syncthreads();
  if (tx == 0 && ty == 0) last = atomicAdd(tickets + blockIdx.x, 1u) == gridDim.y - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (mine) {
    double u1 = 0.0, u2 = 0.0;
    long long un = 0;
    for (unsigned y = 0; y < gridDim.y; ++y) {
      const long long at = (long long)y * cols + col;
      u1 += __ldcg(p1 + at);
      u2 += __ldcg(p2 + at);
      un += __ldcg(pn + at);
    }
    sum[col] += u1;
    sumsq[col] += u2;
    nonzero[col] += un;
  }
  if (tx == 0 && ty == 0) tickets[blockIdx.x] = 0u;  // ready for the next launch
}

static long long moments_slabs(long long rows) {
  return (rows + kMomentsSlabRows - 1) / kMomentsSlabRows;
}

}  // namespace cc

extern "C" int64_t cc_col_moments_ws_bytes(int64_t rows, int64_t cols) {
  using namespace cc;
  if (rows <= 0 || cols <= 0) return 0;
  const long long gy = moments_slabs(rows);
  return gy > 1 ? kMomentsTicketBytes + gy * (long long)cols * 24 : 0;
}

extern "C" int cc_col_moments(const float* x, int64_t ld, int64_t rows, int64_t cols,
                              int32_t round_half_even, double* sum, double* sumsq,
                              int64_t* nonzero, void* ws, int64_t ws_bytes, cc_stream_t stream) {
  using namespace cc;
  CC_REQUIRE(rows >= 0 && cols >= 0, "cc_col_moments: rows %lld / cols %lld < 0",
             (long long)rows, (long long)cols);
  CC_REQUIRE(ld >= cols, "cc_col_moments: ld %lld < cols %lld", (long long)ld, (long long)cols);
  CC_REQUIRE(cols <= kMomentsMaxCols, "cc_col_moments: %lld columns exceed the %lld the "
             "workspace's ticket counters cover", (long long)cols, kMomentsMaxCols);
  CC_REQUIRE(moments_slabs(rows) <= 65535, "cc_col_moments: %lld rows: launch at most %lld at "
             "a time", (long long)rows, 65535 * kMomentsSlabRows);
  if (rows == 0 || cols == 0) return 0;
  CC_REQUIRE(x != nullptr && sum != nullptr && sumsq != nullptr && nonzero != nullptr,
             "cc_col_moments: null pointer");
  const long long need = cc_col_moments_ws_bytes(rows, cols);
  CC_REQUIRE(ws_bytes >= need && (need == 0 || ws != nullptr),
             "cc_col_moments of [%lld, %lld]: workspace of %lld bytes, needs %lld "
             "(cc_col_moments_ws_bytes)", (long long)rows, (long long)cols,
             (long long)(ws == nullptr ? 0 : ws_bytes), need);
  CC_REQUIRE(need == 0 || (((uintptr_t)ws) & 15) == 0,
             "cc_col_moments: workspace must be 16-byte aligned");
  const dim3 grid((unsigned)((cols + 127) / 128), (unsigned)moments_slabs(rows)), block(32, 8);
  unsigned* tickets = static_cast<unsigned*>(ws);
  double* part = need ? reinterpret_cast<double*>(static_cast<char*>(ws) + kMomentsTicketBytes)
                      : nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = ld % 4 == 0 && (((uintptr_t)x) & 15) == 0;
  long long* nz = reinterpret_cast<long long*>(nonzero);
#define CC_MOMENTS_LAUNCH(V, R) \
  col_moments_kernel<V, R><<<grid, block, 0, st>>>(x, ld, rows, cols, sum, sumsq, nz, part, tickets)
  if (vec && round_half_even) CC_MOMENTS_LAUNCH(true, true);
  else if (vec) CC_MOMENTS_LAUNCH(true, false);
  else if (round_half_even) CC_MOMENTS_LAUNCH(false, true);
  else CC_MOMENTS_LAUNCH(false, false);
#undef CC_MOMENTS_LAUNCH
  CC_CHECK_LAUNCH();
  return 0;
}
