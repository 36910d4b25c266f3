// Generated cells -> CSR rows: round-half-even + compaction of a dense fp32 generator tile.
//
// Replaces the dense tail of generate_cells() (src/bigan_basic.py:40-44: G.predict -> host
// copy of the whole (n, genes) fp32 output -> np.round) for the streamed generate pass
// (BiGanEngine.generate_csr): each generator tile becomes CSR rows on the device, and only
// the non-zero counts cross the bus.
//
// Three launches, no atomics, so the output is a pure function of the tile:
//   count : one CTA per row, rintf(x) != 0 counted with float4 loads, block reduction
//           -> rowptr[1 + r] = nnz(row r)
//   scan  : one CTA, inclusive scan over the rows, seeded with rowptr[0] (the base offset)
//   fill  : one CTA per row; per pass every thread loads kFillVec float4s (vector j of thread
//           t covers columns 4 * (j * blockDim + t) ...), counts each vector's non-zeros, and
//           ONE block scan over the counts packed as 16-bit fields of a uint64 gives every
//           vector its output position in ascending column order (skipped for passes without
//           an entry; empty rows are not read at all).
// Columns [cols, ldx) may be loaded (the float4 path stays inside the row's ld) but are never
// counted or written.
#include "common.cuh"

namespace cc {

constexpr int kFillVec = 4;  // float4 loads per thread per pass of the fill kernel

__device__ __forceinline__ float4 load_vec4(const float* __restrict__ row, long long c,
                                            long long cols, bool vec) {
  if (vec) return *reinterpret_cast<const float4*>(row + c);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c + 0 < cols) v.x = row[c + 0];
  if (c + 1 < cols) v.y = row[c + 1];
  if (c + 2 < cols) v.z = row[c + 2];
  if (c + 3 < cols) v.w = row[c + 3];
  return v;
}

// rounded values of the 4 columns [c, c+4), zero beyond `cols`
__device__ __forceinline__ void round4(float4 v, long long c, long long cols, float (&f)[4]) {
  f[0] = rintf(v.x);
  f[1] = rintf(v.y);
  f[2] = rintf(v.z);
  f[3] = rintf(v.w);
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (c + k >= cols) f[k] = 0.f;
}

__device__ __forceinline__ int nz4(const float (&f)[4]) {
  return (f[0] != 0.f) + (f[1] != 0.f) + (f[2] != 0.f) + (f[3] != 0.f);
}

// inclusive scan over the block (blockDim.x a multiple of 32, at most 1024); `total` gets the
// block's sum.  scratch: 32 elements of shared memory.  Contains __syncthreads.
template <typename T>
__device__ __forceinline__ T block_inclusive_scan(T v, T* scratch, T* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  if (lane == 31) scratch[warp] = v;
  __syncthreads();
  if (warp == 0) {
    T w = lane < nwarps ? scratch[lane] : T(0);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const T u = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += u;
    }
    scratch[lane] = w;  // inclusive prefix over warps
  }
  __syncthreads();
  if (warp > 0) v += scratch[warp - 1];
  *total = scratch[nwarps - 1];
  __syncthreads();  // scratch may be reused by the caller's next scan
  return v;
}

template <bool VEC>
__global__ void __launch_bounds__(512, 4)
round_csr_count_kernel(const float* __restrict__ x, long long ldx, long long cols,
                       long long* __restrict__ rowptr) {
  __shared__ long long scratch[32];
  const long long r = blockIdx.x;
  const float* row = x + r * ldx;
  long long n = 0;
  for (long long c = 4ll * threadIdx.x; c < cols; c += 4ll * blockDim.x) {
    float f[4];
    round4(load_vec4(row, c, cols, VEC), c, cols, f);
    n += nz4(f);
  }
  long long total;
  block_inclusive_scan(n, scratch, &total);
  if (threadIdx.x == 0) rowptr[1 + r] = total;
}

// rowptr[1 + r] (counts) -> rowptr[0] + inclusive prefix sums; one CTA
__global__ void __launch_bounds__(1024)
round_csr_scan_kernel(long long rows, long long* __restrict__ rowptr) {
  __shared__ long long scratch[32];
  long long carry = rowptr[0];
  for (long long r0 = 0; r0 < rows; r0 += blockDim.x) {
    const long long r = r0 + threadIdx.x;
    const long long v = r < rows ? rowptr[1 + r] : 0;
    long long total;
    const long long incl = block_inclusive_scan(v, scratch, &total);
    if (r < rows) rowptr[1 + r] = carry + incl;
    carry += total;
  }
}

template <bool VEC>
__global__ void __launch_bounds__(512, 2)
round_csr_fill_kernel(const float* __restrict__ x, long long ldx, long long cols,
                      const long long* __restrict__ rowptr, int* __restrict__ colidx,
                      float* __restrict__ values) {
  static_assert(kFillVec <= 4, "four 16-bit count fields in a uint64");
  __shared__ unsigned long long scratch[32];
  const long long r = blockIdx.x;
  const float* row = x + r * ldx;
  long long out = rowptr[r] - rowptr[0];
  if (rowptr[r + 1] == rowptr[r]) return;  // an empty row: nothing to read
  const long long B = blockDim.x;
  for (long long base = 0; base < cols; base += 4 * kFillVec * B) {
    float f[kFillVec][4];
    unsigned long long packed = 0;
#pragma unroll
    for (int j = 0; j < kFillVec; ++j) {
      const long long c = base + 4 * (j * B + threadIdx.x);
      if (c < cols) {
        round4(load_vec4(row, c, cols, VEC), c, cols, f[j]);
      } else {
        f[j][0] = f[j][1] = f[j][2] = f[j][3] = 0.f;
      }
      // per field: at most 4 * blockDim.x <= 4096 < 2^16
      packed |= (unsigned long long)nz4(f[j]) << (16 * j);
    }
    if (!__syncthreads_or(packed != 0)) continue;  // no entry in this pass: skip the scan
    unsigned long long total;
    const unsigned long long incl = block_inclusive_scan(packed, scratch, &total);
    const unsigned long long excl = incl - packed;
    long long pos = out;
#pragma unroll
    for (int j = 0; j < kFillVec; ++j) {
      long long o = pos + (long long)((excl >> (16 * j)) & 0xffffu);
      const long long c = base + 4 * (j * B + threadIdx.x);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (f[j][k] != 0.f) {
          colidx[o] = (int)(c + k);
          values[o] = f[j][k];
          ++o;
        }
      pos += (long long)((total >> (16 * j)) & 0xffffu);  // vectors j' < j come first
    }
    out = pos;
  }
}

// threads per row CTA: enough for one pass over the row, 32..512
static int row_threads(long long cols, int per_thread) {
  int t = 32;
  while (t < 512 && (long long)t * per_thread < cols) t <<= 1;
  return t;
}

static int check_tile(const char* fn, const float* x, int64_t ldx, int64_t rows, int64_t cols,
                      const void* rowptr) {
  CC_REQUIRE(rows >= 0 && cols >= 0, "%s: rows %lld / cols %lld < 0", fn, (long long)rows,
             (long long)cols);
  CC_REQUIRE(ldx >= cols, "%s: ldx %lld < cols %lld", fn, (long long)ldx, (long long)cols);
  CC_REQUIRE(cols <= INT32_MAX, "%s: cols %lld do not fit the int32 column index", fn,
             (long long)cols);
  CC_REQUIRE(rows <= INT32_MAX, "%s: %lld rows: launch one tile at a time", fn, (long long)rows);
  CC_REQUIRE(rows == 0 || ((cols == 0 || x != nullptr) && rowptr != nullptr), "%s: null pointer",
             fn);
  return 0;
}

static bool vec_ok(const float* x, int64_t ldx) {
  return ldx % 4 == 0 && (((uintptr_t)x) & 15) == 0;
}

}  // namespace cc

extern "C" int cc_round_csr_count(const float* x, int64_t ldx, int64_t rows, int64_t cols,
                                  int64_t* rowptr, cc_stream_t stream) {
  using namespace cc;
  if (int rc = check_tile("cc_round_csr_count", x, ldx, rows, cols, rowptr)) return rc;
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int threads = row_threads(cols, 4 * 4);
  if (vec_ok(x, ldx))
    round_csr_count_kernel<true><<<(unsigned)rows, threads, 0, st>>>(x, ldx, cols,
                                                                     (long long*)rowptr);
  else
    round_csr_count_kernel<false><<<(unsigned)rows, threads, 0, st>>>(x, ldx, cols,
                                                                      (long long*)rowptr);
  CC_CHECK_LAUNCH();
  round_csr_scan_kernel<<<1, 1024, 0, st>>>(rows, (long long*)rowptr);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_round_csr_fill(const float* x, int64_t ldx, int64_t rows, int64_t cols,
                                 const int64_t* rowptr, int32_t* colidx, float* values,
                                 cc_stream_t stream) {
  using namespace cc;
  if (int rc = check_tile("cc_round_csr_fill", x, ldx, rows, cols, rowptr)) return rc;
  if (rows == 0 || cols == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int threads = row_threads(cols, 4 * kFillVec);
  if (vec_ok(x, ldx))
    round_csr_fill_kernel<true><<<(unsigned)rows, threads, 0, st>>>(
        x, ldx, cols, (const long long*)rowptr, colidx, values);
  else
    round_csr_fill_kernel<false><<<(unsigned)rows, threads, 0, st>>>(
        x, ldx, cols, (const long long*)rowptr, colidx, values);
  CC_CHECK_LAUNCH();
  return 0;
}
