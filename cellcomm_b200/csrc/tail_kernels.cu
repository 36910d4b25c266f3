// HBM-bound tail kernels around the GEMMs: dropout / RNG, activation backward, copies and
// casts, column reductions, BatchNormalization, softmax, losses, rounding, one-hot, RMSprop.
// Every kernel streams row-major [rows, cols] tensors with 16-byte vector accesses where the
// layout allows (ld % 8 == 0, aligned base) and is sized in multiples of the SM count.
//
// Reference semantics: Keras 2.4.0 layers used by src/bigan_classify.py:10-75 and
// src/bigan_cont.py:7-41 (SURVEY.md Appendix A.3-A.6).
#include "common.cuh"

namespace cc {

static int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      n = 148;
  }
  return n;
}

// grid for an elementwise pass over `work` vector items with `threads` per block:
// a multiple of the SM count, capped at 8 resident blocks per SM.
static unsigned ew_grid(long long work, int threads) {
  long long blocks = (work + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

struct alignas(16) bf16x8 {
  __nv_bfloat162 v[4];
};

// A row-major [rows, cols] operand that is either bf16 or fp32 (activations that feed a
// BatchNormalization and all activation gradients are kept in fp32, see DESIGN.md).
struct Mat {
  void* p;
  long long ld;
  int f32;
};
static inline Mat mat(const void* p, long long ld, int f32) {
  return Mat{const_cast<void*>(p), ld, f32};
}

__device__ __forceinline__ void load8(const Mat& m, long long r, long long c0, int n,
                                      float (&f)[8]) {
  if (m.f32) {
    const float* p = reinterpret_cast<const float*>(m.p) + r * m.ld + c0;
    if (n == 8 && (m.ld % 4) == 0 && ((((uintptr_t)m.p) & 15) == 0)) {
      const float4 a = *reinterpret_cast<const float4*>(p);
      const float4 b = *reinterpret_cast<const float4*>(p + 4);
      f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
      f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] = (i < n) ? p[i] : 0.f;
    }
  } else {
    const bf16* p = reinterpret_cast<const bf16*>(m.p) + r * m.ld + c0;
    if (n == 8 && (m.ld % 8) == 0 && ((((uintptr_t)m.p) & 15) == 0)) {
      bf16x8 q = *reinterpret_cast<const bf16x8*>(p);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float2 t = __bfloat1622float2(q.v[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] = (i < n) ? bf2f(p[i]) : 0.f;
    }
  }
}
__device__ __forceinline__ void store8(const Mat& m, long long r, long long c0, int n,
                                       const float (&f)[8]) {
  if (m.f32) {
    float* p = reinterpret_cast<float*>(m.p) + r * m.ld + c0;
    if (n == 8 && (m.ld % 4) == 0 && ((((uintptr_t)m.p) & 15) == 0)) {
      *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
      *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < n) p[i] = f[i];
    }
  } else {
    bf16* p = reinterpret_cast<bf16*>(m.p) + r * m.ld + c0;
    if (n == 8 && (m.ld % 8) == 0 && ((((uintptr_t)m.p) & 15) == 0)) {
      bf16x8 q;
#pragma unroll
      for (int i = 0; i < 4; ++i) q.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      *reinterpret_cast<bf16x8*>(p) = q;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < n) p[i] = f2bf(f[i]);
    }
  }
}
__device__ __forceinline__ float load1(const Mat& m, long long r, long long c) {
  return m.f32 ? reinterpret_cast<const float*>(m.p)[r * m.ld + c]
               : bf2f(reinterpret_cast<const bf16*>(m.p)[r * m.ld + c]);
}
__device__ __forceinline__ void store1(const Mat& m, long long r, long long c, float v) {
  if (m.f32) reinterpret_cast<float*>(m.p)[r * m.ld + c] = v;
  else reinterpret_cast<bf16*>(m.p)[r * m.ld + c] = f2bf(v);
}

// Iterate over [rows, cols] in chunks of 8 consecutive columns; F(row, col0, nvalid).
// One division per thread, not per chunk: the T threads of the launch form T / cpr "row lanes"
// of cpr threads each (cpr = chunks per row); a thread keeps its column chunk and walks down
// the rows.  When a row has more chunks than the launch has threads, the plain grid-stride
// walk (with its division) is used.
template <typename F>
__device__ __forceinline__ void for_each_chunk8(long long rows, long long cols, F f) {
  const long long cpr = (cols + 7) / 8;
  const long long T = (long long)gridDim.x * blockDim.x;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (cpr <= T && cpr < (1ll << 31)) {
    const unsigned lanes = (unsigned)(T / cpr);
    const unsigned lane = (unsigned)(tid / cpr);
    if (lane >= lanes) return;
    const long long c0 = (tid - (long long)lane * cpr) * 8;
    const int n = (int)min((long long)8, cols - c0);
    for (long long r = lane; r < rows; r += lanes) f(r, c0, n);
  } else {
    const long long total = rows * cpr;
    for (long long i = tid; i < total; i += T) {
      const long long r = i / cpr;
      const long long c0 = (i - r * cpr) * 8;
      const int n = (int)min((long long)8, cols - c0);
      f(r, c0, n);
    }
  }
}

// eight consecutive fp32 per-column parameters (BN gamma / beta / mean / rstd): two float4
// when aligned (c0 is a multiple of 8), scalars at a ragged edge
__device__ __forceinline__ void load8_param(const float* __restrict__ p, long long c0, int n,
                                            float (&f)[8]) {
  if (n == 8 && ((((uintptr_t)(p + c0)) & 15) == 0)) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p + c0));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + c0 + 4));
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
    f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = (i < n) ? __ldg(p + c0 + i) : 0.f;
  }
}

// ------------------------------------------------------------------ RNG / dropout
__device__ __forceinline__ void rng8(uint64_t seed, uint64_t step, uint32_t stream_id, long long r,
                                     long long c0, long long cols, float (&u)[8]) {
  // two Philox blocks per 8 columns; the counter is the (row, column/4) position, so the
  // stream does not depend on the launch geometry.
  const uint64_t blocks_per_row = (uint64_t)((cols + 3) / 4);
  const uint64_t hi = ((uint64_t)stream_id << 40) ^ step;
  uint32_t o[4];
  Philox::block(seed, hi, (uint64_t)r * blocks_per_row + (uint64_t)(c0 / 4), o);
#pragma unroll
  for (int i = 0; i < 4; ++i) u[i] = u32_to_unit(o[i]);
  Philox::block(seed, hi, (uint64_t)r * blocks_per_row + (uint64_t)(c0 / 4) + 1, o);
#pragma unroll
  for (int i = 0; i < 4; ++i) u[4 + i] = u32_to_unit(o[i]);
}

__global__ void dropout_kernel(const Mat x, const Mat out, long long rows, long long cols,
                               float rate, const uint8_t* __restrict__ mask, long long ldm,
                               uint64_t seed, const uint64_t* __restrict__ counter,
                               uint32_t stream_id) {
  const float scale = 1.f / (1.f - rate);
  const uint64_t step = counter ? *counter : 0;
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float f[8];
    load8(x, r, c0, n, f);
    if (mask != nullptr) {
      const uint8_t* m = mask + r * ldm + c0;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < n) f[i] = m[i] ? f[i] * scale : 0.f;
    } else {
      float u[8];
      rng8(seed, step, stream_id, r, c0, cols, u);
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] = (u[i] >= rate) ? f[i] * scale : 0.f;
    }
    store8(out, r, c0, n, f);
  });
}

__global__ void dropout_mask_kernel(uint8_t* __restrict__ mask, long long ldm, long long rows,
                                    long long cols, float rate, uint64_t seed,
                                    const uint64_t* __restrict__ counter, uint32_t stream_id) {
  const uint64_t step = counter ? *counter : 0;
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float u[8];
    rng8(seed, step, stream_id, r, c0, cols, u);
    for (int i = 0; i < n; ++i) mask[r * ldm + c0 + i] = (u[i] >= rate) ? 1 : 0;
  });
}

__global__ void uniform_kernel(float* __restrict__ out32, bf16* __restrict__ out16, long long ld,
                               long long rows, long long cols, uint64_t seed,
                               const uint64_t* __restrict__ counter, uint32_t stream_id) {
  const uint64_t step = counter ? *counter : 0;
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float u[8];
    rng8(seed, step, stream_id, r, c0, cols, u);
    for (int i = 0; i < n; ++i) {
      if (out32) out32[r * ld + c0 + i] = u[i];
      if (out16) out16[r * ld + c0 + i] = f2bf(u[i]);
    }
  });
}

__global__ void counter_add_kernel(uint64_t* counter, uint64_t inc) { *counter += inc; }

// ------------------------------------------------------------------ simple elementwise
__global__ void act_bwd_kernel(const Mat dy, const Mat y, const Mat dz, long long rows,
                               long long cols, int act) {
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float g[8], a[8];
    load8(dy, r, c0, n, g);
    load8(y, r, c0, n, a);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      g[i] *= (act == CC_ACT_SIGMOID) ? a[i] * (1.f - a[i])
                                      : (act == CC_ACT_RELU ? (a[i] > 0.f ? 1.f : 0.f) : 1.f);
    store8(dz, r, c0, n, g);
  });
}

__global__ void copy2d_kernel(const Mat src, const Mat dst, long long rows, long long cols,
                              int beta, float scale) {
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float f[8];
    load8(src, r, c0, n, f);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] *= scale;
    if (beta) {
      float o[8];
      load8(dst, r, c0, n, o);
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] += o[i];
    }
    store8(dst, r, c0, n, f);
  });
}

// hi = bf16(x), lo = bf16(x - hi): a two-term bf16 expansion of an fp32 activation, consumed
// as two accumulating GEMM segments where 8 mantissa bits are not enough (inputs of the Dense
// layers that feed a BatchNormalization, see DESIGN.md "precision policy").
__global__ void split_kernel(const Mat x, const Mat hi, const Mat lo, long long rows,
                             long long cols) {
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float f[8], h[8], l[8];
    load8(x, r, c0, n, f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      h[i] = bf2f(f2bf(f[i]));
      l[i] = f[i] - h[i];
    }
    store8(hi, r, c0, n, h);
    store8(lo, r, c0, n, l);
  });
}

__global__ void round_kernel(const Mat x, const Mat out, float* __restrict__ out32,
                             long long ldo32, long long rows, long long cols) {
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float f[8];
    load8(x, r, c0, n, f);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = rintf(f[i]);  // round half to even (tf.math.round)
    if (out.p) store8(out, r, c0, n, f);
    if (out32)
      for (int i = 0; i < n; ++i) out32[r * ldo32 + c0 + i] = f[i];
  });
}

// y[r, c] = act(bias[c]) for every row: a Dense layer whose input width is 0 (the reference's
// 5-gene fixture yields Dense(0) layers, SURVEY.md D10)
__global__ void bias_act_kernel(const float* __restrict__ bias, int act, bf16* __restrict__ out16,
                                long long ld16, float* __restrict__ out32, long long ld32,
                                long long rows, long long cols) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < rows * cols;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols, c = i - r * cols;
    float v = bias ? bias[c] : 0.f;
    if (act == CC_ACT_SIGMOID) v = sigmoidf_(v);
    else if (act == CC_ACT_RELU) v = fmaxf(v, 0.f);
    if (out16) out16[r * ld16 + c] = f2bf(v);
    if (out32) out32[r * ld32 + c] = v;
  }
}

__global__ void fill_f32_kernel(float* dst, float v, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    dst[i] = v;
}

// ------------------------------------------------------------------ column reductions
// four adjacent columns of one row (16-byte / 8-byte vector access when whole and aligned)
__device__ __forceinline__ void load_quad(const Mat& m, long long r, long long c, int nv,
                                          float (&x)[4]) {
  if (m.f32) {
    const float* p = reinterpret_cast<const float*>(m.p) + r * m.ld + c;
    if (nv == 4 && (m.ld & 3) == 0 && ((((uintptr_t)m.p) & 15) == 0)) {
      const float4 t = *reinterpret_cast<const float4*>(p);
      x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = (i < nv) ? p[i] : 0.f;
    }
  } else {
    const bf16* p = reinterpret_cast<const bf16*>(m.p) + r * m.ld + c;
    if (nv == 4 && (m.ld & 3) == 0 && ((((uintptr_t)m.p) & 7) == 0)) {
      const uint2 t = *reinterpret_cast<const uint2*>(p);
      const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
      const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
      x[0] = lo.x; x[1] = lo.y; x[2] = hi.x; x[3] = hi.y;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = (i < nv) ? bf2f(p[i]) : 0.f;
    }
  }
}
__device__ __forceinline__ void store_quad(const Mat& m, long long r, long long c, int nv,
                                           const float (&x)[4]) {
  if (m.f32) {
    float* p = reinterpret_cast<float*>(m.p) + r * m.ld + c;
    if (nv == 4 && (m.ld & 3) == 0 && ((((uintptr_t)m.p) & 15) == 0)) {
      *reinterpret_cast<float4*>(p) = make_float4(x[0], x[1], x[2], x[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < nv) p[i] = x[i];
    }
  } else {
    bf16* p = reinterpret_cast<bf16*>(m.p) + r * m.ld + c;
    if (nv == 4 && (m.ld & 3) == 0 && ((((uintptr_t)m.p) & 7) == 0)) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(x[0], x[1]);
      __nv_bfloat162 hi = __floats2bfloat162_rn(x[2], x[3]);
      uint2 t;
      t.x = *reinterpret_cast<uint32_t*>(&lo);
      t.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(p) = t;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < nv) p[i] = f2bf(x[i]);
    }
  }
}

// out[c] = sum_r f0(r,c), out[cols + c] = sum_r f1(r,c).  A block of 32 x 8 threads owns 128
// columns (four adjacent columns per thread: a warp reads 512 B (fp32) / 256 B (bf16) of a
// row per instruction) and strides over a slab of rows, four rows' loads in flight per
// thread.  With more than one slab (grid.y > 1) the slabs combine either with atomics
// (part == nullptr: run-dependent order) or in fixed order: every CTA stores its per-column
// partials to part[y][c] (second moment at part[grid.y + y][c]), then takes a ticket from its
// column block's counter; the CTA that draws the last ticket sums the grid.y partials in slab
// order 0..grid.y-1, writes (or adds to) out, and re-zeroes the counter.  No CTA waits for
// another, so the scheme cannot deadlock on CTAs that are not resident; only WHICH CTA
// finalises depends on timing, never the order of the additions.
template <int MODE>  // 0: x (1 output)  1: x, x^2   2: dy, dy*xhat   3: dy*act'(y) (1 output)
__global__ void __launch_bounds__(256)
colreduce_kernel(const Mat a, const Mat b, long long rows, long long cols,
                 const float* __restrict__ mean, const float* __restrict__ rstd,
                 float* __restrict__ out, int accumulate, int act, float* __restrict__ part,
                 unsigned int* __restrict__ tickets,
                 const Mat dz = Mat{nullptr, 0, 0}, const Mat dzlo = Mat{nullptr, 0, 0}) {
  __shared__ float s0[8][128], s1[8][128];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const long long c = (long long)blockIdx.x * 128 + tx * 4;
  const long long rows_per_slab = (rows + gridDim.y - 1) / gridDim.y;
  const long long r_begin = (long long)blockIdx.y * rows_per_slab;
  const long long r_end = min(rows, r_begin + rows_per_slab);
  const int nv = (int)max(0ll, min(4ll, cols - c));
  float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
  float mu[4] = {0.f, 0.f, 0.f, 0.f}, rs[4] = {0.f, 0.f, 0.f, 0.f};
  if (MODE == 2) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < nv) { mu[i] = mean[c + i]; rs[i] = rstd[c + i]; }
  }
  const bool need_b = MODE == 2 || (MODE == 3 && act != 0);
  auto consume = [&](long long r, const float (&x)[4], const float (&y)[4]) {
    if (MODE == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) acc0[i] += x[i];
    } else if (MODE == 1) {
#pragma unroll
      for (int i = 0; i < 4; ++i) { acc0[i] += x[i]; acc1[i] += x[i] * x[i]; }
    } else if (MODE == 2) {
#pragma unroll
      for (int i = 0; i < 4; ++i) { acc0[i] += x[i]; acc1[i] += x[i] * ((y[i] - mu[i]) * rs[i]); }
    } else {
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        v[i] = x[i] * (act == CC_ACT_SIGMOID ? y[i] * (1.f - y[i])
                                             : (act == CC_ACT_RELU ? (y[i] > 0.f ? 1.f : 0.f) : 1.f));
        acc0[i] += v[i];
      }
      if (dz.p != nullptr) store_quad(dz, r, c, nv, v);
      if (dzlo.p != nullptr) {  // two-term bf16 expansion of dz: the low-order term
        float l[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) l[i] = v[i] - bf2f(f2bf(v[i]));
        store_quad(dzlo, r, c, nv, l);
      }
    }
  };
  if (nv > 0) {
    long long r = r_begin + ty;
    for (; r + 24 < r_end; r += 32) {
      float x[4][4], y[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        load_quad(a, r + 8 * u, c, nv, x[u]);
        if (need_b) load_quad(b, r + 8 * u, c, nv, y[u]);
        else y[u][0] = y[u][1] = y[u][2] = y[u][3] = 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) consume(r + 8 * u, x[u], y[u]);
    }
    for (; r < r_end; r += 8) {
      float x[4], y[4] = {0.f, 0.f, 0.f, 0.f};
      load_quad(a, r, c, nv, x);
      if (need_b) load_quad(b, r, c, nv, y);
      consume(r, x, y);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    s0[ty][tx * 4 + i] = acc0[i];
    s1[ty][tx * 4 + i] = acc1[i];
  }
  __syncthreads();
  constexpr bool two = MODE == 1 || MODE == 2;
  const int j = ty * 32 + tx;  // ty < 4: one column of the block per thread
  const long long cc_ = (long long)blockIdx.x * 128 + j;
  if (part == nullptr) {
    if (ty < 4 && cc_ < cols && out != nullptr) {
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        t0 += s0[y][j];
        t1 += s1[y][j];
      }
      if (gridDim.y > 1 || accumulate) {
        atomicAdd(out + cc_, t0);
        if (two) atomicAdd(out + cols + cc_, t1);
      } else {
        out[cc_] = t0;
        if (two) out[cols + cc_] = t1;
      }
    }
    return;
  }
  // fixed-order combine of the slabs (out != nullptr and gridDim.y > 1 here)
  if (ty < 4 && cc_ < cols) {
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      t0 += s0[y][j];
      t1 += s1[y][j];
    }
    part[(long long)blockIdx.y * cols + cc_] = t0;
    if (two) part[(long long)(gridDim.y + blockIdx.y) * cols + cc_] = t1;
  }
  __threadfence();  // partials visible device-wide before the ticket is taken
  __syncthreads();
  __shared__ bool last;
  if (tx == 0 && ty == 0) last = atomicAdd(tickets + blockIdx.x, 1u) == gridDim.y - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (ty < 4 && cc_ < cols) {
    float t0 = 0.f, t1 = 0.f;
    for (unsigned y = 0; y < gridDim.y; ++y) {
      t0 += __ldcg(part + (long long)y * cols + cc_);
      if (two) t1 += __ldcg(part + (long long)(gridDim.y + y) * cols + cc_);
    }
    if (accumulate) {  // the only writer of these columns: a plain read-add-write
      out[cc_] += t0;
      if (two) out[cols + cc_] += t1;
    } else {
      out[cc_] = t0;
      if (two) out[cols + cc_] = t1;
    }
  }
  if (tx == 0 && ty == 0) tickets[blockIdx.x] = 0u;  // ready for the next launch / graph replay
}

// Fixed-order reduction workspace (cc_reduce_ws_floats): reduce_tickets() uint32 counters
// first, then the partials.  Only launches with more than one slab use it, and those have fewer
// than 2 * SMs column blocks, so every column-block counter index is below reduce_tickets()
// whatever the shape; the partials of one call never overlap the counters of another.
static long long reduce_tickets() { return 2ll * num_sms(); }

// the slab geometry of launch_colreduce: (column blocks, row slabs)
static void colreduce_grid(long long rows, long long cols, unsigned& gx, unsigned& gy) {
  gx = (unsigned)((cols + 127) / 128);
  // enough row slabs to cover ~2 waves of the machine when there are few column blocks
  gy = 1;
  const unsigned target = 2u * (unsigned)num_sms();
  if (gx < target) {
    gy = (target + gx - 1) / gx;
    const unsigned maxy = (unsigned)((rows + 63) / 64);
    if (gy > maxy) gy = maxy;
    if (gy < 1) gy = 1;
  }
}

// floats of workspace one fixed-order colreduce launch uses (0: it needs none)
static long long colreduce_ws_floats(long long rows, long long cols, int outputs) {
  unsigned gx, gy;
  colreduce_grid(rows, cols, gx, gy);
  return gy > 1 ? reduce_tickets() + (long long)outputs * gy * cols : 0;
}

static long long mse_blocks(long long rows, long long cols) {
  return ew_grid(rows * ((cols + 7) / 8), 256);
}

// ws == nullptr: slabs combine with atomics; else in fixed order through ws (ws_floats long)
template <int MODE>
static int launch_colreduce(const Mat& a, const Mat& b, long long rows, long long cols,
                            const float* mean, const float* rstd, float* out, int accumulate,
                            float* ws, long long ws_floats, cudaStream_t st, int act = 0,
                            const Mat dz = Mat{nullptr, 0, 0}, const Mat dzlo = Mat{nullptr, 0, 0}) {
  constexpr int outputs = (MODE == 0 || MODE == 3) ? 1 : 2;
  unsigned gx, gy;
  colreduce_grid(rows, cols, gx, gy);
  // one slab, or nothing to sum (a dz-only bias_grad): each column has a single writer already
  const bool fixed = ws != nullptr && gy > 1 && out != nullptr;
  if (fixed) {
    const long long need = colreduce_ws_floats(rows, cols, outputs);
    CC_REQUIRE(ws_floats >= need,
               "column reduction of [%lld, %lld]: workspace of %lld floats, needs %lld "
               "(cc_reduce_ws_floats)", rows, cols, (long long)ws_floats, need);
  } else if (gy > 1 && !accumulate && out != nullptr) {
    const long long n = outputs * cols;
    fill_f32_kernel<<<ew_grid(n, 256), 256, 0, st>>>(out, 0.f, n);
    CC_CHECK_LAUNCH();
  }
  colreduce_kernel<MODE><<<dim3(gx, gy), dim3(32, 8), 0, st>>>(
      a, b, rows, cols, mean, rstd, out, accumulate, act,
      fixed ? ws + reduce_tickets() : nullptr, fixed ? reinterpret_cast<unsigned int*>(ws) : nullptr,
      dz, dzlo);
  CC_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------ BatchNorm
// one thread per column: derive batch mean / rstd from the (possibly all-reduced) sums and
// update the moving statistics the way Keras does (biased variance, momentum 0.99).
__global__ void bn_finalize_kernel(const float* __restrict__ sums, long long cols, double inv_n,
                                   float eps, float momentum, float* __restrict__ moving_mean,
                                   float* __restrict__ moving_var, float* __restrict__ save_mean,
                                   float* __restrict__ save_rstd) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const double mean_d = (double)sums[c] * inv_n;
  double var_d = (double)sums[cols + c] * inv_n - mean_d * mean_d;
  const float mean = (float)mean_d;
  const float var = fmaxf((float)var_d, 0.f);
  save_mean[c] = mean;
  save_rstd[c] = rsqrtf(var + eps);
  if (moving_mean) moving_mean[c] = moving_mean[c] * momentum + mean * (1.f - momentum);
  if (moving_var) moving_var[c] = moving_var[c] * momentum + var * (1.f - momentum);
}

// y = (x - mean) * (gamma * rstd) + beta ; (mean, rstd) either saved batch stats or derived
// from moving stats (infer != 0: rstd := 1/sqrt(var+eps))
__global__ void bn_apply_kernel(const Mat x, const Mat y, long long rows, long long cols,
                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                const float* __restrict__ mean, const float* __restrict__ stat,
                                int infer, float eps) {
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float f[8], mu[8], st[8], ga[8], be[8];
    load8(x, r, c0, n, f);
    load8_param(mean, c0, n, mu);
    load8_param(stat, c0, n, st);
    load8_param(gamma, c0, n, ga);
    load8_param(beta, c0, n, be);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < n) {
        const float rs = infer ? rsqrtf(st[i] + eps) : st[i];
        f[i] = (f[i] - mu[i]) * (ga[i] * rs) + be[i];
      }
    }
    store8(y, r, c0, n, f);
  });
}

// dx = gamma*rstd*(dy - sum_dy/n - xhat*sum_dyxhat/n)
__global__ void bn_bwd_apply_kernel(const Mat dy, const Mat x, const Mat dx, long long rows,
                                    long long cols, const float* __restrict__ gamma,
                                    const float* __restrict__ mean, const float* __restrict__ rstd,
                                    const float* __restrict__ sums2, float inv_n) {
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float g[8], a[8], mu[8], rs[8], ga[8], s0[8], s1[8];
    load8(dy, r, c0, n, g);
    load8(x, r, c0, n, a);
    load8_param(mean, c0, n, mu);
    load8_param(rstd, c0, n, rs);
    load8_param(gamma, c0, n, ga);
    load8_param(sums2, c0, n, s0);
    load8_param(sums2 + cols, c0, n, s1);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < n) {
        const float xhat = (a[i] - mu[i]) * rs[i];
        g[i] = ga[i] * rs[i] * (g[i] - s0[i] * inv_n - xhat * s1[i] * inv_n);
      }
    }
    store8(dx, r, c0, n, g);
  });
}

__global__ void bn_param_grad_kernel(const float* __restrict__ sums2, long long cols,
                                     float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  if (dbeta) dbeta[c] = sums2[c];
  if (dgamma) dgamma[c] = sums2[cols + c];
}

__global__ void bn_infer_bwd_kernel(const Mat dy, const Mat dx, long long rows, long long cols,
                                    const float* __restrict__ gamma,
                                    const float* __restrict__ var, float eps) {
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float g[8];
    load8(dy, r, c0, n, g);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < n) g[i] *= gamma[c0 + i] * rsqrtf(var[c0 + i] + eps);
    store8(dx, r, c0, n, g);
  });
}

// ------------------------------------------------------------------ softmax / one-hot
__global__ void softmax_fwd_kernel(const Mat x, const Mat y, float* __restrict__ y32,
                                   long long ldy32, long long rows, long long cols) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float mx = -INFINITY;
  for (long long c = 0; c < cols; ++c) mx = fmaxf(mx, load1(x, r, c));
  float sum = 0.f;
  for (long long c = 0; c < cols; ++c) sum += __expf(load1(x, r, c) - mx);
  const float inv = 1.f / sum;
  for (long long c = 0; c < cols; ++c) {
    const float v = __expf(load1(x, r, c) - mx) * inv;
    if (y.p) store1(y, r, c, v);
    if (y32) y32[r * ldy32 + c] = v;
  }
}

__global__ void softmax_bwd_kernel(const Mat dy, const Mat y, const Mat dx, long long rows,
                                   long long cols) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float dot = 0.f;
  for (long long c = 0; c < cols; ++c) dot += load1(dy, r, c) * load1(y, r, c);
  for (long long c = 0; c < cols; ++c)
    store1(dx, r, c, load1(y, r, c) * (load1(dy, r, c) - dot));
}

__global__ void argmax_onehot_kernel(const float* __restrict__ p, long long ldp,
                                     bf16* __restrict__ out16, long long ldo,
                                     float* __restrict__ out32, long long ldo32, long long rows,
                                     long long cols) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  long long best = 0;
  float bv = p[r * ldp];
  for (long long c = 1; c < cols; ++c) {
    const float v = p[r * ldp + c];
    if (v > bv) {  // first maximum wins, like tf.math.argmax
      bv = v;
      best = c;
    }
  }
  for (long long c = 0; c < cols; ++c) {
    const float v = (c == best) ? 1.f : 0.f;
    if (out16) out16[r * ldo + c] = f2bf(v);
    if (out32) out32[r * ldo32 + c] = v;
  }
}

// ------------------------------------------------------------------ losses
__device__ __forceinline__ float block_sum(float v) {
  __shared__ float sh[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  v = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.f;
  if (w == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  }
  return v;  // valid in thread 0
}

// Keras binary_crossentropy for a sigmoid output (logits form, see cellcomm_b200.h).
__global__ void bce_kernel(const float* __restrict__ x, long long ldx, long long rows,
                           int from_logits, float target, float inv_n,
                           float* __restrict__ loss_out, const Mat dz) {
  float acc = 0.f;
  for (long long r = threadIdx.x; r < rows; r += blockDim.x) {
    const float raw = x[r * ldx];
    float loss, p;
    if (from_logits) {
      // max(x,0) - x*t + log(1+exp(-|x|))   (tf.nn.sigmoid_cross_entropy_with_logits)
      loss = fmaxf(raw, 0.f) - raw * target + log1pf(expf(-fabsf(raw)));
      p = 1.f / (1.f + expf(-raw));
    } else {
      const float eps = 1e-7f;
      p = raw;
      const float q = fminf(fmaxf(raw, eps), 1.f - eps);
      loss = -(target * logf(q) + (1.f - target) * logf(1.f - q));
    }
    acc += loss;
    if (dz.p) store1(dz, r, 0, (p - target) * inv_n);
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) atomicAdd(loss_out, acc * inv_n);
}

// part == nullptr: every block adds its partial loss with an atomic (run-dependent order);
// else the blocks combine in fixed order like colreduce_kernel: partial to part[block], ticket,
// and the block with the last ticket sums part[] (thread t: blocks t, t + 256, ... in order,
// then the fixed block_sum tree), adds the total to loss_out and re-zeroes the ticket.
__global__ void mse_kernel(const Mat pred, const Mat target, long long rows, long long cols,
                           float inv_total, float* __restrict__ loss_out, const Mat dpred,
                           float* __restrict__ part, unsigned int* __restrict__ ticket) {
  float acc = 0.f;
  for_each_chunk8(rows, cols, [&](long long r, long long c0, int n) {
    float a[8], t[8];
    load8(pred, r, c0, n, a);
    load8(target, r, c0, n, t);
    float g[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float d = (i < n) ? a[i] - t[i] : 0.f;
      acc += d * d;
      g[i] = 2.f * d * inv_total;
    }
    if (dpred.p) store8(dpred, r, c0, n, g);
  });
  acc = block_sum(acc);
  if (part == nullptr) {
    if (threadIdx.x == 0) atomicAdd(loss_out, acc * inv_total);
    return;
  }
  __shared__ bool last;
  if (threadIdx.x == 0) {
    part[blockIdx.x] = acc;
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  float t = 0.f;
  for (unsigned i = threadIdx.x; i < gridDim.x; i += blockDim.x) t += __ldcg(part + i);
  t = block_sum(t);
  if (threadIdx.x == 0) {
    *loss_out += t * inv_total;
    *ticket = 0u;
  }
}

// ------------------------------------------------------------------ RMSprop (Keras, momentum>0)
__global__ void rmsprop_kernel(float* __restrict__ p32, bf16* __restrict__ p16,
                               const float* __restrict__ g, float* __restrict__ ms,
                               float* __restrict__ mom, long long rows, long long cols,
                               long long ld, float lr, float rho, float momentum, float eps,
                               float grad_scale) {
  const bool vec = (ld % 4 == 0) && ((((uintptr_t)p32) & 15) == 0) && ((((uintptr_t)g) & 15) == 0) &&
                   ((((uintptr_t)ms) & 15) == 0) && ((((uintptr_t)mom) & 15) == 0) &&
                   (p16 == nullptr || (((uintptr_t)p16) & 7) == 0);
  const long long cpr = (cols + 3) / 4;
  const long long total = rows * cpr;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cpr;
    const long long c0 = (i - r * cpr) * 4;
    const int n = (int)min((long long)4, cols - c0);
    const long long off = r * ld + c0;
    float w[4], gg[4], s[4], m[4];
    if (vec && n == 4) {
      float4 a = *reinterpret_cast<const float4*>(p32 + off);
      float4 b = *reinterpret_cast<const float4*>(g + off);
      float4 c = *reinterpret_cast<const float4*>(ms + off);
      float4 d = *reinterpret_cast<const float4*>(mom + off);
      w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
      gg[0] = b.x; gg[1] = b.y; gg[2] = b.z; gg[3] = b.w;
      s[0] = c.x; s[1] = c.y; s[2] = c.z; s[3] = c.w;
      m[0] = d.x; m[1] = d.y; m[2] = d.z; m[3] = d.w;
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k < n) {
          w[k] = p32[off + k];
          gg[k] = g[off + k];
          s[k] = ms[off + k];
          m[k] = mom[off + k];
        } else {
          w[k] = gg[k] = s[k] = m[k] = 0.f;
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = gg[k] * grad_scale;
      s[k] = rho * s[k] + (1.f - rho) * gk * gk;
      m[k] = momentum * m[k] + lr * gk * rsqrtf(s[k] + eps);
      w[k] -= m[k];
    }
    if (vec && n == 4) {
      *reinterpret_cast<float4*>(p32 + off) = make_float4(w[0], w[1], w[2], w[3]);
      *reinterpret_cast<float4*>(ms + off) = make_float4(s[0], s[1], s[2], s[3]);
      *reinterpret_cast<float4*>(mom + off) = make_float4(m[0], m[1], m[2], m[3]);
      if (p16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(w[0], w[1]);
        __nv_bfloat162 hi = __floats2bfloat162_rn(w[2], w[3]);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&lo);
        u.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(p16 + off) = u;
      }
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k < n) {
          p32[off + k] = w[k];
          ms[off + k] = s[k];
          mom[off + k] = m[k];
          if (p16) p16[off + k] = f2bf(w[k]);
        }
      }
    }
  }
}

}  // namespace cc

using namespace cc;

#define ST(s) ((cudaStream_t)(s))
#define F32(mask, bit) (((mask) >> (bit)) & 1)
#define EW_LAUNCH(kern, rows, cols, stream, ...)                                        \
  do {                                                                                  \
    if ((rows) <= 0 || (cols) <= 0) return 0;                                           \
    const long long _work = (long long)(rows) * (((cols) + 7) / 8);                     \
    kern<<<ew_grid(_work, 256), 256, 0, ST(stream)>>>(__VA_ARGS__);                     \
    CC_CHECK_LAUNCH();                                                                  \
    return 0;                                                                           \
  } while (0)

extern "C" int64_t cc_reduce_ws_floats(int64_t rows, int64_t cols) {
  // the largest need of any colreduce (two outputs) or MSE launch of at most rows x cols: the
  // slab count depends on the column-block count, so every column-block count up to cols'
  // is visited (multi-slab launches have fewer than 2 * SMs of them)
  if (rows <= 0 || cols <= 0) return 0;
  long long need = reduce_tickets() + mse_blocks(rows, cols);
  const long long gx_max = (cols + 127) / 128;
  for (long long gx = 1; gx <= gx_max && gx < reduce_tickets(); ++gx) {
    const long long n = colreduce_ws_floats(rows, gx == gx_max ? cols : gx * 128, 2);
    if (n > need) need = n;
  }
  return need;
}

extern "C" int cc_colsum(const void* x, int64_t ld, int64_t rows, int64_t cols, float* out,
                         int32_t beta, int32_t dtypes, cc_stream_t stream) {
  return cc_colsum_ws(x, ld, rows, cols, out, beta, dtypes, nullptr, 0, stream);
}

extern "C" int cc_colsum_ws(const void* x, int64_t ld, int64_t rows, int64_t cols, float* out,
                            int32_t beta, int32_t dtypes, float* ws, int64_t ws_floats,
                            cc_stream_t stream) {
  if (cols <= 0) return 0;
  if (rows <= 0) {
    if (!beta) {
      fill_f32_kernel<<<ew_grid(cols, 256), 256, 0, ST(stream)>>>(out, 0.f, cols);
      CC_CHECK_LAUNCH();
    }
    return 0;
  }
  return launch_colreduce<0>(mat(x, ld, F32(dtypes, 0)), mat(nullptr, 0, 0), rows, cols, nullptr,
                             nullptr, out, beta, ws, ws_floats, ST(stream));
}

extern "C" int cc_bias_grad(const void* dy, int64_t lddy, const void* y, int64_t ldy, int64_t rows,
                            int64_t cols, int32_t act, float* out, int32_t beta, void* dz,
                            int64_t lddz, void* dz_lo, int64_t lddz_lo, int32_t dtypes,
                            cc_stream_t stream) {
  return cc_bias_grad_ws(dy, lddy, y, ldy, rows, cols, act, out, beta, dz, lddz, dz_lo, lddz_lo,
                         dtypes, nullptr, 0, stream);
}

extern "C" int cc_bias_grad_ws(const void* dy, int64_t lddy, const void* y, int64_t ldy,
                               int64_t rows, int64_t cols, int32_t act, float* out, int32_t beta,
                               void* dz, int64_t lddz, void* dz_lo, int64_t lddz_lo,
                               int32_t dtypes, float* ws, int64_t ws_floats, cc_stream_t stream) {
  if (cols <= 0) return 0;
  CC_REQUIRE(out != nullptr || dz != nullptr, "cc_bias_grad: nothing to compute");
  CC_REQUIRE(dz_lo == nullptr || (dz != nullptr && !F32(dtypes, 2)),
             "cc_bias_grad: dz_lo needs a bf16 dz (the high-order term)");
  if (rows <= 0) {
    if (!beta && out != nullptr) {
      fill_f32_kernel<<<ew_grid(cols, 256), 256, 0, ST(stream)>>>(out, 0.f, cols);
      CC_CHECK_LAUNCH();
    }
    return 0;
  }
  return launch_colreduce<3>(mat(dy, lddy, F32(dtypes, 0)), mat(y, ldy, F32(dtypes, 1)), rows, cols,
                             nullptr, nullptr, out, beta, ws, ws_floats, ST(stream), act,
                             mat(dz, lddz, F32(dtypes, 2)), mat(dz_lo, lddz_lo, 0));
}

extern "C" int cc_split_bf16(const void* x, int64_t ldx, void* hi, int64_t ldhi, void* lo,
                             int64_t ldlo, int64_t rows, int64_t cols, int32_t dtypes,
                             cc_stream_t stream) {
  EW_LAUNCH(split_kernel, rows, cols, stream, mat(x, ldx, F32(dtypes, 0)), mat(hi, ldhi, 0),
            mat(lo, ldlo, 0), rows, cols);
}

extern "C" int cc_dropout(const void* x, int64_t ldx, void* out, int64_t ldo, int64_t rows,
                          int64_t cols, float rate, const uint8_t* mask_u8, int64_t ldm,
                          uint64_t seed, const uint64_t* counter_dev, uint32_t stream_id,
                          int32_t dtypes, cc_stream_t stream) {
  CC_REQUIRE(rate >= 0.f && rate < 1.f, "cc_dropout: rate %f out of range", rate);
  EW_LAUNCH(dropout_kernel, rows, cols, stream, mat(x, ldx, F32(dtypes, 0)),
            mat(out, ldo, F32(dtypes, 1)), rows, cols, rate, mask_u8, ldm, seed, counter_dev,
            stream_id);
}

extern "C" int cc_dropout_mask(uint8_t* mask_u8, int64_t ldm, int64_t rows, int64_t cols,
                               float rate, uint64_t seed, const uint64_t* counter_dev,
                               uint32_t stream_id, cc_stream_t stream) {
  EW_LAUNCH(dropout_mask_kernel, rows, cols, stream, mask_u8, ldm, rows, cols, rate, seed,
            counter_dev, stream_id);
}

extern "C" int cc_uniform(float* out32, void* out16, int64_t ld, int64_t rows, int64_t cols,
                          uint64_t seed, const uint64_t* counter_dev, uint32_t stream_id,
                          cc_stream_t stream) {
  EW_LAUNCH(uniform_kernel, rows, cols, stream, out32, (bf16*)out16, ld, rows, cols, seed,
            counter_dev, stream_id);
}

extern "C" int cc_counter_add(uint64_t* counter_dev, uint64_t inc, cc_stream_t stream) {
  counter_add_kernel<<<1, 1, 0, ST(stream)>>>(counter_dev, inc);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_act_bwd(const void* dy, int64_t lddy, const void* y, int64_t ldy, void* dz,
                          int64_t lddz, int64_t rows, int64_t cols, int32_t act, int32_t dtypes,
                          cc_stream_t stream) {
  EW_LAUNCH(act_bwd_kernel, rows, cols, stream, mat(dy, lddy, F32(dtypes, 0)),
            mat(y, ldy, F32(dtypes, 1)), mat(dz, lddz, F32(dtypes, 2)), rows, cols, act);
}

extern "C" int cc_copy2d(const void* src, int64_t lds, void* dst, int64_t ldd, int64_t rows,
                         int64_t cols, int32_t beta, float scale, int32_t dtypes,
                         cc_stream_t stream) {
  EW_LAUNCH(copy2d_kernel, rows, cols, stream, mat(src, lds, F32(dtypes, 0)),
            mat(dst, ldd, F32(dtypes, 1)), rows, cols, beta, scale);
}

extern "C" int cc_bn_stats(const void* x, int64_t ld, int64_t rows, int64_t cols, float* sums,
                           int32_t dtypes, cc_stream_t stream) {
  return cc_bn_stats_ws(x, ld, rows, cols, sums, dtypes, nullptr, 0, stream);
}

extern "C" int cc_bn_stats_ws(const void* x, int64_t ld, int64_t rows, int64_t cols, float* sums,
                              int32_t dtypes, float* ws, int64_t ws_floats, cc_stream_t stream) {
  if (cols <= 0) return 0;
  CC_REQUIRE(rows > 0, "cc_bn_stats: empty batch");
  return launch_colreduce<1>(mat(x, ld, F32(dtypes, 0)), mat(nullptr, 0, 0), rows, cols, nullptr,
                             nullptr, sums, 0, ws, ws_floats, ST(stream));
}

extern "C" int cc_bn_train_apply(const void* x, int64_t ldx, void* y, int64_t ldy, int64_t rows,
                                 int64_t cols, const float* sums, int64_t n_total,
                                 const float* gamma, const float* beta, float eps, float momentum,
                                 float* moving_mean, float* moving_var, float* save_mean,
                                 float* save_rstd, int32_t dtypes, cc_stream_t stream) {
  if (cols <= 0) return 0;
  CC_REQUIRE(n_total > 0, "cc_bn_train_apply: n_total must be positive");
  bn_finalize_kernel<<<(unsigned)((cols + 255) / 256), 256, 0, ST(stream)>>>(
      sums, cols, 1.0 / (double)n_total, eps, momentum, moving_mean, moving_var, save_mean,
      save_rstd);
  CC_CHECK_LAUNCH();
  EW_LAUNCH(bn_apply_kernel, rows, cols, stream, mat(x, ldx, F32(dtypes, 0)),
            mat(y, ldy, F32(dtypes, 1)), rows, cols, gamma, beta, save_mean, save_rstd, 0, eps);
}

extern "C" int cc_bn_infer(const void* x, int64_t ldx, void* y, int64_t ldy, int64_t rows,
                           int64_t cols, const float* gamma, const float* beta,
                           const float* moving_mean, const float* moving_var, float eps,
                           int32_t dtypes, cc_stream_t stream) {
  EW_LAUNCH(bn_apply_kernel, rows, cols, stream, mat(x, ldx, F32(dtypes, 0)),
            mat(y, ldy, F32(dtypes, 1)), rows, cols, gamma, beta, moving_mean, moving_var, 1, eps);
}

extern "C" int cc_bn_bwd_stats(const void* dy, int64_t lddy, const void* x, int64_t ldx,
                               int64_t rows, int64_t cols, const float* save_mean,
                               const float* save_rstd, float* sums2, int32_t dtypes,
                               cc_stream_t stream) {
  return cc_bn_bwd_stats_ws(dy, lddy, x, ldx, rows, cols, save_mean, save_rstd, sums2, dtypes,
                            nullptr, 0, stream);
}

extern "C" int cc_bn_bwd_stats_ws(const void* dy, int64_t lddy, const void* x, int64_t ldx,
                                  int64_t rows, int64_t cols, const float* save_mean,
                                  const float* save_rstd, float* sums2, int32_t dtypes, float* ws,
                                  int64_t ws_floats, cc_stream_t stream) {
  if (cols <= 0) return 0;
  CC_REQUIRE(rows > 0, "cc_bn_bwd_stats: empty batch");
  return launch_colreduce<2>(mat(dy, lddy, F32(dtypes, 0)), mat(x, ldx, F32(dtypes, 1)), rows, cols,
                             save_mean, save_rstd, sums2, 0, ws, ws_floats, ST(stream));
}

extern "C" int cc_bn_bwd_apply(const void* dy, int64_t lddy, const void* x, int64_t ldx, void* dx,
                               int64_t lddx, int64_t rows, int64_t cols, const float* gamma,
                               const float* save_mean, const float* save_rstd, const float* sums2,
                               int64_t n_total, float* dgamma, float* dbeta, int32_t dtypes,
                               cc_stream_t stream) {
  if (cols <= 0) return 0;
  if (dgamma || dbeta) {
    bn_param_grad_kernel<<<(unsigned)((cols + 255) / 256), 256, 0, ST(stream)>>>(sums2, cols,
                                                                                 dgamma, dbeta);
    CC_CHECK_LAUNCH();
  }
  if (dx == nullptr) return 0;
  EW_LAUNCH(bn_bwd_apply_kernel, rows, cols, stream, mat(dy, lddy, F32(dtypes, 0)),
            mat(x, ldx, F32(dtypes, 1)), mat(dx, lddx, F32(dtypes, 2)), rows, cols, gamma,
            save_mean, save_rstd, sums2, 1.f / (float)n_total);
}

extern "C" int cc_bn_infer_bwd(const void* dy, int64_t lddy, void* dx, int64_t lddx, int64_t rows,
                               int64_t cols, const float* gamma, const float* moving_var,
                               float eps, int32_t dtypes, cc_stream_t stream) {
  EW_LAUNCH(bn_infer_bwd_kernel, rows, cols, stream, mat(dy, lddy, F32(dtypes, 0)),
            mat(dx, lddx, F32(dtypes, 1)), rows, cols, gamma, moving_var, eps);
}

extern "C" int cc_softmax_fwd(const void* x, int64_t ldx, void* y, int64_t ldy, float* y32,
                              int64_t ldy32, int64_t rows, int64_t cols, int32_t dtypes,
                              cc_stream_t stream) {
  if (rows <= 0 || cols <= 0) return 0;
  softmax_fwd_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, ST(stream)>>>(
      mat(x, ldx, F32(dtypes, 0)), mat(y, ldy, F32(dtypes, 1)), y32, ldy32, rows, cols);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_softmax_bwd(const void* dy, int64_t lddy, const void* y, int64_t ldy, void* dx,
                              int64_t lddx, int64_t rows, int64_t cols, int32_t dtypes,
                              cc_stream_t stream) {
  if (rows <= 0 || cols <= 0) return 0;
  softmax_bwd_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, ST(stream)>>>(
      mat(dy, lddy, F32(dtypes, 0)), mat(y, ldy, F32(dtypes, 1)), mat(dx, lddx, F32(dtypes, 2)),
      rows, cols);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_bce_fwd_bwd(const float* x32, int64_t ldx, int64_t rows, int32_t from_logits,
                              float target, int64_t n_total, float* loss_out, void* dz,
                              int64_t lddz, int32_t dtypes, cc_stream_t stream) {
  CC_REQUIRE(rows > 0 && n_total > 0, "cc_bce_fwd_bwd: empty batch");
  bce_kernel<<<1, 256, 0, ST(stream)>>>(x32, ldx, rows, from_logits, target, 1.f / (float)n_total,
                                        loss_out, mat(dz, lddz, F32(dtypes, 0)));
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_mse_fwd_bwd(const void* pred, int64_t ldp, const void* target, int64_t ldt,
                              int64_t rows, int64_t cols, int64_t n_total, float* loss_out,
                              void* dpred, int64_t lddp, int32_t dtypes, cc_stream_t stream) {
  return cc_mse_fwd_bwd_ws(pred, ldp, target, ldt, rows, cols, n_total, loss_out, dpred, lddp,
                           dtypes, nullptr, 0, stream);
}

extern "C" int cc_mse_fwd_bwd_ws(const void* pred, int64_t ldp, const void* target, int64_t ldt,
                                 int64_t rows, int64_t cols, int64_t n_total, float* loss_out,
                                 void* dpred, int64_t lddp, int32_t dtypes, float* ws,
                                 int64_t ws_floats, cc_stream_t stream) {
  CC_REQUIRE(target != nullptr, "cc_mse_fwd_bwd: no target");
  if (rows <= 0 || cols <= 0) return 0;
  const float inv_total = 1.f / ((float)n_total * (float)cols);
  const long long blocks = mse_blocks(rows, cols);
  if (ws != nullptr) {
    const long long need = reduce_tickets() + blocks;
    CC_REQUIRE(ws_floats >= need,
               "cc_mse_fwd_bwd_ws of [%lld, %lld]: workspace of %lld floats, needs %lld "
               "(cc_reduce_ws_floats)", (long long)rows, (long long)cols, (long long)ws_floats,
               need);
  }
  mse_kernel<<<(unsigned)blocks, 256, 0, ST(stream)>>>(
      mat(pred, ldp, F32(dtypes, 0)), mat(target, ldt, F32(dtypes, 1)), rows, cols, inv_total,
      loss_out, mat(dpred, lddp, F32(dtypes, 2)), ws ? ws + reduce_tickets() : nullptr,
      reinterpret_cast<unsigned int*>(ws));
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_round_half_even(const void* x, int64_t ldx, void* out, int64_t ldo, float* out32,
                                  int64_t ldo32, int64_t rows, int64_t cols, int32_t dtypes,
                                  cc_stream_t stream) {
  EW_LAUNCH(round_kernel, rows, cols, stream, mat(x, ldx, F32(dtypes, 0)),
            mat(out, ldo, F32(dtypes, 1)), out32, ldo32, rows, cols);
}

extern "C" int cc_argmax_onehot(const float* p32, int64_t ldp, void* out16, int64_t ldo,
                                float* out32, int64_t ldo32, int64_t rows, int64_t cols,
                                cc_stream_t stream) {
  if (rows <= 0 || cols <= 0) return 0;
  argmax_onehot_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, ST(stream)>>>(
      p32, ldp, (bf16*)out16, ldo, out32, ldo32, rows, cols);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_rmsprop_step(float* p32, void* p16, const float* g, float* ms, float* mom,
                               int64_t rows, int64_t cols, int64_t ld, float lr, float rho,
                               float momentum, float eps, float grad_scale, cc_stream_t stream) {
  if (rows <= 0 || cols <= 0) return 0;
  const long long work = (long long)rows * ((cols + 3) / 4);
  // CC_RMS_BLOCKS_PER_SM (default 8 = full occupancy): a smaller value leaves thread slots for
  // GEMM CTAs when the sweep runs on the side stream next to the following forward pass
  static int bps = 0;
  if (bps == 0) {
    const char* v = getenv("CC_RMS_BLOCKS_PER_SM");
    bps = v ? atoi(v) : 8;
    if (bps < 1 || bps > 8) bps = 8;
  }
  long long blocks = (work + 255) / 256;
  if (blocks > (long long)num_sms() * bps) blocks = (long long)num_sms() * bps;
  rmsprop_kernel<<<(unsigned)blocks, 256, 0, ST(stream)>>>(p32, (bf16*)p16, g, ms, mom, rows,
                                                             cols, ld, lr, rho, momentum, eps,
                                                             grad_scale);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_bias_act(const float* bias, int32_t act, void* out16, int64_t ld16, float* out32,
                           int64_t ld32, int64_t rows, int64_t cols, cc_stream_t stream) {
  if (rows <= 0 || cols <= 0) return 0;
  bias_act_kernel<<<ew_grid(rows * cols, 256), 256, 0, ST(stream)>>>(bias, act, (bf16*)out16, ld16,
                                                                    out32, ld32, rows, cols);
  CC_CHECK_LAUNCH();
  return 0;
}

extern "C" int cc_fill_f32(float* dst, float value, int64_t n, cc_stream_t stream) {
  if (n <= 0) return 0;
  fill_f32_kernel<<<ew_grid(n, 256), 256, 0, ST(stream)>>>(dst, value, n);
  CC_CHECK_LAUNCH();
  return 0;
}
