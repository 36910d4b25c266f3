/*
 * cellcomm_b200.h — C ABI of libcellcomm_b200.so
 *
 * The reference (mikemey/cellcomm) has no FFI/plugin interface: its hot path is
 * Python calling tensorflow==2.4.0 Keras (requirements.txt:3).  This header is
 * the boundary this repo introduces *underneath* the unchanged Python surface
 * (SURVEY.md §8b): each entry point names the reference call it replaces.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, no torch types.
 *  - every call returns int: 0 = ok, <0 = error; cc_last_error() gives the text
 *    (thread-local).
 *  - device pointers are owned by the caller (torch's allocator in this repo).
 *    The library allocates only inside opaque handles with an explicit
 *    *_destroy, and inside host-side cc_coo/cc_csr objects.
 *  - every device call is asynchronous on the cudaStream_t passed (as void*),
 *    never synchronises, and is CUDA-graph capturable.
 *  - 2-D device tensors are row-major with an explicit leading dimension `ld`
 *    in ELEMENTS; bf16 tensors consumed by cc_gemm need ld % 8 == 0 and a
 *    16-byte aligned base (TMA constraint).
 */
#ifndef CELLCOMM_B200_H
#define CELLCOMM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* cc_stream_t; /* cudaStream_t */

/* ------------------------------------------------------------------ misc */
const char* cc_last_error(void);
int cc_version(void);
/* number of kernels this library has launched in this process (bench.py's
 * gpu_launches claim) */
long long cc_launch_count(void);
/* compiled-for architecture string, e.g. "sm_100a" */
const char* cc_arch(void);
/* The library reads its tuning / debug environment variables (CC_GEMM_*) once, at the first
 * cc_gemm call; this makes the next call read them again (tests and sweep tools that change
 * them at run time). */
void cc_reload_env(void);

/* ------------------------------------------------- loader (host, no GPU)
 * replaces: load_matrix()  src/cell_type_training.py:9-17
 *   pd.read_csv(skiprows=3, delim_whitespace=True, names=[gene,barcode,p])
 *   .pivot_table(index=barcode, columns=gene, values=p, fill_value=0)
 * Semantics (SURVEY.md App. A.1): skip exactly 3 lines, ignore the dims line,
 * rows = distinct barcode ids ascending, cols = distinct gene ids ascending,
 * duplicate (gene,barcode) entries averaged in float64, explicit zeros keep
 * their row/column alive.
 */
typedef struct cc_csr cc_csr; /* opaque host CSR */

int cc_mtx_load_csr(const char* path, cc_csr** out);
/* build the same CSR from in-memory COO triplets (1-based ids as in the file) */
int cc_coo_to_csr(const int64_t* gene, const int64_t* barcode, const double* val,
                  int64_t nnz, cc_csr** out);
void cc_csr_destroy(cc_csr* csr);
int64_t cc_csr_rows(const cc_csr* csr);
int64_t cc_csr_cols(const cc_csr* csr);
int64_t cc_csr_nnz(const cc_csr* csr);
/* host views, valid until cc_csr_destroy */
const int64_t* cc_csr_rowptr(const cc_csr* csr);   /* rows+1 */
const int32_t* cc_csr_colidx(const cc_csr* csr);   /* nnz, compact column index, ascending per row */
const float* cc_csr_values(const cc_csr* csr);     /* nnz, float32(mean as float64) */
const double* cc_csr_values64(const cc_csr* csr);  /* nnz, the float64 means (DataFrame dtype) */
const int64_t* cc_csr_row_ids(const cc_csr* csr);  /* rows, original barcode ids */
const int64_t* cc_csr_col_ids(const cc_csr* csr);  /* cols, original gene ids */

/* The file's triplets in FILE ORDER (one threaded parse shared with cc_mtx_load_csr).
 * replaces: load_file(matrix_file, ..., skip=3) + the per-line walk of convert_matrix()
 *   src/intercepts/import_barcodes.py:4-11,14-45,76 -- cells are runs of equal barcode ids in
 *   file order, genes are listed in first-seen order, so the importer needs the file order
 *   that the CSR no longer has. */
typedef struct cc_coo cc_coo; /* opaque host triplets */
int cc_mtx_load_coo(const char* path, cc_coo** out);
void cc_coo_destroy(cc_coo* coo);
int64_t cc_coo_nnz(const cc_coo* coo);
/* host views, valid until cc_coo_destroy */
const int64_t* cc_coo_gene(const cc_coo* coo);    /* nnz, 1-based gene line numbers */
const int64_t* cc_coo_barcode(const cc_coo* coo); /* nnz, 1-based barcode line numbers */
const double* cc_coo_value(const cc_coo* coo);    /* nnz */
/* the CSR of load_matrix() from already parsed triplets (no second read of the file) */
int cc_coo_build_csr(const cc_coo* coo, cc_csr** out);

/* --------------------------------------------------- batch gather (device)
 * replaces: DataFrame.sample(B) dense row gather, src/cell_type_training.py:37-38,
 * and the DataFrame -> float32 tensor feed of train_on_batch/predict.
 * row_idx_dev != NULL: output row i is CSR row row_idx_dev[i] (sampled batch);
 * row_idx_dev == NULL: output row i is CSR row row_start + i (encode-all pass).
 * out16/out32 may each be NULL.  Columns [0, n_cols) of every output row are written (zeros
 * where the CSR has no entry); the padding columns [n_cols, ld) are not touched, so an output
 * may be a column slice of a wider buffer.
 */
int cc_gather_rows(const int64_t* rowptr_dev, const int32_t* colidx_dev, const float* values_dev,
                   const int64_t* row_idx_dev, int64_t row_start, int64_t n_rows, int64_t n_cols,
                   void* out16, int64_t ld16, float* out32, int64_t ld32, cc_stream_t stream);

/* ------------------------------------------------------------- dense GEMM
 * replaces: layers.Dense forward/backward inside Model.train_on_batch /
 * Model.predict (src/bigan_classify.py:10-75,144-155; src/bigan_cont.py:7-41).
 *
 * D[M,N] = epilogue( sum_s A_s[M,K_s] * B_s[K_s,N] ), bf16 operands, fp32
 * accumulation in tensor memory (tcgen05).  Up to CC_GEMM_MAX_SEG (A_s,B_s) segments
 * accumulate into one tile: that is how Concatenate() is consumed without
 * materialising it.
 *
 * a_mn_major = 0: A_s is stored [M, K_s] row-major (K contiguous)
 *            = 1: A_s is stored [K_s, M] row-major (M contiguous)
 * b_mn_major = 0: B_s is stored [N, K_s] row-major (K contiguous)
 *            = 1: B_s is stored [K_s, N] row-major (N contiguous)
 *
 * epilogue, per element (r,c), v = acc:
 *   v = alpha * v
 *   if bias:   v += bias[c]
 *   act:       0 none, 1 sigmoid, 2 relu
 *   if dact:   v *= act'(y[r,c])   (1: y(1-y)  2: y>0)   y = dact_y (bf16)
 *   if out32:  out32[r,c] = v + (beta32 ? out32[r,c] : 0)
 *   if out16:  out16[r,c] = bf16(v + (beta16 ? out16[r,c] : 0))
 *   if rms_p32: fused RMSprop update of the parameter block with gradient v (see below)
 */
enum { CC_ACT_NONE = 0, CC_ACT_SIGMOID = 1, CC_ACT_RELU = 2 };
#define CC_GEMM_MAX_SEG 4

typedef struct cc_gemm_desc {
  int32_t M, N;
  int32_t a_mn_major, b_mn_major;
  int32_t nseg;
  const void* a[CC_GEMM_MAX_SEG];
  int64_t lda[CC_GEMM_MAX_SEG];
  const void* b[CC_GEMM_MAX_SEG];
  int64_t ldb[CC_GEMM_MAX_SEG];
  int32_t k[CC_GEMM_MAX_SEG];
  /* epilogue */
  float alpha;
  const float* bias;
  int32_t act;
  const void* dact_y;
  int64_t ld_dact;
  int32_t dact;
  void* out16;
  int64_t ld16;
  int32_t beta16;
  float* out32;
  int64_t ld32;
  int32_t beta32;
  /* split-K scratch (fp32), may be NULL => no split-K */
  float* workspace;
  int64_t workspace_elems;
  /* tuning / debug overrides, 0 = automatic */
  int32_t force_splits;
  int32_t force_bn;
  /* optional fused optimiser (weight-gradient GEMMs): when rms_p32 != NULL the epilogue
   * treats v as the gradient of the [M,N] parameter block at rms_p32 (leading dimension
   * rms_ld, shared by rms_ms / rms_mom / rms_p16) and applies Keras RMSprop(momentum)
   * in place -- ms = rho*ms + (1-rho) v^2; mom = momentum*mom + lr*v/sqrt(ms+eps);
   * w -= mom; p16 = bf16(w) -- so the gradient never round-trips through HBM
   * (optimizers.RMSprop, src/bigan_classify.py:88).  out32/out16 stay optional. */
  float* rms_p32;
  float* rms_ms;
  float* rms_mom;
  void* rms_p16;
  int64_t rms_ld;
  float rms_lr, rms_rho, rms_momentum, rms_eps;
  /* optional routed fp32 output (data-parallel weight-gradient GEMMs): the GEMM itself performs
   * the reduce-scatter's data movement.  The output lies in a gradient bucket of the flat
   * parameter layout that is sharded evenly over route_world ranks; element `rel` (offset from
   * the bucket start, = route_off0 + row*ld32 + col) belongs to rank rel / route_shard and is
   * stored to route_base[owner] + rel -- this rank's slot in the OWNER's staging buffer, a
   * peer-mapped pointer over NVLink (the own share goes to local memory).  out32 must be set
   * (it is the local address of element (0,0)); beta32 and split-K are not available. */
  int32_t route_world;   /* 0: off */
  int64_t route_shard;   /* elements per rank, multiple of 8 */
  int64_t route_off0;    /* offset of out32[0,0] from the bucket start, multiple of 4 */
  float* route_base[16];
  /* optional second bf16 output: the low-order term bf16(v - float(bf16(v))) of a two-term
   * expansion whose high-order term is out16 (fp32 activations that the next Dense consumes
   * as hi + lo GEMM segments: the producer writes both, no cc_split_bf16 pass).  Needs out16,
   * beta16 == 0. */
  void* out16_lo;
  int64_t ld16_lo;
  /* optional BLOCKED layout of the fused optimiser's fp32 state (rms_blocked != 0; weight-
   * gradient GEMMs with N > 128 only).  rms_p32 / rms_ms / rms_mom then point at the LAYER's
   * arrays (not at this GEMM's row slice), stored as 32-row x 32-column blocks of 4 KB: layer
   * element (r, c) lives at
   *     ((r / 32) * (rms_ld / 32) + c / 32) * 1024 + ((c % 32) / 4) * 128 + (r % 32) * 4 + c % 4
   * floats (rms_ld % 32 == 0; the arrays hold ceil(rows / 32) * 32 rows), which is the order a
   * warp receives its accumulators from tensor memory, so that every access of the epilogue is
   * 512 contiguous bytes and each 32 x 32 chunk one DRAM-page-local 4 KB block per array.
   * rms_row0 is the layer row of this GEMM's row 0 (the row offset of a Concatenate segment;
   * any value >= 0).  rms_p16 (the bf16 compute copy, a TMA operand elsewhere) and out32 stay
   * row-major views of this GEMM's own [M, N] slice. */
  int32_t rms_blocked;
  int32_t rms_row0;
  /* blocked layout only, optional: the low-order bf16 term bf16(w - float(bf16(w))) of the
   * updated weights, row-major [M, N] with leading dimension rms_ld like rms_p16 (kernels the
   * forward GEMMs consume as hi + lo segments; replaces a cc_split_bf16 pass over the layer) */
  void* rms_p16_lo;
} cc_gemm_desc;

int cc_gemm(const cc_gemm_desc* desc, cc_stream_t stream);
/* how many fp32 workspace elements cc_gemm may want for this shape */
int64_t cc_gemm_workspace_elems(int32_t M, int32_t N);

/* Layer-level wrappers (Keras kernel layout W[in,out], row-major, bf16):
 *   fwd  : Y[M,N]   = act(sum_s X_s[M,K_s] W[roff_s : roff_s+K_s, :] + b)
 *   dgrad: dX[M,K]  = (sum_s dZ_s[M,N_s] W_s[roff_s : roff_s+K, :]^T) * act'(y)
 *   wgrad: dW[K,N]  = X[M,K]^T dZ[M,N]       (fp32 out)
 * They fill a cc_gemm_desc and call cc_gemm; see gemm_api.cu.
 */
int cc_dense_fwd(int32_t M, int32_t N, int32_t nseg, const void* const* x, const int64_t* ldx,
                 const int32_t* k, const void* const* w, const int64_t* ldw, const float* bias,
                 int32_t act, void* out16, int64_t ld16, float* out32, int64_t ld32,
                 float* workspace, int64_t workspace_elems, cc_stream_t stream);
int cc_dense_dgrad(int32_t M, int32_t K, int32_t nseg, const void* const* dz, const int64_t* lddz,
                   const int32_t* n, const void* const* w, const int64_t* ldw, const void* dact_y,
                   int64_t ld_dact, int32_t dact, float alpha, void* out16, int64_t ld16,
                   int32_t beta16, float* workspace, int64_t workspace_elems, cc_stream_t stream);
int cc_dense_wgrad(int32_t M, int32_t K, int32_t N, const void* x, int64_t ldx, const void* dz,
                   int64_t lddz, float* dw, int64_t lddw, int32_t beta, cc_stream_t stream);

/* --------------------------------------------------------- tail kernels
 * All elementwise / reduction kernels below work on row-major [rows, cols]
 * tensors with explicit ld.  Activation-like operands are bf16 OR fp32: the
 * trailing `dtypes` bitmask has bit i set when the i-th such operand (in the
 * order listed beside each function) is fp32.  Activations that feed a
 * BatchNormalization and all activation gradients are kept in fp32 (1/sigma
 * amplification and the cancellation in BN backward make bf16 storage too
 * lossy there, DESIGN.md "precision policy"); GEMM operands are bf16.
 */

/* Fixed-order (deterministic) column reductions and MSE loss.
 * cc_colsum, cc_bias_grad, cc_bn_stats, cc_bn_bwd_stats and cc_mse_fwd_bwd combine the partial
 * sums of their CTAs with float atomics, so the last bits of a result depend on scheduling.
 * Each has a `_ws` sibling taking `float* ws, int64_t ws_floats` before the stream:
 *  - ws == NULL: the atomic path (what the plain entry point does).
 *  - ws != NULL: every CTA stores its partials to ws, and the CTA that finishes last sums them
 *    in a fixed order (row slab 0, 1, ... / block 0, 1, ...).  No CTA waits for another.
 *    Results are bit-identical for identical inputs and launch geometry (same shapes and SM
 *    count).  The same launch geometry is used as on the atomic path, and no zero-fill launch
 *    precedes a multi-slab call with beta == 0.
 * Workspace contract: ws holds ws_floats floats, at least cc_reduce_ws_floats(rows, cols) for
 * any call of at most rows x cols; a smaller one fails (cc_last_error), never falls back to
 * atomics.  Its leading counters must be zero before the first use (zero the whole buffer
 * once); every call leaves them zero again, also across CUDA-graph replays.  One workspace per
 * stream: two reductions that may run at the same time must not share one. */
int64_t cc_reduce_ws_floats(int64_t rows, int64_t cols);

/* column sums into fp32: db = sum_rows dZ (Dense bias grad).  dtypes: x */
int cc_colsum(const void* x, int64_t ld, int64_t rows, int64_t cols, float* out, int32_t beta,
              int32_t dtypes, cc_stream_t stream);
int cc_colsum_ws(const void* x, int64_t ld, int64_t rows, int64_t cols, float* out, int32_t beta,
                 int32_t dtypes, float* ws, int64_t ws_floats, cc_stream_t stream);

/* Dense bias gradient from the fp32 upstream gradient: out[c] = sum_r dy[r,c]*act'(y[r,c]).
 * (Summing the bf16 dZ instead loses the near-cancelling sums of biases that feed a
 * BatchNormalization.)  dz (optional, NULL to skip): also write dz[r,c] = dy*act'(y), the
 * operand of the wgrad / dgrad GEMMs, in the same pass (replaces a cc_act_bwd launch for
 * trained layers).  dz_lo (optional, with a bf16 dz): also write the low-order term
 * bf16(dz - float(bf16(dz))) of the two-term expansion (layers whose dz feeds the GEMMs as
 * hi + lo: one launch instead of cc_act_bwd + cc_split_bf16 + cc_bias_grad).  out may be NULL
 * (frozen layers: only dz is wanted).  beta != 0: out += the sums (the caller zeroed a whole
 * bias region with one fill instead of one per layer).  dtypes: dy, y, dz */
int cc_bias_grad(const void* dy, int64_t lddy, const void* y, int64_t ldy, int64_t rows,
                 int64_t cols, int32_t act, float* out, int32_t beta, void* dz, int64_t lddz,
                 void* dz_lo, int64_t lddz_lo, int32_t dtypes, cc_stream_t stream);
int cc_bias_grad_ws(const void* dy, int64_t lddy, const void* y, int64_t ldy, int64_t rows,
                    int64_t cols, int32_t act, float* out, int32_t beta, void* dz, int64_t lddz,
                    void* dz_lo, int64_t lddz_lo, int32_t dtypes, float* ws, int64_t ws_floats,
                    cc_stream_t stream);
/* hi = bf16(x), lo = bf16(x - hi): two-term bf16 expansion of an activation, fed to cc_gemm
 * as two accumulating segments where 8 mantissa bits are too few.  dtypes: x */
int cc_split_bf16(const void* x, int64_t ldx, void* hi, int64_t ldhi, void* lo, int64_t ldlo,
                  int64_t rows, int64_t cols, int32_t dtypes, cc_stream_t stream);

/* Dropout (layers.Dropout, training=True): out = x * keep / (1-rate).
 * mask_u8 != NULL: explicit keep mask (parity tests inject TF's masks this way).
 * mask_u8 == NULL: keep = philox(seed, *counter_dev, stream_id, r, c) >= rate;
 * the same call with the same arguments regenerates the mask in backward.
 * dtypes: x, out */
int cc_dropout(const void* x, int64_t ldx, void* out, int64_t ldo, int64_t rows, int64_t cols,
               float rate, const uint8_t* mask_u8, int64_t ldm, uint64_t seed,
               const uint64_t* counter_dev, uint32_t stream_id, int32_t dtypes,
               cc_stream_t stream);
/* write the keep mask the RNG path would use (tests / debugging) */
int cc_dropout_mask(uint8_t* mask_u8, int64_t ldm, int64_t rows, int64_t cols, float rate,
                    uint64_t seed, const uint64_t* counter_dev, uint32_t stream_id,
                    cc_stream_t stream);
/* uniform [0,1) floats: tf.random.uniform (src/bigan_basic.py:36-37, bigan_cont.py:52-53) */
int cc_uniform(float* out32, void* out16, int64_t ld, int64_t rows, int64_t cols, uint64_t seed,
               const uint64_t* counter_dev, uint32_t stream_id, cc_stream_t stream);
int cc_counter_add(uint64_t* counter_dev, uint64_t inc, cc_stream_t stream);

/* dz = dy * act'(y)  (act: 0 copy, 1 sigmoid, 2 relu).  dtypes: dy, y, dz */
int cc_act_bwd(const void* dy, int64_t lddy, const void* y, int64_t ldy, void* dz, int64_t lddz,
               int64_t rows, int64_t cols, int32_t act, int32_t dtypes, cc_stream_t stream);

/* dst (+)= scale * src on a [rows, cols] block: concat materialisation, slicing, gradient
 * accumulation (beta=1) and bf16<->fp32 casts.  dtypes: src, dst */
int cc_copy2d(const void* src, int64_t lds, void* dst, int64_t ldd, int64_t rows, int64_t cols,
              int32_t beta, float scale, int32_t dtypes, cc_stream_t stream);

/* BatchNormalization (Keras 2.4 defaults: eps=1e-3, momentum=0.99), SURVEY A.3.
 * stats: sums[0:cols] = sum_r x, sums[cols:2cols] = sum_r x^2 (fp32, overwritten).
 * The caller may all-reduce `sums` across ranks before cc_bn_train_apply.  dtypes: x */
int cc_bn_stats(const void* x, int64_t ld, int64_t rows, int64_t cols, float* sums,
                int32_t dtypes, cc_stream_t stream);
int cc_bn_stats_ws(const void* x, int64_t ld, int64_t rows, int64_t cols, float* sums,
                   int32_t dtypes, float* ws, int64_t ws_floats, cc_stream_t stream);
/* y = gamma*(x-mean)*rstd+beta with batch stats from sums/n_total; writes
 * mean/rstd (fp32, cols each) for backward; updates moving stats:
 * moving = momentum*moving + (1-momentum)*batch (biased variance).  dtypes: x, y */
int cc_bn_train_apply(const void* x, int64_t ldx, void* y, int64_t ldy, int64_t rows,
                      int64_t cols, const float* sums, int64_t n_total, const float* gamma,
                      const float* beta, float eps, float momentum, float* moving_mean,
                      float* moving_var, float* save_mean, float* save_rstd, int32_t dtypes,
                      cc_stream_t stream);
/* inference: y = gamma*(x-moving_mean)/sqrt(moving_var+eps)+beta.  dtypes: x, y */
int cc_bn_infer(const void* x, int64_t ldx, void* y, int64_t ldy, int64_t rows, int64_t cols,
                const float* gamma, const float* beta, const float* moving_mean,
                const float* moving_var, float eps, int32_t dtypes, cc_stream_t stream);
/* backward, training mode.  sums2[0:cols] = sum dy, sums2[cols:2cols] = sum dy*xhat.
 * dtypes: dy, x */
int cc_bn_bwd_stats(const void* dy, int64_t lddy, const void* x, int64_t ldx, int64_t rows,
                    int64_t cols, const float* save_mean, const float* save_rstd, float* sums2,
                    int32_t dtypes, cc_stream_t stream);
int cc_bn_bwd_stats_ws(const void* dy, int64_t lddy, const void* x, int64_t ldx, int64_t rows,
                       int64_t cols, const float* save_mean, const float* save_rstd,
                       float* sums2, int32_t dtypes, float* ws, int64_t ws_floats,
                       cc_stream_t stream);
/* dx = gamma*rstd*(dy - sum_dy/n - xhat*sum_dyxhat/n); dgamma = sum_dyxhat, dbeta = sum_dy
 * (dgamma/dbeta may be NULL when the BN is not being trained; dx may be NULL).
 * dtypes: dy, x, dx */
int cc_bn_bwd_apply(const void* dy, int64_t lddy, const void* x, int64_t ldx, void* dx,
                    int64_t lddx, int64_t rows, int64_t cols, const float* gamma,
                    const float* save_mean, const float* save_rstd, const float* sums2,
                    int64_t n_total, float* dgamma, float* dbeta, int32_t dtypes,
                    cc_stream_t stream);
/* backward through an inference-mode (frozen) BN: dx = dy*gamma/sqrt(var+eps).  dtypes: dy, dx */
int cc_bn_infer_bwd(const void* dy, int64_t lddy, void* dx, int64_t lddx, int64_t rows,
                    int64_t cols, const float* gamma, const float* moving_var, float eps,
                    int32_t dtypes, cc_stream_t stream);

/* softmax over the last axis (classify encoder, src/bigan_classify.py:39).  dtypes: x, y */
int cc_softmax_fwd(const void* x, int64_t ldx, void* y, int64_t ldy, float* y32, int64_t ldy32,
                   int64_t rows, int64_t cols, int32_t dtypes, cc_stream_t stream);
/* dtypes: dy, y, dx */
int cc_softmax_bwd(const void* dy, int64_t lddy, const void* y, int64_t ldy, void* dx,
                   int64_t lddx, int64_t rows, int64_t cols, int32_t dtypes, cc_stream_t stream);

/* losses.binary_crossentropy on the (rows,1) discriminator output against a
 * constant target (0.95 / 0: src/bigan_classify.py:128-129).  Keras 2.4 uses the
 * logits of the producing Sigmoid op (sigmoid_cross_entropy_with_logits), so the
 * input is the PRE-activation (from_logits=1); from_logits=0 takes probabilities
 * and clips them to [1e-7, 1-1e-7] (Keras backend epsilon).
 * loss_out[0] += sum_r bce_r / n_total;  dz = dLoss/dlogit = (sigmoid(x)-t)/n_total
 * (may be NULL).  n_total is the GLOBAL batch so sharded batches sum to the
 * global mean.  dtypes: dz */
int cc_bce_fwd_bwd(const float* x32, int64_t ldx, int64_t rows, int32_t from_logits, float target,
                   int64_t n_total, float* loss_out, void* dz, int64_t lddz, int32_t dtypes,
                   cc_stream_t stream);
/* losses.mse: mean over all rows*cols elements; dpred = 2*(pred-target)/(n_total*cols)
 * (may be NULL).  dtypes: pred, target, dpred */
int cc_mse_fwd_bwd(const void* pred, int64_t ldp, const void* target, int64_t ldt, int64_t rows,
                   int64_t cols, int64_t n_total, float* loss_out, void* dpred, int64_t lddp,
                   int32_t dtypes, cc_stream_t stream);
int cc_mse_fwd_bwd_ws(const void* pred, int64_t ldp, const void* target, int64_t ldt,
                      int64_t rows, int64_t cols, int64_t n_total, float* loss_out, void* dpred,
                      int64_t lddp, int32_t dtypes, float* ws, int64_t ws_floats,
                      cc_stream_t stream);

/* tf.math.round (half to even) for generate_cells, src/bigan_basic.py:40-44 */
/* dtypes: x, out */
int cc_round_half_even(const void* x, int64_t ldx, void* out, int64_t ldo, float* out32,
                       int64_t ldo32, int64_t rows, int64_t cols, int32_t dtypes,
                       cc_stream_t stream);
/* to_categorical(argmax(p,-1)): src/bigan_classify.py:121-124 */
int cc_argmax_onehot(const float* p32, int64_t ldp, void* out16, int64_t ldo, float* out32,
                     int64_t ldo32, int64_t rows, int64_t cols, cc_stream_t stream);

/* Keras RMSprop with momentum (optimizers.RMSprop(lr=0.0075, rho=0.85,
 * momentum=0.1), src/bigan_classify.py:88; SURVEY A.6):
 *   ms  = rho*ms + (1-rho)*g^2 ; mom = momentum*mom + lr*g/sqrt(ms+eps) ; w -= mom
 * Works on a [rows, cols] view with leading dimensions so that padded weight
 * matrices can be updated in place; p16 (bf16 compute copy) may be NULL. */
int cc_rmsprop_step(float* p32, void* p16, const float* g, float* ms, float* mom, int64_t rows,
                    int64_t cols, int64_t ld, float lr, float rho, float momentum, float eps,
                    float grad_scale, cc_stream_t stream);

/* ---- data-parallel optimiser step over NVLink peer memory (csrc/peer_optimizer.cu) --------
 * One process per GPU on one node; every rank's flat gradient buffer and bf16 weight buffer
 * are mapped into every process (torch symmetric memory / CUDA IPC does the mapping, the
 * library only sees device pointers).  cc_peer_rmsprop fuses
 *     reduce-scatter (P2P loads) -> Keras RMSprop on this rank's shard -> all-gather of the
 *     bf16 weights (P2P stores)
 * for the element range [start, start+count) of the flat buffers.  The reference has no
 * counterpart (single process); under data parallelism this is the gradient exchange around
 * `optimizer.apply_gradients` of src/bigan_classify.py:88,144-155.
 *   grad[q], p16[q] : rank q's buffers (q < world), the same flat layout on every rank
 *   broadcast = 1   : sharded update, bf16 result stored to all ranks;
 *   broadcast = 0   : replicated update (biases / BN parameters): every rank updates the
 *                     whole range from the sum of all gradients, local stores only
 *   ready[q]        : LOCAL flags; the kernel starts once ready[q] >= epoch for all q
 *   grad[q]         : in the push design (cc_gemm_desc.route_*) these are this rank's LOCAL
 *                     staging slots, already filled by every rank's wgrad GEMM epilogues
 * cc_peer_signal stores `value` to n remote/local flags after a system-scope fence (everything
 * the stream did before is visible to the peers first); cc_peer_wait blocks the stream until
 * n consecutive local flags are >= value.  Epochs are compared modulo 2^32; every entry point
 * accepts a device counter `epoch_ctr` that is added to the host-side value (NULL: none). */
#define CC_PEER_MAX 16
typedef struct cc_peer_rmsprop_desc {
  int32_t world, rank;
  const float* grad[CC_PEER_MAX];
  void* p16[CC_PEER_MAX];
  float* p32;
  float* ms;
  float* mom;
  int64_t start, count;
  int32_t broadcast;
  float lr, rho, momentum, eps;
  const uint32_t* ready;
  uint32_t epoch;
  /* optional device-resident epoch base: effective epoch = epoch + *epoch_ctr.  With it the
   * whole step (hand-shakes included) can be captured in a CUDA graph: every replay sees the
   * counter the previous update left behind (cc_peer_wait(bump = 1) / cc_peer_allreduce
   * advance it). NULL: epoch is the host's value. */
  const uint32_t* epoch_ctr;
  /* optional NVLS multicast address of the bf16 weight buffer (NVSwitch multimem mapping of
   * the same symmetric allocation): with broadcast = 1 ONE multimem.st per 16 bytes delivers
   * the updated weights to every rank, instead of world P2P stores (7/8 less NVLink egress
   * for the all-gather at 8 GPUs).  NULL: P2P stores. */
  void* p16_multicast;
  /* optional low-order bf16 term (kernels kept as hi + lo, see cc_split_bf16): for elements of
   * the flat ranges [lo_begin[k], lo_end[k]), k < 2, the kernel also delivers
   * bf16(w - float(bf16(w))) to every rank's p16lo buffer (p16lo_multicast when non-NULL).
   * p16lo[0] == NULL: off. */
  void* p16lo[CC_PEER_MAX];
  void* p16lo_multicast;
  int64_t lo_begin[2], lo_end[2];
} cc_peer_rmsprop_desc;
int cc_peer_rmsprop(const cc_peer_rmsprop_desc* desc, cc_stream_t stream);
int cc_peer_signal(uint32_t* const* targets, int32_t n, uint32_t value,
                   const uint32_t* epoch_ctr, cc_stream_t stream);
int cc_peer_wait(const uint32_t* flags, int32_t n, uint32_t value, uint32_t* epoch_ctr,
                 int32_t bump, cc_stream_t stream);
/* In-place sum all-reduce of n <= cap floats over peer memory in one kernel (BatchNorm batch
 * statistics, BN-backward sums, loss buffer).  slots[q]: rank q's [2][world][cap] staging array,
 * flags[q]: rank q's [world] flags (both peer-mapped); epoch grows by one per call, identically
 * on every rank.  Sums in rank order, so every rank gets bit-identical results. */
int cc_peer_allreduce(float* data, int32_t n, int32_t world, int32_t rank, float* const* slots,
                      uint32_t* const* flags, int64_t cap, uint32_t epoch, uint32_t* epoch_ctr,
                      cc_stream_t stream);

/* Dense layer with zero input width: y[r,c] = act(bias[c]).  The reference's 5-gene fixture
 * produces Dense(0) layers (int(5*0.1) == 0; src/bigan_cont.py:8,29) whose consumers see K=0. */
int cc_bias_act(const float* bias, int32_t act, void* out16, int64_t ld16, float* out32,
                int64_t ld32, int64_t rows, int64_t cols, cc_stream_t stream);

/* fp32 scalar helpers */
int cc_fill_f32(float* dst, float value, int64_t n, cc_stream_t stream);

/* ------------------------------------------------ encode-all-cells pass (one call)
 * replaces: BasicBiGan.encoding_prediction(trainer.data) = encoder.predict(all cells)
 *   src/bigan_basic.py:29-30, called from src/intercepts/db_recorder.py:85 (and the
 *   plot / .enc interceptors): Keras runs it 32 rows at a time on the dense DataFrame.
 * Here: for every tile of `tile_rows` cells of rows [row_begin, row_end) of the device CSR --
 * cc_gather_rows into slot 0, then the encoder's layers in inference mode as the op list below
 * -- enqueued on `stream` from this one call.  out32: [row_end - row_begin, Z] fp32, leading
 * dimension ld_out.  Rows shard over GPUs by giving each rank its own [row_begin, row_end).
 *
 * The encoder is a small program over scratch slots (slot 0 = the gathered bf16 cell tile,
 * slot -1 = the output tile): the caller derives it from its layer graph, so both reference
 * encoders (src/bigan_cont.py:28-41, src/bigan_classify.py:28-40) run through the same entry
 * point.  Slot s is a [tile_rows, pad64(slot_width[s])] bf16 (or fp32) tile carved out of
 * `scratch` (zero-initialised by the caller once; cc_encode_scratch_bytes gives its size). */
#define CC_ENC_MAX_OPS 32
#define CC_ENC_MAX_SLOTS 32
enum {
  CC_ENC_DENSE = 0,    /* out = act(sum_s in[s] @ w16[w_row[s] : w_row[s]+width(in[s]), :] + bias) */
  CC_ENC_SPLIT = 1,    /* fp32 in[0] -> bf16 hi (out) + lo (out2): two-term GEMM operand */
  CC_ENC_COPY = 2,     /* out = in[0] (dtype cast as the slots say) */
  CC_ENC_BN_INFER = 3, /* BatchNormalization on the moving statistics */
  CC_ENC_SOFTMAX = 4   /* out = softmax(in[0]); the fp32 result also goes to the output tile */
};
typedef struct cc_enc_op {
  int32_t kind;
  int32_t n_in;
  int32_t in[CC_GEMM_MAX_SEG];
  int32_t w_row[CC_GEMM_MAX_SEG]; /* DENSE: first kernel row of each input segment */
  int32_t out, out2;
  int32_t width;                  /* DENSE: output width N */
  int32_t act;                    /* DENSE: cc_act */
  const void* w16;                /* DENSE: bf16 kernel [K_total, width], leading dimension ldw */
  int64_t ldw;
  const float* bias;
  const float *gamma, *beta, *mean, *var; /* BN_INFER */
  float eps;
} cc_enc_op;
typedef struct cc_encode_plan {
  int32_t n_cols;    /* gene_size */
  int32_t tile_rows; /* cells per tile */
  int32_t n_slots, n_ops;
  int32_t slot_width[CC_ENC_MAX_SLOTS];
  int32_t slot_fp32[CC_ENC_MAX_SLOTS];
  cc_enc_op ops[CC_ENC_MAX_OPS];
  void* scratch;
  int64_t scratch_bytes;
  float* workspace; /* split-K scratch for cc_gemm (may be NULL) */
  int64_t workspace_elems;
} cc_encode_plan;
int64_t cc_encode_scratch_bytes(const cc_encode_plan* plan);
int cc_encode_stream(const int64_t* rowptr_dev, const int32_t* colidx_dev, const float* values_dev,
                     int64_t row_begin, int64_t row_end, const cc_encode_plan* plan, float* out32,
                     int64_t ld_out, cc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CELLCOMM_B200_H */
