/*
 * pipegcn_b200 -- C ABI of the B200-native PipeGCN hot path (libpipegcn_b200.so).
 *
 * The reference (GATECH-EIC/PipeGCN @ 73ab949) is pure Python; it has no FFI.  Its
 * plug-in seam is a set of Python objects (helper/context.py:4-5, module/layer.py:8).
 * These entry points are what a ctypes binding of those objects calls; each one
 * names the reference code it replaces.  All pointers are raw device pointers
 * unless stated otherwise, every call is asynchronous on `stream`
 * (a cudaStream_t passed as void*), never synchronises the host, and returns 0 on
 * success or a negative pg_status; pg_last_error() describes the last failure of
 * the calling thread.  The caller owns all memory.
 */
#ifndef PIPEGCN_B200_H
#define PIPEGCN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG_ABI_VERSION 2

/* element types of activations / gradients */
#define PG_F32  0
#define PG_BF16 1

enum pg_status {
  PG_OK = 0,
  PG_ERR_INVALID = -1,      /* bad argument (null pointer, misaligned, unsupported width) */
  PG_ERR_CUDA = -2,         /* a CUDA runtime/driver call failed */
  PG_ERR_UNSUPPORTED = -3,  /* not available on this device / build */
  PG_ERR_TIMEOUT = -4       /* a halo flag did not arrive within the spin bound */
};

int pg_abi_version(void);
const char* pg_last_error(void);
/* writes sm major*10+minor, SM count and L2 bytes of `device`; needs a GPU */
int pg_device_info(int device, int* sm_arch, int* sm_count, int64_t* l2_bytes);
/* tuning knobs (process-wide; the defaults are the measured best, the other values keep earlier code paths selectable):
 * "agg_impl" = 1 | 2 | 3 (row-per-group, chunked, chunked + cp.async long rows); "agg_unroll" = 4 | 8 neighbour rows in
 * flight per lane group; "agg_pack_short" = 0 | 1; "agg_occ" = 4 | 5; "agg_overlap" = 0 | 1 (short rows on a side
 * stream); "agg_narrow" = 0 | 1 (sub-warp kernels for rows of <= 16 vectors); "agg_l2_hint" = 0 | 1;
 * "ln_stage" = 0 | 1 | 2 (LayerNorm rows through the cp.async ring: never / one vector per lane / always);
 * "ce_subwarp" = 0 | 1 (several cross-entropy rows per warp); "gemm_epi_batch" = 0 | 1, "gemm_epi_slabs" = 1 | 2
 * (GEMM epilogue: TMEM loads of a chunk batched, staging slabs per warp).  Unknown names return PG_ERR_INVALID. */
int pg_set_option(const char* name, int value);

/* ------------------------------------------------------------------------------------------
 * Adjacency of one partition in CSR form plus the split of its long rows.
 * Forward: rows = destination (`_V`) nodes, columns = source (`_U`) ids  (layer.py:47-49).
 * Backward: rows = source ids, columns = destinations (DGL gspmm backward on the reversed graph).
 * Rows with more than seg_len entries are cut into segments of seg_len that different
 * warps reduce into fp32 partials; a fix-up pass sums the partials in segment order, so the
 * result does not depend on scheduling.
 * ---------------------------------------------------------------------------------------- */
typedef struct pg_csr {
  const int32_t* indptr;        /* [n_rows + 1] */
  const int32_t* indices;       /* [nnz] */
  int32_t n_rows;
  int32_t seg_len;              /* > 0 */
  int32_t n_long;               /* rows longer than seg_len */
  int32_t n_seg;                /* total segments of the long rows */
  const int32_t* long_row;      /* [n_long] row id */
  const int32_t* long_seg_ptr;  /* [n_long + 1] first segment of every long row */
  const int32_t* seg_long;      /* [n_seg] index into long_row */
  const int32_t* row_order;     /* [n_rows] processing order of the rows (e.g. by falling degree), or NULL */
  int64_t nnz;                  /* number of entries (indptr[n_rows]); selects the short-row kernel shape */
  /* chunked walk (optional, chunks == NULL selects the row-per-group kernel): the rows in processing order
   * (falling length) with their entries stored contiguously, cut into chunks one warp processes */
  const int32_t* chunks;        /* [n_chunks][4] = {first entry in pidx, n, item, kind | n_rows << 2}:
                                 *   kind 0: n_rows whole rows of n entries each (n_rows * n <= 32), item = first row in prow
                                 *   kind 1: one row of n entries, item = its position in prow
                                 *   kind 2: one segment (n entries) of a long row, item = segment index (scratch slot) */
  int32_t n_chunks;
  int32_t n_chunks_long;        /* the kind 2 and kind 1 chunks come first: chunks [0, n_chunks_long) */
  const int32_t* pidx;          /* [nnz] column ids, rows concatenated in processing order; bit 31 set = "hot" source
                                 * row (referenced often): loaded with an L2 evict_last policy */
  const int32_t* prow;          /* [n_rows] row id of every position of the processing order */
} pg_csr;

/*
 * Dropout (model.py:47) without a stored mask: keep(element) is a pure function of (seed, step, element index), where
 * step = *step_dev + step_off is an epoch counter that lives on the device (CUDA-graph replay).  Every kernel that
 * writes a tensor the next layer consumes can apply it on the way out, so no [num_all, d] dropout pass is needed:
 * the LayerNorm epilogue (inner rows), the halo push (the receiver's halo rows, receiver's row index), and the
 * transposed aggregate / fix-up (the gradient of the dropped tensor).  p == 0 or a NULL pointer: no dropout.
 */
typedef struct pg_drop {
  float p;
  uint64_t seed;
  const uint32_t* step_dev;   /* may be NULL: the mask does not depend on a step */
  int32_t step_off;
} pg_drop;

/*
 * Neighbour aggregate (SURVEY.md K6/K7/K11):
 *   out[r, 0:d] = ( sum_{e in row r} x[indices[e], 0:d] ) / row_div[r]  ( + out[r, 0:d] if r < acc_rows )
 * x and out have element type `dtype`, sums are fp32.  ldx/ldo are row strides in elements.
 * row_div (fp32, [n_rows]) may be NULL (no division); the division is one IEEE reciprocal per row and a multiply per
 * element (within 1 ulp of `/`).  scratch: fp32 [n_seg * d_pad] where
 * d_pad = d rounded up to 8; may be NULL when n_seg == 0.
 * Replaces graph['_E'].update_all(fn.copy_src, fn.sum) and `/ degs` at
 * /root/reference/module/layer.py:47-50, and their autograd.
 */
int pg_aggregate(const pg_csr* g, const void* x, int64_t ldx, void* out, int64_t ldo, int32_t d, int dtype,
                 const float* row_div, int32_t acc_rows, float* scratch, void* stream);
/* the same, with the dropout mask of `drop` applied to every output row as it is written (the backward of
 * `layer(dropout(F))`: out = mask * ((A^T g) (+ out)) / (1 - p)); element index = row * ceil(d / vec) + vector */
int pg_aggregate_drop(const pg_csr* g, const void* x, int64_t ldx, void* out, int64_t ldo, int32_t d, int dtype,
                      const float* row_div, int32_t acc_rows, float* scratch, const pg_drop* drop, void* stream);

/* out[r, 0:d] = x[r, 0:d] / row_div[r]   (gradient of `/ degs`, layer.py:50) */
int pg_row_div(const void* x, int64_t ldx, void* out, int64_t ldo, int32_t n_rows, int32_t d, int dtype,
               const float* row_div, void* stream);

/*
 * Dense part of the layer on the tcgen05 tensor cores (SURVEY.md K8/K10):
 *   c[m, n] = sum_s a_s[m, k_s] * b_s[n, k_s]^T  (+ bias[n])  (/ row_div[m])      1 <= n_src <= 6
 * dtype_in PG_BF16 -> kind::f16 MMA, PG_F32 -> kind::tf32 MMA; fp32 accumulation in TMEM;
 * dtype_out selects the element type of c.  n <= 256.  All operands row-major with 16-byte
 * aligned rows (TMA); k tails and the m tail are zero-filled / masked.  `srcs` is a HOST array.
 * Replaces `self.linear1(feat[0:num_dst]) + self.linear2(ah)` at
 * /root/reference/module/layer.py:51 (two pairs: inner rows x W1, neighbour mean x W2,
 * bias = b1 + b2) and, with one pair, the dX products of its autograd (row_div = in_deg fuses the
 * `/ degs` gradient).  fp32 parity mode passes the hi/lo halves of pg_split_tf32 as three pairs
 * per product (hi*hi + hi*lo + lo*hi: the "3xTF32" product, fp32-grade accuracy).
 */
typedef struct pg_gemm_src {
  const void* a;   /* [m, k] */
  int64_t lda;
  const void* b;   /* [n, k] */
  int64_t ldb;
  int32_t k;
} pg_gemm_src;

int pg_linear(int dtype_in, int dtype_out, const pg_gemm_src* srcs, int32_t n_src, const float* bias,
              const float* row_div, void* c, int64_t ldc, int32_t m, int32_t n, void* stream);
/* the same with the dropout mask of `drop` applied to c as it is written; c's row 0 is row drop_row0 of the tensor the
 * mask is defined on (the gradient of a dropped tensor produced by a GEMM: transform-first layers) */
int pg_linear_drop(int dtype_in, int dtype_out, const pg_gemm_src* srcs, int32_t n_src, const float* bias,
                   const float* row_div, void* c, int64_t ldc, int32_t m, int32_t n, const pg_drop* drop,
                   int64_t drop_row0, void* stream);

/*
 * Weight gradients on the tcgen05 tensor cores (MN-major operands, split-K over the rows, deterministic):
 *   out[n, k] = sum_s sum_m a_s[m, n] * b_s[m, k]        n, k <= 256, fp32 output, 1 <= n_src <= 6
 * a_s = upstream gradient g [m, n], b_s = layer input [m, k], both row-major with 16-byte aligned rows; `srcs[s].k`
 * is ignored.  Replaces the autograd of /root/reference/module/layer.py:51 for the weights: gW1 = g^T feat[:N_in],
 * gW2 = g^T ah (one call each; three pairs per call for the split-fp32 product).  `workspace`: fp32 scratch of
 * pg_wgrad_workspace(m, n, k, dtype_in) floats for the split-K partials.
 */
int64_t pg_wgrad_workspace(int32_t m, int32_t n, int32_t k, int dtype_in);
int pg_wgrad(int dtype_in, const pg_gemm_src* srcs, int32_t n_src, float* out, int64_t ldo, int32_t m, int32_t n,
             int32_t k, float* workspace, int64_t workspace_floats, void* stream);

/* hi = x with the 13 low mantissa bits cleared (a tf32 value), lo = x - hi (exact); [rows, d] fp32 */
int pg_split_tf32(const float* x, int64_t ldx, float* hi, float* lo, int64_t ld, int32_t rows, int32_t d,
                  void* stream);

/* ------------------------------------------------------------------------------------------
 * Row-wise epilogues of the layer loop (model.py:53-56, train.py:320,351).  One warp per row, every tensor
 * read once and written once; column reductions are two-stage (`partial`: fp32 scratch of
 * pg_row_grid(n_rows) * 3 * d floats for the LayerNorm backward, pg_row_grid(n) * max(c, 1) for the loss).
 * ---------------------------------------------------------------------------------------- */
int pg_row_grid(int32_t n_rows);
/* out = keep ? x / (1 - p) : 0 with keep a pure function of (seed, element index) -- the backward calls it again on
 * the gradient with the same seed instead of storing a mask (dropout of model.py:47; in place allowed) */
int pg_dropout(const void* x, int64_t ldx, void* out, int64_t ldo, int32_t n_rows, int32_t d, int dtype, float p,
               uint64_t seed, const uint32_t* step_dev, void* stream);
/* the same with the general mask key: rows are numbered from row0 (a slice of a larger tensor) */
int pg_dropout_rows(const void* x, int64_t ldx, void* out, int64_t ldo, int64_t row0, int32_t n_rows, int32_t d, int dtype,
                    const pg_drop* drop, void* stream);
/* out = relu?(LayerNorm(y) * gamma + beta), mean/rstd [n_rows] kept for the backward; d % (16/elem) == 0 */
int pg_ln_relu_fwd(const void* y, int64_t ldy, const float* gamma, const float* beta, float eps, int relu,
                   void* out, int64_t ldo, float* mean, float* rstd, int32_t n_rows, int32_t d, int dtype,
                   void* stream);
/* the same with the next layer's dropout fused: `out` receives dropout(result) (what the next layer's aggregate and
 * GEMM read), `out_clean` the result itself (what the halo push sends and the backward needs) */
int pg_ln_relu_drop_fwd(const void* y, int64_t ldy, const float* gamma, const float* beta, float eps, int relu,
                        void* out, int64_t ldo, void* out_clean, int64_t ldc, float* mean, float* rstd, int32_t n_rows,
                        int32_t d, int dtype, const pg_drop* drop, void* stream);
/* g_y, dgamma[d], dbeta[d] and colsum[d] = column sums of g_y (the bias gradient of the producing linear) */
int pg_ln_relu_bwd(const void* g_out, int64_t ldg, const void* out, int64_t ldo, const void* y, int64_t ldy,
                   const float* mean, const float* rstd, const float* gamma, int relu, void* g_y, int64_t ldgy,
                   float* dgamma, float* dbeta, float* colsum, float* partial, int32_t n_rows, int32_t d,
                   int dtype, void* stream);
/* the same; with beta given the ReLU mask is recomputed from y (the forward's expression) and `out` is not read */
int pg_ln_relu_bwd2(const void* g_out, int64_t ldg, const void* out, int64_t ldo, const void* y, int64_t ldy,
                    const float* mean, const float* rstd, const float* gamma, const float* beta, int relu, void* g_y,
                    int64_t ldgy, float* dgamma, float* dbeta, float* colsum, float* partial, int32_t n_rows, int32_t d,
                    int dtype, void* stream);
/* loss[0] = sum_rows (logsumexp(z) - z[label]) over the first n_rows rows: CrossEntropyLoss(reduction='sum') */
int pg_ce_fwd(const void* z, int64_t ld, const int64_t* labels, int32_t n_rows, int32_t c, int dtype, float* lse,
              float* partial, float* loss, void* stream);
/* g[r] = (softmax(z[r]) - onehot) * upstream[0] for r < n_rows, 0 for n_rows <= r < n_total; colsum[c] optional */
int pg_ce_bwd(const void* z, int64_t ld, const int64_t* labels, const float* lse, const float* upstream,
              int32_t n_rows, int32_t n_total, int32_t c, int dtype, void* g, int64_t ldg, float* colsum,
              float* partial, void* stream);

/*
 * Multi-label targets (BCEWithLogitsLoss, f1_score(average='micro'): train.py:11-17,317-318) are bit-packed:
 * ybits is uint32 [rows, lw] with lw >= ceil(c / 32), label j of a row is bit j % 32 of word j / 32, bits >= c are 0.
 * Logit (and gradient) rows must be 16-byte aligned with ld >= c; any c >= 1 (rows wider than 512 fp32 / 1024 bf16
 * classes are processed in column chunks of that width).  Outside that: PG_ERR_INVALID.
 */
/* loss[0] = sum_{r < n_rows, j < c} max(z, 0) - z * y + log1p(exp(-|z|)), fp32, deterministic;
 * partial: pg_row_grid(n_rows) * max(c, 1) floats of scratch */
int pg_bce_fwd(const void* z, int64_t ld, const uint32_t* ybits, int32_t lw, int32_t n_rows, int32_t c, int dtype,
               float* partial, float* loss, void* stream);
/* g[r] = (sigmoid(z[r]) - y[r]) * upstream[0] for r < n_rows, 0 for n_rows <= r < n_total; colsum[c] (optional) = the
 * column sums of g as stored; partial: pg_row_grid(n_total) * c floats */
int pg_bce_bwd(const void* z, int64_t ld, const uint32_t* ybits, int32_t lw, const float* upstream, int32_t n_rows,
               int32_t n_total, int32_t c, int dtype, void* g, int64_t ldg, float* colsum, float* partial, void* stream);
/* counts[0..2] += micro TP, FP, FN of the prediction z > 0 over the rows rows[0..n) (int32 ids into z and ybits; NULL:
 * rows 0..n); integer adds, deterministic.  The caller zeroes counts. */
int pg_f1_counts(const void* z, int64_t ld, const uint32_t* ybits, int32_t lw, const int32_t* rows, int32_t n, int32_t c,
                 int dtype, unsigned long long* counts, void* stream);

/* ------------------------------------------------------------------------------------------
 * Halo exchange (feature_buffer.py:165-194).  One descriptor per message of a launch; the
 * array lives in device memory and is built once by Buffer.init_buffer.
 * A message copies n_rows rows of `src` (gathered through idx, or contiguous from src_row0)
 * to `dst` -- normally peer memory mapped over NVLink.  With `ema` set the sender first
 * updates its fp32 mirror  ema <- m*ema + (1-m)*row  (feature_buffer.py:189-191) and ships
 * the smoothed row.  When the last CTA of a message has stored its rows it publishes `value`
 * to *flag with system-scope release semantics.
 * ---------------------------------------------------------------------------------------- */
typedef struct pg_msg {
  const int32_t* idx;      /* [n_rows] source row ids, or NULL */
  int64_t src_row0;        /* first source row when idx == NULL */
  int32_t n_rows;
  int32_t cta_begin;       /* first CTA of this message inside the launch (filled by the host) */
  void* dst;               /* destination of row 0 */
  int64_t ld_dst;          /* elements */
  float* ema;              /* [n_rows, ld_ema] fp32 sender-side EMA mirror, or NULL */
  int64_t ld_ema;
  uint32_t* flag;          /* flag word to publish (peer memory), or NULL */
  uint32_t* counter;       /* local arrival counter of this message (self resetting) */
  int64_t dst_row0;        /* row index of `dst` inside the receiver's tensor (key of the receiver's dropout mask) */
} pg_msg;

/* rows per CTA used by pg_halo_push when the host fills cta_begin */
int pg_push_rows_per_cta(void);

/* momentum = m and one_minus = (float)(1 - m) evaluated in double precision by the caller, exactly the two
 * scalars of `t *= m; t += (1 - m) * recv` (feature_buffer.py:190-191) */
/* the flag value published is `value` (+ *value_dev when value_dev != NULL: an epoch counter that lives on the
 * device, so that a captured CUDA graph of an epoch can be replayed) */
int pg_halo_push(const pg_msg* msgs, int32_t n_msgs, int32_t n_ctas, const void* src, int64_t ld_src, int32_t d,
                 int dtype, float momentum, float one_minus, uint32_t value, const uint32_t* value_dev, void* stream);
/* the same with the RECEIVER's dropout applied to every row as it is stored into peer memory (after the EMA, whose
 * mirror stays clean): the halo rows arrive as the rows of dropout(cat(feat, halo)) the receiver will consume */
int pg_halo_push_drop(const pg_msg* msgs, int32_t n_msgs, int32_t n_ctas, const void* src, int64_t ld_src, int32_t d,
                      int dtype, float momentum, float one_minus, uint32_t value, const uint32_t* value_dev,
                      const pg_drop* drop, void* stream);

/*
 * Block the stream until every flags[i] >= value (acquire, system scope).  A bounded spin:
 * after `timeout_ms` the kernel stores PG_ERR_TIMEOUT to *status (device word, may be NULL)
 * and returns, so a dead peer cannot hang the GPU (the reference hangs in gloo wait(),
 * feature_buffer.py:184).  wait_ns (device word, may be NULL): the nanoseconds (%globaltimer) this launch
 * spent blocked are ADDED to it -- the exposed communication time of comm_timer.py:17-27, readable after
 * a region of CUDA-graph replays where host-recorded events are not available.
 */
int pg_halo_wait(const uint32_t* const* flags, int32_t n_flags, uint32_t value, const uint32_t* value_dev,
                 int32_t timeout_ms, int32_t* status, uint64_t* wait_ns, void* stream);

/*
 * Static-layer-0 shortcut: dst[r, 0:d] = c * src[r, 0:d] with c = 0 for k <= 0, else 1 (corr == 0) or
 * 1 - m^k (corr != 0), k = k_host (+ *k_dev).  The input features never change, so the halo rows of layer 0 after
 * k EMA updates of feature_buffer.py:186-191 are the closed form (1 - m^k) * x of the one-shot exchanged rows.
 */
int pg_scale_rows(const void* src, int64_t ld_src, void* dst, int64_t ld_dst, int32_t n_rows, int32_t d, int dtype,
                  float momentum, int corr, int32_t k_host, const uint32_t* k_dev, void* stream);

/*
 * grad[urow[i], 0:d] += sum_k recv[usrc[k], 0:d]  for k in [uptr[i], uptr[i+1]), in that order
 * (peers ascending), replacing the per-peer loop at feature_buffer.py:208-217.
 */
int pg_boundary_add(void* grad, int64_t ld_grad, const void* recv, int64_t ld_recv, int32_t d, int dtype,
                    const int32_t* urow, const int32_t* uptr, const int32_t* usrc, int32_t n_urow, void* stream);

/* ------------------------------------------------------------------------------------------
 * Symmetric heap: device memory that peers map through CUDA IPC (host pointers out).
 * ---------------------------------------------------------------------------------------- */
#define PG_IPC_HANDLE_BYTES 64
int pg_heap_alloc(size_t bytes, void** ptr);
int pg_heap_free(void* ptr);
int pg_ipc_export(void* ptr, unsigned char* handle);
int pg_ipc_import(const unsigned char* handle, void** ptr);
int pg_ipc_close(void* ptr);
int pg_enable_peer_access(int peer_device);

#ifdef __cplusplus
}
#endif
#endif /* PIPEGCN_B200_H */
