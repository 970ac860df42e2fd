/*
 * rsb.h — C ABI of the B200-native CTR hot path (librsb.so).
 *
 * Drop-in boundary for chenxing1999/recsys-benchmark: these are the entry
 * points a Python/ctypes (or any FFI) binding behind the reference's
 * IEmbedding plugin API (src/models/embeddings/base.py:8-20) and its
 * DeepFM / DCN_Mix models (src/models/deepfm.py:79-105, src/models/dcn.py:76-96,
 * src/models/layer_dcn.py:8-115) calls.  Every function cites the reference
 * interface it replaces.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, no torch / C++ types.
 *  - all data pointers are DEVICE pointers on the current CUDA device unless
 *    the parameter name starts with `h_` (host).
 *  - `stream` is a cudaStream_t passed as void*.  Nothing synchronises the
 *    host; nothing allocates or frees; scratch memory is a caller-provided
 *    workspace sized by the matching `*_workspace_bytes` query.
 *  - return value: 0 = ok, 1..9999 = cudaError_t of the failed launch,
 *    >= 10000 = rsb_status.  No exception crosses this ABI.
 *  - floating point is fp32, row ids are int64 (or int32 where stated).
 */
#ifndef RSB_H_
#define RSB_H_

#include <stdint.h>

#if defined(__GNUC__)
#define RSB_API __attribute__((visibility("default")))
#else
#define RSB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  RSB_OK = 0,
  RSB_ERR_BAD_ARG = 10001,     /* null pointer / negative size / unknown enum */
  RSB_ERR_UNSUPPORTED = 10002, /* row width outside the kernels' range (see rsb_row_width_supported) */
  RSB_ERR_WORKSPACE = 10003    /* workspace too small */
} rsb_status;

/* Which lightweight-embedding variant is applied INSIDE the gather. */
typedef enum {
  RSB_KIND_VANILLA = 0,  /* VanillaEmbedding            src/models/embeddings/base.py:23-75          */
  RSB_KIND_QR_MULT = 1,  /* QRHashingEmbedding "mult"   src/models/embeddings/qr_embedding.py:95-109 */
  RSB_KIND_QR_ADD = 2,   /*                   "add"                                                  */
  RSB_KIND_QR_CAT = 3,   /*                   "cat" (concat on the FIELD axis, like the reference)   */
  RSB_KIND_PEP = 4,      /* PepEmbeeding soft threshold src/models/embeddings/pep_embedding.py:82-92 */
  RSB_KIND_MASK = 5,     /* RetrainPepEmbedding / RetrainOptEmbed: weight * bool mask
                            pep_embedding.py:215-221 ; deepfm_opt_embed.py:693-706                   */
  RSB_KIND_OPTEMBED = 6  /* OptEmbed supernet training  deepfm_opt_embed.py:219-226 ; optembed_utils.py:101-104 */
} rsb_kind;

/* PEP threshold shapes (pep_embedding.py:94-117): value of `aux_mode` for RSB_KIND_PEP. */
typedef enum {
  RSB_PEP_GLOBAL = 0,     /* s[1]    */
  RSB_PEP_DIMENSION = 1,  /* s[D]    */
  RSB_PEP_FEATURE = 2,    /* s[N,1]  */
  RSB_PEP_FEATURE_DIM = 3 /* s[N,D]  */
} rsb_pep_threshold;

/* What the segmented reduction does with each unique row's summed gradient. */
typedef enum {
  RSB_APPLY_DENSE = 0,       /* dst[row,:] = sum  (dst is a zero-filled dense [N,E] grad:
                                aten embedding_dense_backward semantics, base.py:53-57)             */
  RSB_APPLY_SPARSE_ADAM = 1, /* torch.optim.SparseAdam row update (src/models/deepfm.py:173-184;
                                torch/optim/_functional.py:24-84)                                    */
  RSB_APPLY_SPARSE_SGD = 2,  /* sparse SGD, p += -lr*g (src/models/deepfm.py:203-216)              */
  RSB_APPLY_SHARD_ATOMIC = 3 /* (internal to rsb_segment_scatter_shards) vector atomic add into the owner's shard */
} rsb_apply;

RSB_API const char* rsb_version(void);
/* Human-readable text for a non-zero return value (cudaGetErrorString for CUDA codes). */
RSB_API const char* rsb_error_string(int code);
/* Number of kernels this library has launched in this process (bench.py's `gpu_launches`). */
RSB_API int64_t rsb_launch_count(void);
/* 1 if a row of `width` floats (16-byte aligned when width % 4 == 0) is handled. */
RSB_API int rsb_row_width_supported(int32_t width);

/* ------------------------------------------------------------------------
 * Forward: fused gather (+ variant transform) (+ FM second order + first order).
 *
 * Replaces, in one launch: `x + offsets` (deepfm.py:88 / dcn.py:84),
 * IEmbedding.forward (F.embedding call sites base.py:75, qr_embedding.py:99-107,
 * pep_embedding.py:82-89,215-221, deepfm_opt_embed.py:219-226,704),
 * the EmbeddingBag first-order term + bias (deepfm.py:49,95) and the FM
 * interaction (deepfm.py:91-92,98).
 *
 *  idx        [B,F] per-field ids, int32 if idx_is_i32 else int64
 *  offsets    [F] int64 field offsets added to idx, or NULL (ids already global)
 *  D          embedding width (num_factor).  QR_CAT: out is [B,2F,D/2]
 *  table      main table [n_rows, E]   (QR: emb2 [(N-1)/divider+1, E])
 *  table1     QR only: emb1 [divider, E]; divider = QR divider
 *  aux        PEP: s ; MASK: uint8/bool mask [n_rows,D] ; OPTEMBED: t_param [F] or NULL (mask-E off)
 *  aux_mode   PEP: rsb_pep_threshold ; OPTEMBED: norm (1 or 2) ; QR kinds: if > 0, the modulus of the
 *             remainder index (i1 = id % aux_mode, i2 = id / divider): CERP's bucket size
 *             (src/models/embeddings/cerp_embedding.py:142-153); 0 = divider (plain QR)
 *  mask_d_idx OPTEMBED: int64 [B,F] draw of torch.randint(0,D) (dims 0..k kept) or NULL
 *  fc, bias   first-order weights [N_global,1] and bias [1]; NULL -> no FM head (DCN-Mix)
 *  out_emb    [B,F,D] fp32 (always written)
 *  out_yfm    [B]  y_fm = first order + 0.5*sum_d((sum_f e)^2 - sum_f e^2), or NULL
 *  out_sum    [B,E] S = sum_f e, saved for the backward, or NULL
 *  out_rows   [B,F] int64 global row ids (idx + offsets), or NULL
 *  err_flag   device int32, set to 1 when an id is out of [0, n_global) (the read is
 *             clamped to row 0 instead of faulting; torch raises IndexError there)
 *  n_global   number of addressable ids (sum(field_dims)); for non-QR kinds == n_rows
 * ---------------------------------------------------------------------- */
RSB_API int rsb_lookup_fwd(int32_t kind, const void* idx, int32_t idx_is_i32, const int64_t* offsets,
                   int64_t B, int32_t F, int32_t D,
                   const float* table, int64_t n_rows, int64_t n_global,
                   const float* table1, int64_t divider,
                   const void* aux, int32_t aux_mode, const int64_t* mask_d_idx,
                   const float* fc, const float* bias,
                   float* out_emb, float* out_yfm, float* out_sum, int64_t* out_rows,
                   int32_t* err_flag, float* amax_slots, void* stream);
/* amax_slots (optional, NULL = off): device array of RSB_LOOKUP_AMAX_SLOTS zero-initialised floats; every warp raises
 * one slot to the largest |out_emb| it wrote, so max(amax_slots) == max |out_emb| - the bound the dense tail's FP16X2
 * operand split needs (rsb_absmax over the slots), without another pass over the [B, F*D] activation. */
#define RSB_LOOKUP_AMAX_SLOTS 1024

/* ------------------------------------------------------------------------
 * Backward, stage 1: per-lookup row gradients.
 *
 * g_out[b,f,:] = g_deep[b,f,:] + g_yfm[b] * (S[b,:] - emb[b,f,:])   (autograd of deepfm.py:91-102)
 * then the variant's chain rule, written as one compact row per lookup:
 *   VANILLA   rg_main = g_out
 *   MASK      rg_main = g_out * mask[row]
 *   QR_MULT   rg_main(emb2) = g_out * emb1[i1] ; rg_aux(emb1) = g_out * emb2[i2]
 *   QR_ADD    rg_main = rg_aux = g_out (rg_aux may be NULL: same array)
 *   QR_CAT    rg_aux = g_out[:, :F] ; rg_main = g_out[:, F:]
 *   PEP       rg_main = g_out * 1[|v|>sig(s)] ; rg_aux = -g_out*sign(v)*1[..]*sig(s)(1-sig(s))
 *   OPTEMBED  rg_main = d/d weight row incl. the BinaryStep surrogate (optembed_utils.py:35-44);
 *             rg_aux[b,f] (ONE float per lookup) = g_z, so that g_t[f] = -sum_b rg_aux[b,f]
 * Also accumulates the first-order weight gradient fc_grad[row] += g_yfm[b] (dense [N,1]; a second
 * launch that merges equal rows of 32 consecutive samples per field before one atomic per distinct row).
 *
 *  rows      [B,F] int64 global ids saved by the forward
 *  emb, S    forward outputs (emb may be NULL when g_yfm is NULL and the kind does not need it)
 *  g_yfm     [B] or NULL ; g_deep [B,F*D] or NULL (at least one non-NULL)
 * ---------------------------------------------------------------------- */
RSB_API int rsb_lookup_bwd_rows(int32_t kind, const int64_t* rows, int64_t B, int32_t F, int32_t D,
                        const float* table, int64_t n_rows, const float* table1, int64_t divider,
                        const void* aux, int32_t aux_mode, const int64_t* mask_d_idx,
                        const float* emb, const float* S, const float* g_yfm, const float* g_deep,
                        float* rg_main, float* rg_aux, float* fc_grad, void* stream);

/* First-order weight gradient alone: fc_grad[row] += g_yfm[b] for every lookup (dense [N,1], pre-zeroed).
 * rsb_lookup_bwd_rows / rsb_qr_bwd_fused run it too when their fc_grad argument is non-NULL. */
RSB_API int rsb_fc_grad(const int64_t* rows, const float* g_yfm, int64_t B, int32_t F, float* fc_grad, void* stream);

/* The same gradient from the row-sorted lookups (rsb_sort_rows of the full row ids: sorted_keys[i] is the row of
 * lookup perm[i] = b * F + f): one writer per touched row, fixed summation order - bit-reproducible where rsb_fc_grad
 * (float atomics) is not.  fc_grad is the zero-filled dense [N] gradient of FeaturesLinear's nn.Embedding(N, 1)
 * (src/models/deepfm.py:71-76 / aten embedding_dense_backward).  workspace: rsb_segment_workspace_bytes(n, 1). */
RSB_API int rsb_fc_grad_sorted(const uint32_t* sorted_keys, const uint32_t* perm, int64_t n, const float* g_yfm, int32_t F,
                               float* fc_grad, void* workspace, int64_t workspace_bytes, void* stream);

/* QR (mult / add) variant of stage 1 with the emb1 gradient fused in: emb1 has only `divider`
 * rows (2/5/20 in configs/deepfm/qr_*.yaml), so every lane group keeps one accumulator per emb1
 * row in registers while it streams the lookups; no per-lookup emb1 gradient is written and no
 * second pass over the lookups is needed.  divider <= 8, else RSB_ERR_UNSUPPORTED (callers then
 * use rsb_lookup_bwd_rows + rsb_small_table_grad).  table1_grad [divider, D] is overwritten. */
RSB_API int64_t rsb_qr_bwd_fused_workspace_bytes(int64_t B, int32_t D);
RSB_API int rsb_qr_bwd_fused(int32_t kind, const int64_t* rows, int64_t B, int32_t F, int32_t D,
                             const float* table, int64_t n_rows, const float* table1, int64_t divider,
                             const float* emb, const float* S, const float* g_yfm, const float* g_deep,
                             float* rg_main, float* table1_grad, float* fc_grad, void* workspace,
                             int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Backward, stage 2: stable LSD radix sort of the lookups by target row.
 *
 *  keys       [n] int64 row ids in [0, n_rows)  (optionally transformed: key = id / key_div
 *             when key_div > 1, key = id % key_mod when key_mod > 0 — the bit-exact QR index
 *             math of qr_embedding.py:96-97)
 *  sorted_keys [n] uint32, perm [n] uint32 (perm[j] = original lookup position)
 * ---------------------------------------------------------------------- */
RSB_API int64_t rsb_sort_workspace_bytes(int64_t n);
RSB_API int rsb_sort_rows(const int64_t* keys, int64_t n, int64_t n_rows, int64_t key_div, int64_t key_mod,
                  uint32_t* sorted_keys, uint32_t* perm, void* workspace, int64_t workspace_bytes,
                  void* stream);

/* ------------------------------------------------------------------------
 * Backward, stage 3: deterministic segmented reduction over the sorted lookups
 * and application of the result (dense grad row / fused SparseAdam / fused SGD).
 * Replaces aten embedding_dense_backward resp. coalesce + torch.optim.SparseAdam /
 * SGD (src/models/deepfm.py:173-216).
 *
 *  row_grads  [n, E] per-lookup gradients (stage 1), E = row width
 *  dst        APPLY_DENSE: zero-filled dense grad [n_rows,E]; ADAM/SGD: the weight table
 *  exp_avg, exp_avg_sq   SparseAdam state [n_rows,E] (ADAM only)
 *  lr, beta1, beta2, eps, step   optimizer hyper-parameters; step is the 1-based step count
 * ---------------------------------------------------------------------- */
RSB_API int64_t rsb_segment_workspace_bytes(int64_t n, int32_t E);
RSB_API int rsb_segment_reduce_apply(int32_t apply, const uint32_t* sorted_keys, const uint32_t* perm, int64_t n,
                             const float* row_grads, int32_t E,
                             float* dst, float* exp_avg, float* exp_avg_sq,
                             float lr, float beta1, float beta2, float eps, int64_t step,
                             void* workspace, int64_t workspace_bytes, void* stream);

/* Small-table gradient (QR emb1 has `divider` = 2..~1000 rows; qr_embedding.py:59): shared-memory
 * accumulation per CTA, fixed-order cross-CTA reduction.  dst[n_rows,E] is overwritten.
 * keys as in rsb_sort_rows (key_div / key_mod transform).  */
RSB_API int64_t rsb_small_table_workspace_bytes(int64_t n_rows, int32_t E);
RSB_API int rsb_small_table_grad(const int64_t* keys, int64_t n, int64_t key_div, int64_t key_mod,
                         const float* row_grads, int32_t E, int64_t n_rows, float* dst,
                         void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Full-table helpers of the variants.
 * ---------------------------------------------------------------------- */
/* PEP get_weight / get_num_params (pep_embedding.py:78-80,127-130): out (may be NULL) =
 * soft_threshold(weight, s); *count (device int64, may be NULL) += number of non-zeros. */
RSB_API int rsb_pep_threshold_table(const float* weight, const float* s, int32_t threshold_type, int64_t n_rows,
                            int32_t D, float* out, int64_t* count, void* stream);
/* PEP dense backward epilogue: given g_table (dense grad wrt the thresholded table) produce
 * g_weight and g_s_full [N,D] in one pass (autograd of pep_embedding.py:91-92). */
RSB_API int rsb_pep_dense_bwd(const float* weight, const float* s, int32_t threshold_type, int64_t n_rows, int32_t D,
                      const float* g_table, float* g_weight, float* g_s_full, void* stream);
/* OptEmbed eval-mode weight (deepfm_opt_embed.py:148-202; optembed_utils.py:88-99):
 * out[row,:] = weight[row,:] * 1[norm(weight[row]) - t_row[row] > 0] * tril[d <= mask_d_row[row]].
 * t_row [N] per-feature thresholds or NULL; mask_d_row [N] int64 or NULL. count as above. */
RSB_API int rsb_optembed_eval_weight(const float* weight, const float* t_row, const int64_t* mask_d_row, int32_t norm,
                             int64_t n_rows, int32_t D, float* out, int64_t* count, void* stream);
/* out = weight * mask (uint8) : RetrainPepEmbedding.get_weight / RetrainOptEmbed.get_weight. */
RSB_API int rsb_mask_table(const float* weight, const uint8_t* mask, int64_t numel, float* out, void* stream);
/* out[i] = sigmoid(s[i]) in the arithmetic every PEP / CERP kernel of this library uses for its thresholds,
 * 1 / (1 + expf(-s)) - the formula of torch.sigmoid on CUDA (pep_embedding.py:86,91 run on the trainer's device),
 * so `abs(v) > sigmoid(s)` mask decisions are bit-identical to the reference's GPU path (tested bit-for-bit). */
RSB_API int rsb_sigmoid(const float* s, int64_t numel, float* out, void* stream);

/* ------------------------------------------------------------------------
 * Inference gather from a pruned table kept as CSR (SURVEY 8 f-4).  Replaces PrunedEmbedding.forward
 * and its numba kernel csr_embedding_lookup (src/models/embeddings/pruned_embedding.py:89-173: one thread
 * per id, zero-fill + scattered stores), fused with DeepFM's offsets add, first order and FM second order
 * (src/models/deepfm.py:88-98) like rsb_lookup_fwd.
 *   values [nnz] f32, crow [n_rows+1] (crow_bytes 8 = int64 like torch / the reference, or 4),
 *   col [nnz] (col_bytes 8, 4 or 1); columns must be sorted and unique inside a row (torch's
 *   to_sparse_csr() order).  D <= 32.  out_emb [B,F,D]; out_yfm [B] or NULL (then fc/bias unused).
 *   Out-of-range ids are clamped to row 0 and raise *err_flag like rsb_lookup_fwd. */
RSB_API int rsb_csr_lookup_fwd(const void* idx, int32_t idx_is_i32, const int64_t* offsets, int64_t B, int32_t F,
                               int32_t D, const float* values, const void* crow, int32_t crow_bytes, const void* col,
                               int32_t col_bytes, int64_t n_rows, const float* fc, const float* bias, float* out_emb,
                               float* out_yfm, int32_t* err_flag, void* stream);

/* ------------------------------------------------------------------------
 * Deep hash embedding encoder (SURVEY 8 f-3).  Replaces the cached [N,k] code table of DHEmbedding and its
 * builders _get_universal_hash / _get_universal_hash_batch / _init_all_hash
 * (src/models/embeddings/dh_embedding.py:194-236,250-268) and the F.embedding(inp, cache) gather at :312-315:
 *   out[i,j] = float(((slopes[j]*(ids[i]+prefix+1) + bias[j]) mod primes[j]) mod m) / float(m-1) * 2 - 1
 * int64 arithmetic with Python's sign convention for mod, bit-exact.  ids [n] int64 or int32; slopes, bias,
 * primes [k] int64; 2 <= m <= 2^24; out [n,k] fp32.  small_operands != 0 promises |slopes|,|bias| < 2^31,
 * 2 <= primes < 2^31 and 0 <= ids+prefix+1 < 2^30 (enables the fp64-reciprocal modulo); 0 = generic int64 path. */
RSB_API int rsb_dhe_encode(const void* ids, int32_t ids_is_i32, int64_t n, int64_t prefix, const int64_t* slopes,
                           const int64_t* bias, const int64_t* primes, int32_t k, int64_t m, int32_t small_operands,
                           float* out, void* stream);

/* ------------------------------------------------------------------------
 * fp32-accurate tensor-core GEMM on PRE-SPLIT operands ("planes"), hand-written TMA + tcgen05 + TMEM kernel
 * (csrc/gemm/planes_gemm.cu).  An fp32 matrix X is held as three bf16 matrices X0 + X1 + X2 (8 mantissa bits each);
 * the kernel issues the six plane products >= 2^-16 |a||b| as bf16 tensor-core MMAs, smallest first, and drains the
 * TMEM accumulator into fp32 registers every 32 k.  Replaces the reference's fp32 cuBLAS GEMMs of nn.Linear
 * (src/models/deepfm.py:55-66, src/models/dcn.py:56-66) and of the DCN-Mix expert projections
 * (src/models/layer_dcn.py:20-23); planes are written once by rsb_split_planes (or a producer's epilogue) and reused by
 * every GEMM that reads the operand (forward + weight gradient share the activation planes).
 *
 * rsb_planes_operand: `planes` = bf16 [3][rows][ld] (plane p at planes + p * plane_stride elements), the STORED matrix
 *   is [rows, cols] row-major.  mn_major = 0: the stored rows are the M (or N) index and the columns the K index
 *   ("K-major": activations [B, in] for y = x W^T, nn.Linear weights [out, in]); mn_major = 1: the stored rows are K
 *   and the columns M (or N) (both operands of a weight gradient dW = gz^T x, whose K is the batch).
 *   batch_row_step / batch_col_step: added to the stored row / column coordinate per batch index (strided batches
 *   that live inside one matrix, e.g. the E experts of layer_dcn.py:22 as column blocks).
 * ld, plane_stride multiples of 8 elements; planes 16-byte aligned; N, ldd multiples of 4.
 * D[l] = alpha * A[l] B[l]^T-or-B[l] + beta * C[l] + bias;  split_k = 0 picks a split that fills the SMs when there
 * are fewer tiles than SMs (partials in the workspace, summed in fixed order by a second launch).
 * ---------------------------------------------------------------------- */
/* Operand formats.  RSB_PLANES_BF16X3 (default): three bf16 planes, every fp32 value exactly, 6 MMAs per product.
 * RSB_PLANES_FP16X2: two fp16 planes of X * s, s = the power of two that puts the bound *amax >= max |X| (a DEVICE
 * scalar, written by whoever knows it: rsb_absmax, the BatchNorm statistics kernels) into [2^13, 2^14), at most
 * 2^max_scale_exp: 22 bits for the big elements, 2^-38 of the bound for every element, 3 MMAs per product - the
 * error stays below the fp32 rounding of the sum itself (tests/test_gemm_split_math.py).  Writers and the GEMM derive s
 * from the same scalar, so no host round trip is involved.  Both operands of one GEMM must use the same format. */
typedef enum { RSB_PLANES_BF16X3 = 0, RSB_PLANES_FP16X2 = 1 } rsb_planes_format_id;
typedef struct {
  int32_t format;          /* rsb_planes_format_id */
  int32_t max_scale_exp;   /* FP16X2: scale <= 2^max_scale_exp (14 when the planes carry a ones column, which stores s) */
  float* amax;             /* FP16X2: device scalar bound on |X| (read; written first by rsb_bn_train_bwd_planes) */
} rsb_planes_format;

typedef struct {
  const void* planes;
  int64_t rows, cols, ld, plane_stride;
  int32_t mn_major;
  int64_t batch_row_step, batch_col_step;
  rsb_planes_format fmt;   /* zero-initialised = BF16X3 */
} rsb_planes_operand;

/* What rsb_gemm_planes does with the accumulator (fused epilogues of the dense tail, src/models/deepfm.py:55-66):
 *   RSB_EPI_LINEAR               D = alpha * acc + beta * C + bias                                   (fp32)
 *   RSB_EPI_RELU_DROPOUT_PLANES  y = dropout_p(relu(alpha * acc + bias)) written as bf16 planes (the next layer's GEMM
 *                                operand): the forward of Linear -> ReLU -> Dropout.  `mask` [M, N] holds the dropout
 *                                keep bits on entry (rsb_dropout_keep_mask: same Philox stream as rsb_relu_dropout_fwd,
 *                                so the masks equal the un-fused pass bit for bit) and keep && (pre-activation > 0),
 *                                the mask the backward needs, on exit.
 *   RSB_EPI_MASK_PLANES          g = alpha * acc * mask / (1 - p) written as planes: dX of a hidden layer, i.e. the
 *                                gradient w.r.t. the previous layer's pre-activation, ready for its dX / dW GEMMs.
 *   RSB_EPI_MASK_F32             the same as fp32 D (a BatchNorm backward sits in between).
 * ones_col: the plane writers also store a column of ones right after the (8-padded) data columns; a weight-gradient
 * GEMM gz^T [x | 1] over such planes yields the bias gradient as its last column, with no extra reduction pass. */
typedef enum {
  RSB_EPI_LINEAR = 0,
  RSB_EPI_RELU_DROPOUT_PLANES = 1,
  RSB_EPI_MASK_PLANES = 2,
  RSB_EPI_MASK_F32 = 3
} rsb_epilogue_mode;

typedef struct {
  int32_t mode;
  void* out_planes;            /* bf16 [3][M][out_ld] (modes 1, 2) */
  int64_t out_ld, out_plane_stride;
  int32_t ones_col;
  uint8_t* mask;               /* [M, N]: updated in place by mode 1, read by modes 2, 3 */
  float p;                     /* dropout probability */
  float* d_amax;               /* modes 0, 3 (fp32 D, no split-K), optional: *d_amax is raised to max |D| - the bound an
                                  FP16X2 consumer of D needs (rsb_bn_train_bwd_planes), formed in the epilogue for free */
  float* bn_partials;          /* mode 0, optional: BatchNorm batch statistics of D as per-32-row-group shifted column sums
                                  [row_groups][3][N] = (sum (d - k), sum (d - k)^2, k = the group's first row), reduced from
                                  the accumulator registers in the epilogue; rsb_bn_finalize_partials turns them into mean /
                                  rstd / affine, so the statistics pass over D (rsb_bn_train_fwd_stats) disappears.
                                  Size and availability: rsb_gemm_bn_partials_bytes */
} rsb_gemm_epilogue;

/* y = dropout_p(relu(x)) of an fp32 [M, N] activation (ldx) written as planes (+ ones column) and the 1-byte
 * keep-and-positive mask [M, N]: rsb_relu_dropout_fwd + rsb_split_planes in one pass, same Philox stream. */
RSB_API int rsb_relu_dropout_planes(const float* x, int64_t M, int32_t N, int64_t ldx, float p, uint64_t seed, uint64_t offset,
                                    const uint64_t* offset_dev, int32_t ones_col, void* out_planes, int64_t out_ld,
                                    int64_t plane_stride, uint8_t* mask, void* stream);
/* mask[i] = 1 with probability 1 - p: the dropout keep bits of an activation of `numel` (multiple of 4) elements, drawn
 * from the Philox stream (seed, offset [+ *offset_dev]) exactly like rsb_relu_dropout_fwd draws them. */
RSB_API int rsb_dropout_keep_mask(uint8_t* mask, int64_t numel, float p, uint64_t seed, uint64_t offset,
                                  const uint64_t* offset_dev, void* stream);

/* fp32 [rows, cols] (ld) -> bf16 planes [3][rows][out_ld] (columns cols..out_ld-1 zero); transpose = 1 writes the
 * planes of in^T ([cols][out_ld >= rows]); ones_col = 1 additionally writes 1.0 at column roundup8(cols). */
RSB_API int rsb_split_planes(const float* in, int64_t rows, int64_t cols, int64_t ld, int32_t transpose, int32_t ones_col,
                             void* out_planes, int64_t out_ld, int64_t plane_stride, const rsb_planes_format* fmt /* NULL = BF16X3 */,
                             void* stream);
/* *amax_out = max(*amax_out, mul * max |g_row| * max |w_col|): bound on the rank-1 head gradient
 * g_row[r] * w_col[c] * mask / (1 - p) of rsb_relu_dropout_bwd_rank1 (mul = 1 / (1 - p)). */
RSB_API int rsb_rank1_absmax(const float* g_row, int64_t M, const float* w_col, int64_t N, float mul, float* amax_out,
                             void* stream);
/* *amax_out = max(*amax_out, max |in[r, c]|): the bound an FP16X2 split of `in` needs (zero the scalar first). */
RSB_API int rsb_absmax(const float* in, int64_t rows, int64_t cols, int64_t ld, float* amax_out, void* stream);
/* gz[r, c] = g_row[r] * w_col[c] * mask[r, c] / (1 - p) written as planes (N, out_ld multiples of 8): the backward of
 * dropout(relu(.)) for the rank-1 upstream gradient of the MLP's one-output Linear (src/models/deepfm.py:64). */
RSB_API int rsb_rank1_mask_planes(const float* g_row, const float* w_col, const uint8_t* mask, int64_t M, int32_t N, float p,
                                  void* out_planes, int64_t out_ld, int64_t plane_stride, void* stream);
RSB_API int64_t rsb_gemm_planes_workspace_bytes(int64_t M, int64_t N, int64_t K, int64_t batch, int32_t split_k);
RSB_API int rsb_gemm_planes(const rsb_planes_operand* A, const rsb_planes_operand* B, int64_t M, int64_t N, int64_t K,
                            int64_t batch, int32_t split_k, const float* C, float* D, int64_t ldd, int64_t d_batch_stride,
                            const float* bias, float alpha, float beta, const rsb_gemm_epilogue* epilogue /* NULL = linear */,
                            void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * BatchNorm1d in training mode, fused with its neighbours (csrc/batchnorm.cu).  Replaces torch.nn.BatchNorm1d +
 * ReLU + Dropout of the dense tails (src/models/deepfm.py:57-60, src/models/dcn.py:56-66) forward and backward; torch
 * semantics: biased batch variance for the normalisation, unbiased for running_var, eps inside the square root,
 * running = (1 - momentum) * running + momentum * batch.  All reductions are two-stage with a fixed order.
 *   rsb_bn_train_fwd_stats      z [M,N] (ldz) -> stats [2N] = (mean, rstd), affine [2N] = (gamma * rstd, beta - mean * scale),
 *                               running_mean / running_var updated in place (NULL: not tracked); act_amax (optional,
 *                               zero on entry) receives bound_mul * max_c (|gamma_c| sqrt(M) + |beta_c|) >= the largest
 *                               dropout(relu(BN(z))) (|xhat| <= sqrt(M)): the bound an FP16X2 rsb_bn_relu_dropout_planes
 *                               needs (bound_mul = 1 / (1 - p))
 *   rsb_bn_relu_dropout_planes  y = dropout_p(relu(z * scale + shift)) as bf16 planes (+ ones column) + the 1-byte
 *                               keep-and-positive mask; Philox stream as rsb_relu_dropout_fwd; p = 0: no dropout
 *   rsb_bn_train_bwd_planes     g [M,N] = gradient w.r.t. the BatchNorm output -> sums [2N] = (d beta, d gamma) and
 *                               gz = gamma * rstd * (g - d beta / M - xhat * d gamma / M) as planes
 * N, ldz, ldg multiples of 4; workspace from rsb_bn_workspace_bytes.
 * ---------------------------------------------------------------------- */
RSB_API int64_t rsb_bn_workspace_bytes(int64_t M, int32_t N);
RSB_API int rsb_bn_train_fwd_stats(const float* z, int64_t M, int32_t N, int64_t ldz, const float* gamma, const float* beta,
                                   float eps, float momentum, float* running_mean, float* running_var, float* stats,
                                   float* affine, float bound_mul, float* act_amax, void* workspace, int64_t workspace_bytes,
                                   void* stream);
/* bytes of the statistics buffer for rsb_gemm_epilogue.bn_partials, or -1 if this GEMM cannot carry them */
RSB_API int64_t rsb_gemm_bn_partials_bytes(int64_t M, int64_t N, int64_t K, int32_t format);
/* rsb_bn_train_fwd_stats' outputs from the partials a GEMM epilogue wrote: the group sums are re-based to one common shift
 * (exact identity) and folded in fixed order; workspace >= 16 * 2 * N * 4 + 256 bytes (rsb_bn_workspace_bytes suffices) */
RSB_API int rsb_bn_finalize_partials(const float* parts, int64_t M, int32_t N, const float* gamma, const float* beta, float eps,
                                     float momentum, float* running_mean, float* running_var, float* stats, float* affine,
                                     float bound_mul, float* act_amax, void* workspace, int64_t workspace_bytes, void* stream);
RSB_API int rsb_bn_relu_dropout_planes(const float* z, int64_t M, int32_t N, int64_t ldz, const float* affine, float p,
                                       uint64_t seed, uint64_t offset, const uint64_t* offset_dev, int32_t ones_col,
                                       void* out_planes, int64_t out_ld, int64_t plane_stride, uint8_t* mask,
                                       const rsb_planes_format* fmt /* NULL = BF16X3 */, void* stream);
RSB_API int rsb_bn_train_bwd_planes(const float* g, const float* z, int64_t M, int32_t N, int64_t ldg, int64_t ldz,
                                    const float* stats, const float* gamma, float* sums, void* out_planes, int64_t out_ld,
                                    int64_t plane_stride, const rsb_planes_format* fmt /* NULL = BF16X3; FP16X2: *amax
                                    (zero on entry) is set to a bound on |gz| before gz is written */,
                                    const float* g_amax /* FP16X2: device scalar >= max |g| */, void* workspace,
                                    int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Bandwidth-bound glue of the dense tails (Linear -> [BatchNorm1d] -> ReLU -> Dropout,
 * src/models/deepfm.py:55-66, src/models/dcn.py:56-66), one pass per direction.
 *  rsb_relu_dropout_fwd  y = dropout_p(relu(x)), mask[i] = 1 iff x[i] > 0 and kept (Philox4x32-10 keyed by
 *                        seed/offset; numel % 4 == 0, 16-byte aligned)
 *  rsb_relu_dropout_bwd  gx = g * mask / (1-p) for g [M,N]; colsum [N] (may be NULL) = column sums of gx,
 *                        i.e. the bias gradient of the preceding Linear, accumulated in the same pass
 *  rsb_colsum            out[N] = sum over rows of x [M,N] (row stride ld), deterministic two-stage
 * ---------------------------------------------------------------------- */
RSB_API int rsb_relu_dropout_fwd(const float* x, int64_t numel, float p, uint64_t seed, uint64_t offset,
                                 const uint64_t* offset_dev /* device, added to offset; may be NULL */, float* y,
                                 uint8_t* mask, void* stream);
RSB_API int rsb_relu_dropout_bwd(const float* g, const uint8_t* mask, int64_t M, int32_t N, float p, float* gx,
                                 float* colsum, void* workspace, int64_t workspace_bytes, void* stream);
RSB_API int64_t rsb_colsum_workspace_bytes(int64_t M, int32_t N);
RSB_API int rsb_colsum(const float* x, int64_t M, int32_t N, int64_t ld, float* out, void* workspace,
                       int64_t workspace_bytes, void* stream);
/* The MLPs end in a Linear with ONE output (src/models/deepfm.py:64, src/models/dcn.py:65: Linear(hidden, 1)):
 * a matrix-vector product whose three passes are folded into the neighbouring glue instead of library GEMV calls.
 *  rsb_relu_dropout_dot_fwd   y = dropout(relu(x)), mask as rsb_relu_dropout_fwd, and out[r] = y[r,:].w + bias[0];
 *                             affine [2N] (optional): x is first mapped to x * affine[c] + affine[N + c] (the BatchNorm
 *                             normalisation of rsb_bn_train_fwd_stats folded into the same pass)
 *  rsb_relu_dropout_bwd_rank1 rsb_relu_dropout_bwd with the upstream gradient g[r,c] = g_row[r] * w_col[c] formed
 *                             on the fly (the Linear's dX is never written)
 *  rsb_colsum_weighted        out[c] = sum_r row_weight[r] * x[r,c]  (the Linear's weight gradient)
 * Workspaces as rsb_colsum_workspace_bytes(M, N). */
RSB_API int rsb_relu_dropout_dot_fwd(const float* x, int64_t M, int32_t N, float p, uint64_t seed, uint64_t offset,
                                     const uint64_t* offset_dev, const float* w, const float* bias, const float* affine,
                                     float* y, uint8_t* mask, float* out, void* stream);
RSB_API int rsb_relu_dropout_bwd_rank1(const float* g_row, const float* w_col, const uint8_t* mask, int64_t M, int32_t N,
                                       float p, float* gx, float* colsum, void* workspace, int64_t workspace_bytes,
                                       void* stream);
RSB_API int rsb_colsum_weighted(const float* x, const float* row_weight, int64_t M, int32_t N, int64_t ld, float* out,
                                void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * DCN-Mix cross layer glue (src/models/layer_dcn.py:8-24,90-115), identity gate.  With
 *   P1 = x_l V_cat (GEMM), H1 = tanh(P1), P2 = H1 (x) C (block-diagonal GEMM), T0 = G2 U_cat (GEMM):
 *  gate_mix_fwd   g[b,e] = x_l[b,:].gates[e,:] ; H2 = tanh(P2) ; G2 = g[b,e] * H2[b,e,:]
 *  cross_out_fwd  x_next = x_0 * (T0 + bias * sum_e g[b,e]) + x_l
 *  cross_out_bwd  gT = g_next * x_0 ; gx0 = g_next * (T0 + bias * sg) ; dsg[b] = sum_d gT[b,d] * bias[d]
 *  gate_mix_bwd   gP2 = gG2 * g * (1 - H2^2) ; dg[b,e] = sum_k gG2*H2 + dsg[b] ; g_xl = g_next + sum_e dg[b,e]*gates[e,:]
 * x_l, x_0, T0, g_next [B,Dm] ; P2, H2, G2 [B,E*r] ; gates [E,Dm] ; g, dg [B,E] ; bias [Dm].
 * Dm % 4 == 0, r % 4 == 0, E <= 8, 16-byte aligned rows; else RSB_ERR_UNSUPPORTED.
 * ---------------------------------------------------------------------- */
RSB_API int rsb_dcn_gate_mix_fwd(const float* p2, const float* xl, const float* gates, int64_t B, int32_t Dm,
                                 int32_t E, int32_t r, float* h2, float* g, float* g2, void* stream);
RSB_API int rsb_dcn_cross_out_fwd(const float* t0, const float* x0, const float* xl, const float* bias,
                                  const float* g, int64_t B, int32_t Dm, int32_t E, float* x_next, void* stream);
RSB_API int rsb_dcn_cross_out_bwd(const float* g_next, const float* x0, const float* t0, const float* bias,
                                  const float* g, int64_t B, int32_t Dm, int32_t E, float* gT, float* gx0,
                                  float* dsg, void* stream);
RSB_API int rsb_dcn_gate_mix_bwd(const float* g_g2, const float* h2, const float* g, const float* dsg,
                                 const float* gates, const float* g_next, int64_t B, int32_t Dm, int32_t E,
                                 int32_t r, float* g_p2, float* dg, float* g_xl, void* stream);

/* ------------------------------------------------------------------------
 * Row-sharded tables over the GPUs of one box (SURVEY.md section 8e; no reference
 * counterpart: the reference is single-device).  Rank g owns the rows r of the concatenated
 * table with r % G == g, stored at local row r / G.  Shards live in cudaMalloc'ed buffers
 * exported with CUDA IPC; peers read (forward gather) and atomically add (backward) through
 * the mapped pointers, i.e. directly over NVLink / NVSwitch — the index / row / row-grad
 * exchange of an all-to-all design happens inside the gather and scatter kernels.
 * ---------------------------------------------------------------------- */
#define RSB_IPC_HANDLE_BYTES 64
/* The only allocating calls of the library: peer-shareable buffers (zero-filled). */
RSB_API int rsb_shared_alloc(int64_t bytes, void** dev_ptr_out /* host */);
RSB_API int rsb_shared_free(void* dev_ptr);
RSB_API int rsb_ipc_get_handle(const void* dev_ptr, uint8_t* h_handle /* [64] host */);
RSB_API int rsb_ipc_open_handle(const uint8_t* h_handle /* [64] host */, void** dev_ptr_out /* host */);
RSB_API int rsb_ipc_close_handle(void* dev_ptr);
/* rsb_lookup_fwd(kind = VANILLA) over G shards: table_shards is a DEVICE array of G device pointers (own
 * shard + IPC-mapped peers).  The first-order weights are one REPLICATED full-length vector fc_replicated
 * [n_global] (NULL = no FM head): 4-byte peer reads / NVLink atomics cost as many transactions as the 64-byte
 * row traffic for 1/16 of the bytes (measured: a row-sharded first-order gradient took 0.76 ms of a 5.0 ms step
 * at N=8), so their gradient is rsb_fc_grad into a local dense buffer, allreduced with the other dense grads. */
/* Small fields may be REPLICATED instead of sharded (the 31 Criteo fields of <= 16 384 ids hold 4 % of the rows but
 * serve 31 of a sample's 39 lookups; sharded, 7/8 of those cross NVLink at G = 8): hot_map is a device int64 [F, 3]
 * array, one (lo, hi, delta) per field with lo = the field's offset; a lookup of field f whose global row lies in
 * [lo, hi) reads hot_table[row + delta] (a local dense [H, D] table, same values on every rank), hi == lo marks a
 * sharded field.  A row outside [lo, hi) of a replicated field (an id beyond its own field) sets err_flag and takes
 * the sharded path.  hot_table = hot_map = NULL: everything sharded. */
RSB_API int rsb_lookup_fwd_sharded(const void* idx, int32_t idx_is_i32, const int64_t* offsets, int64_t B, int32_t F,
                                   int32_t D, const float* const* table_shards, const float* fc_replicated,
                                   int32_t G, int64_t n_global, const float* bias, const float* hot_table,
                                   const int64_t* hot_map, float* out_emb, float* out_yfm,
                                   float* out_sum, int64_t* out_rows, int32_t* err_flag, float* amax_slots /* as rsb_lookup_fwd */,
                                   void* stream);
/* The same over ANY variant (SURVEY 8e: "for PEP `s`, for masks the mask rows; for QR shard emb2, replicate the
 * <= 20-row emb1").  Sharded like the vanilla table - row r of the MAIN table (the [N, D] weight of VANILLA / PEP / MASK /
 * OPTEMBED, emb2 of QR, n_rows rows in all) lives in shard r % G at local row r / G - are
 *   table_shards [G]  the main table, and
 *   aux_shards   [G]  the per-row aux array: PEP `s` for aux_mode FEATURE [N,1] / FEATURE_DIM [N,D] (fp32), the retrain
 *                     mask [N,D] (uint8) for MASK; NULL for every other kind / mode.
 * Replicated on every rank, passed as for rsb_lookup_fwd: table1 (QR emb1), aux for PEP GLOBAL / DIMENSION and the
 * OPTEMBED per-field thresholds t [F] (NULL = mask-E off), fc_replicated [n_global], bias.  OPTEMBED's mask_d_idx is
 * this rank's own [B, F] draw, one index per lookup, as for rsb_lookup_fwd.  Arguments not listed here are those of
 * rsb_lookup_fwd.  The OptEmbed eval cache (rsb_optembed_eval_weight run on each rank's weight shard) is gathered with
 * kind = VANILLA over the eval shards. */
RSB_API int rsb_lookup_fwd_sharded_kind(int32_t kind, const void* idx, int32_t idx_is_i32, const int64_t* offsets, int64_t B,
                                        int32_t F, int32_t D, const float* const* table_shards, int32_t G, int64_t n_rows,
                                        int64_t n_global, const float* table1, int64_t divider, const void* aux,
                                        const void* const* aux_shards, int32_t aux_mode, const int64_t* mask_d_idx,
                                        const float* fc_replicated, const float* bias, float* out_emb, float* out_yfm,
                                        float* out_sum, int64_t* out_rows, int32_t* err_flag, float* amax_slots, void* stream);
/* rsb_lookup_bwd_rows over the same shards (the variants' chain rules re-read the table / threshold / mask rows from
 * their owners); the per-lookup gradients rg_main / rg_aux stay local and are then pushed to the owners with
 * rsb_segment_scatter_shards (main table; PEP `s` with its own gradient shards), the replicated parameters' gradients
 * are reduced locally (rsb_small_table_grad for emb1; OPTEMBED: g_t[f] = -sum_b rg_aux[b, f] over the [B, F]
 * per-lookup scalars, with t replicated and the forward's mask_d_idx) and averaged by the caller's allreduce. */
RSB_API int rsb_lookup_bwd_rows_sharded(int32_t kind, const int64_t* rows, int64_t B, int32_t F, int32_t D,
                                        const float* const* table_shards, int32_t G, int64_t n_rows, const float* table1,
                                        int64_t divider, const void* aux, const void* const* aux_shards, int32_t aux_mode,
                                        const int64_t* mask_d_idx, const float* emb, const float* S, const float* g_yfm,
                                        const float* g_deep, float* rg_main, float* rg_aux, void* stream);
/* Backward: segmented reduction of this rank's sorted lookups (rsb_sort_rows on GLOBAL row
 * ids), each locally-unique row's sum * scale added into the owner's dense shard gradient
 * with one 128-bit red.global.add per 4 floats.  Rows of replicated fields (hot_map [n_fields, 3] as above, the row's
 * field found by binary search over the offsets) are instead STORED, unscaled, into the zero-filled local dense
 * gradient hot_grad [H, E] (one writer per row, deterministic); the caller averages it over the ranks with the
 * other replicated gradients.  hot_map = hot_grad = NULL: everything sharded. */
RSB_API int rsb_segment_scatter_shards(const uint32_t* sorted_keys, const uint32_t* perm, int64_t n,
                                       const float* row_grads, int32_t E, float* const* grad_shards, int32_t G,
                                       float scale, const int64_t* hot_map, int32_t n_fields, float* hot_grad,
                                       void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Input staging (SURVEY 8 f-2).  The reference's lmdb caches store one uint32 record per sample,
 * [label, id_0 .. id_{F-1}] (src/dataset/criteo/criteo_torchfm.py:72-93, avazu_fm.py:78-97, kdd_dataset.py:53-74:
 * `np.frombuffer(..., dtype=np.uint32)`, `arr[1:]` = ids, `arr[0]` = label).  One pass turns a staged block of records
 * [B, F+1] (uint32 / int32, device) into what the training step consumes: ids_out [B,F] int32 (per-field ids WITHOUT
 * offsets, the batch format rsb_lookup_fwd reads with idx_is_i32 = 1) and labels_out [B] fp32 (`labels.float()` of
 * src/trainer/deepfm.py:52; NULL = skip).  Meant for the copy stream, right behind the H2D copy of the block. */
RSB_API int rsb_records_unpack(const void* records, int64_t B, int32_t F, int32_t* ids_out, float* labels_out, void* stream);

/* ------------------------------------------------------------------------
 * Dense Adam over every parameter of the model in one launch: the non-sparse branch of get_optimizers
 * (src/models/deepfm.py:155-172, `torch.optim.Adam(model.parameters(), lr, weight_decay)`), arithmetic of
 * torch/optim/adam.py::_single_tensor_adam (L2 weight decay folded into the gradient, bias corrections formed in
 * double on the host from `step`, denom = sqrt(v) / sqrt(bc2) + eps).
 *   h_tensors HOST array of n_tensors <= RSB_ADAM_MAX_TENSORS descriptors of DEVICE buffers (fp32, numel elements each;
 *             param / exp_avg / exp_avg_sq updated in place).  They are passed to the kernel by value, so the caller
 *             may rewrite the array right after the call (gradient buffers move from step to step).
 *   block_map DEVICE int32 [n_blocks, 2]: (tensor index, chunk index); chunk c of a tensor covers elements
 *             [c * RSB_ADAM_CHUNK, min(numel, (c + 1) * RSB_ADAM_CHUNK)).  Depends on the numels only: built once.
 *   step      1-based step count shared by these tensors (torch keeps one per parameter; callers group equal counts). */
#define RSB_ADAM_CHUNK 4096
#define RSB_ADAM_MAX_TENSORS 64
typedef struct {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t numel;
} rsb_adam_tensor;
RSB_API int rsb_adam_dense(const rsb_adam_tensor* h_tensors, int32_t n_tensors, const int32_t* block_map, int64_t n_blocks,
                           double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RSB_H_ */
