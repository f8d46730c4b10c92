/*
 * hidvae_b200.h -- C ABI of the B200-native residual-quantisation (RQ) hot path of HiD-VAE.
 *
 * This is the drop-in boundary.  The reference has no FFI or operator registry: its boundary for this path
 * is the Python class API (SURVEY.md section 8b), all arithmetic being PyTorch ATen calls.  Each entry point
 * below replaces the ATen call sequence of one reference function; the host-side mirror of the reference
 * classes (hid-vae_b200/modules, hid-vae_b200/init) binds these symbols with ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); the library never allocates or frees;
 *   - tensors are contiguous row-major fp32 / int64 unless explicit strides (in ELEMENTS) are passed;
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream); all work is
 *     enqueued on it, there is no implicit synchronisation, calls are CUDA-graph capturable;
 *   - return value 0 = HV_OK, otherwise an hv_status_t; hv_last_error() returns a thread-local message;
 *   - no exceptions cross the boundary; the library is re-entrant (no mutable global state besides
 *     per-device function attributes set once).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns HV_ERR_CUDA.
 *
 * "codebooks" always means the EFFECTIVE codebooks C_l = out_proj(embedding.weight) of each level
 * (modules/quantize.py:106), stacked [L, K, D]; PyTorch keeps out_proj (row L2-norm / sim_vq Linear) and
 * back-propagates the returned g_codebooks through it.
 */
#ifndef HIDVAE_B200_H_
#define HIDVAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  HV_OK = 0,
  HV_ERR_BAD_SHAPE = 1,    /* negative / zero / inconsistent sizes                                   */
  HV_ERR_UNSUPPORTED = 2,  /* (D, K, L, mode, algo) combination no kernel is instantiated for         */
  HV_ERR_MISALIGNED = 3,   /* pointer not 16-byte aligned where vector access needs it                */
  HV_ERR_CUDA = 4,         /* a CUDA runtime call failed; message holds cudaGetErrorString            */
  HV_ERR_NULL = 5,         /* required pointer is NULL                                                */
  HV_ERR_WORKSPACE = 6     /* workspace missing or smaller than hv_workspace_bytes() reports          */
} hv_status_t;

/* numeric values follow QuantizeForwardMode (modules/quantize.py:17-20) */
typedef enum { HV_MODE_GUMBEL_SOFTMAX = 1, HV_MODE_STE = 2, HV_MODE_ROTATION_TRICK = 3 } hv_forward_mode_t;

/* which implementation computes distance+argmin.  AUTO picks TCGEN05 when the shape is supported. */
typedef enum {
  HV_ALGO_AUTO = 0,
  HV_ALGO_TCGEN05 = 1, /* tcgen05.mma bf16x3 split (fp32-grade scores), TMEM accumulators, fused argmin  */
  HV_ALGO_SIMT = 2     /* exact fp32 FMA on CUDA cores, GEMM-form distance  |x|^2+|c|^2-2x.c              */
  ,
  HV_ALGO_SIMT_DIFF = 3 /* exact fp32, difference form  sum (x-c)^2  (init/kmeans.py:44-47)               */
  ,
  HV_ALGO_TCGEN05_PREPACKED = 4 /* as TCGEN05, but `workspace` already holds the image written by
                                   hv_rq_pack_codebooks for these codebooks (saves the pack launch when one set
                                   of codebooks serves many calls: bulk encode, train forward + eval encode)   */
} hv_algo_t;

typedef enum { HV_OP_RQ_FORWARD = 0, HV_OP_RQ_BACKWARD = 1 } hv_op_t;

int hv_version(void);
const char* hv_last_error(void);
/* number of SMs / compute capability of the current device; returns HV_ERR_CUDA when there is none */
int hv_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* bytes of scratch the op can use for this shape: HV_OP_RQ_FORWARD -- the packed bf16 codebook images of the tcgen05
 * path (independent of n); HV_OP_RQ_BACKWARD -- replicas of the [L, K, D] codebook gradient that spread the
 * scatter-add over more L2 lines (0 for small n: the op then adds straight into g_codebooks). */
size_t hv_workspace_bytes(int op, int64_t n, int d, int k, int n_levels);

/*
 * Fused L-level residual quantisation, forward.
 * Replaces, per level: the distance table, argmin, gather, STE / rotation-trick value, QuantizeLoss and the
 * residual update -- modules/quantize.py:106-148, modules/loss.py:41-44, modules/h_rqvae.py:515-523,552 --
 * and the output packing of h_rqvae.py:572-574.  The [N, K] table never exists in HBM.
 *
 *   x           [N, D]     level-0 input (the encoder output)
 *   codebooks   [L, K, D]  effective codebooks
 *   mode        HV_MODE_STE | HV_MODE_ROTATION_TRICK (GUMBEL_SOFTMAX: HV_ERR_UNSUPPORTED here -- hv_gumbel_forward)
 *   training    1: emb_out = e (STE value) or the rotated vector; 0: eval semantics emb_out = e
 *   beta        commitment weight; loss_l = (1 + beta) * |r_l - e_l|^2 computed as a + beta*a
 *   ids         int64, element (row, level) at ids[row*ids_row_stride + level*ids_level_stride]
 *   emb_out     [L, N, D] or NULL   (the reference's [N, D, L] `embeddings` is a permuted view of this)
 *   residuals   [L, N, D] or NULL   (input of every level, h_rqvae.py:516)
 *   loss        [N] or NULL         (sum over levels, h_rqvae.py:518)
 *   level_loss  [L, N] or NULL
 *   final_residual [N, D] or NULL   (r_L, what is left after the last level)
 * With emb_out = residuals = loss = level_loss = NULL and training = 0 this is the encode-only path of
 * HSemanticIdTokenizer.precompute_corpus_ids (modules/tokenizer/h_semids.py:127-130).
 */
int hv_rq_forward(const float* x, int64_t n, int d, const float* codebooks, int n_levels, int k, int mode,
                  int training, float beta, int64_t* ids, int64_t ids_row_stride, int64_t ids_level_stride,
                  float* emb_out, float* residuals, float* loss, float* level_loss, float* final_residual,
                  int algo, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Writes the tensor-core operand image of the effective codebooks (bf16 hi/lo split in the UMMA core-matrix
 * layout plus the -|c|^2/2 terms) into `workspace` (>= hv_workspace_bytes(HV_OP_RQ_FORWARD, ...)) and, for shapes
 * whose codebooks stay resident in shared memory (D = 32, K <= 256, L <= 3), a chunk-swizzled fp32 copy of the
 * codebooks behind it (the kernel gathers the chosen code rows from that copy).  hv_rq_forward does this itself for
 * HV_ALGO_TCGEN05 / AUTO; call it once and pass HV_ALGO_TCGEN05_PREPACKED to reuse the image.
 */
int hv_rq_pack_codebooks(const float* codebooks, int n_levels, int k, int d, void* workspace, size_t workspace_bytes,
                         void* stream);

/*
 * Fused backward of hv_rq_forward (the autograd graph of quantize.py:131-148 + h_rqvae.py:552 over L levels;
 * recursion in SURVEY.md section 8a).  Residuals are recomputed from x, ids and the codebooks.
 *
 *   g_emb    gradient w.r.t. emb_out; element (level, row, c) at g_emb[level*ls + row*rs + c] (ls may be 0
 *            for a broadcast such as the backward of embs.sum(-1)); NULL = zero
 *   g_loss   gradient w.r.t. loss, element row at g_loss[row*g_loss_stride] (stride 0 = broadcast scalar)
 *   g_level_loss  [L, N] contiguous or NULL: gradient w.r.t. level_loss (added to g_loss per level)
 *   g_x      [N, D] written
 *   g_codebooks [L, K, D] ACCUMULATED into (caller zeroes); rows are scatter-added by id
 *               (the embedding_dense_backward of quantize.py:97-98)
 *   workspace   optional scratch of hv_workspace_bytes(HV_OP_RQ_BACKWARD, ...) bytes (contents irrelevant, the op
 *               zeroes what it uses); NULL or too small = no replicas, same results up to summation order
 */
int hv_rq_backward(const float* x, int64_t n, int d, const float* codebooks, int n_levels, int k, int mode,
                   int training, float beta, const int64_t* ids, int64_t ids_row_stride,
                   int64_t ids_level_stride, const float* g_emb, int64_t g_emb_level_stride,
                   int64_t g_emb_row_stride, const float* g_loss, int64_t g_loss_stride,
                   const float* g_level_loss, float* g_x, float* g_codebooks, void* workspace,
                   size_t workspace_bytes, void* stream);

/*
 * K-means codebook init (init/kmeans.py:43-61).  Assignment = hv_rq_forward with n_levels = 1 (ids only).
 * hv_kmeans_accumulate: deterministic (bit-reproducible) per-cluster sums and counts of the assigned rows
 *   assign and prev_assign are int64 [n] and every assignment must lie in [0, K): the segmented form's search over keys
 *   sorted on ceil(log2 K) bits assumes it, and the scan form drops other rows.  Each sum is a compensated (Kahan)
 *   fp32 sum in a fixed order, within a few fp32 ulps of sum |x| whatever the cluster's size.
 *   sums [K, D] and counts [K] (float) are OVERWRITTEN; n_changed[0] (int64, may be NULL) receives the number
 *   of rows whose assignment differs from prev_assign (NULL = count every row).
 *   workspace: optional hv_sort_workspace_bytes(n) bytes.  With it, large K * N take the SEGMENTED form: rows are
 *   key-sorted by cluster (stable radix sort) and one warp per cluster adds its members in row order -- O(N), x read
 *   once; without it (or for small shapes) one CTA per cluster scans the assignment vector.
 * hv_kmeans_finalize: centroid_c = sums_c / counts_c, or reseed_rows[c, :] when counts_c == 0 (kmeans.py:54-58);
 *   centroids [K, D] are updated in place; stats[0] = max_c ||new_c - old_c||_2 (kmeans.py:68), stats[1] =
 *   number of empty clusters.  Between the two calls a data-parallel caller all-reduces sums and counts.
 */
size_t hv_sort_workspace_bytes(int64_t n);
int hv_kmeans_accumulate(const float* x, int64_t n, int d, const int64_t* assign, const int64_t* prev_assign,
                         int k, float* sums, float* counts, int64_t* n_changed, void* workspace, size_t workspace_bytes,
                         void* stream);
int hv_kmeans_finalize(const float* sums, const float* counts, const float* reseed_rows, int k, int d,
                       float* centroids, float* stats, void* stream);

/*
 * Semantic-ID uniqueness loss (modules/h_rqvae.py:41-105) and p_unique_ids (:645-648) over `rows` id tuples of
 * `width` int64 each (element (r, c) at ids[r*row_stride + c*col_stride]).
 * Forward: stats[0] = sum over pairs i<j with identical tuples of relu(cos(f_i, f_j) - margin) (double),
 *          stats[1] = number of such pairs, stats[2] = number of rows that have a LATER identical row.
 *          stats is OVERWRITTEN.  loss = weight * stats[0] / stats[1] (0 when stats[1] == 0) is formed by the
 *          caller on the device; p_unique = (rows - stats[2]) / rows.
 * Backward: g_feats [rows, D] (caller zeroes) += g_out[0] * weight / stats[1] * d(sum)/d feats, in a form without
 *          cancellation (exactly 0 for identical feature rows); a row with |f| < 1e-12 takes F.normalize's clamp
 *          derivative.  feats has at least `rows` rows.
 * workspace: optional hv_sort_workspace_bytes(rows) bytes.  With it, batches of >= 4096 rows are key-sorted by tuple and
 *   only runs of identical tuples are walked (O(rows + pairs)); otherwise all pairs i < j are swept (O(rows^2)).
 */
int hv_uniq_forward(const int64_t* ids, int64_t rows, int64_t width, int64_t row_stride, int64_t col_stride,
                    const float* feats, int d, float margin, double* stats, void* workspace, size_t workspace_bytes,
                    void* stream);
int hv_uniq_backward(const int64_t* ids, int64_t rows, int64_t width, int64_t row_stride, int64_t col_stride,
                     const float* feats, int d, float margin, float weight, const double* stats,
                     const float* g_out, float* g_feats, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Collision digit of semantic-ID tuples: the trailing id position of HSemanticIdTokenizer(use_dedup_dim=True), which
 * makes every item's id unique.  Over `rows` tuples of `width` int64 ids (element (r, c) at ids[r*row_stride + c*col_stride]):
 *   digit[r] = prior count of tuple r + #{ r' < r : tuple r' == tuple r }
 * written to digits[r*digit_stride] (digit_stride = L + 1 writes column L of an [N, L + 1] table whose first L columns
 * are `ids`).  Each tuple is packed into the exact key sum_c ids[c] << bits*(width-1-c), which ascends in lexicographic
 * tuple order; width * bits must be <= 63, else HV_ERR_UNSUPPORTED.  Rows are key-sorted (stable radix sort over
 * width*bits bits) and runs of equal keys are numbered by a scan: O(rows), whatever the number of repeats.
 *   bits          >= 1, ceil(log2 K) for codebooks of K codes
 *   prior_keys    [n_prior] ascending keys of tuples seen before these rows (e.g. the lower ranks' shards of a
 *                 catalogue) with their counts prior_counts [n_prior]; NULL / 0 for none
 *   run_keys, run_counts  [rows] capacity: the distinct keys of THIS call, ascending, and how many of its rows hold each
 *                 (prior counts not included); the first stats[0] entries are valid
 *   stats         [3] int64, OVERWRITTEN: number of distinct tuples, largest digit (-1 when there is none), number of rows
 *                 with an id outside [0, 2^bits) -- those rows get digit -1 and belong to no run
 *   workspace     hv_semid_dedup_workspace_bytes(rows) bytes (0 for rows = 0; 0 = unsupported for rows >= 2^31)
 * Argument errors (bad shape, NULL, small workspace, width * bits > 63, rows >= 2^31) return before any CUDA call.  No
 * allocation and no host synchronisation: CUDA-graph capturable.
 */
size_t hv_semid_dedup_workspace_bytes(int64_t rows);
int hv_semid_dedup(const int64_t* ids, int64_t rows, int64_t width, int64_t row_stride, int64_t col_stride, int bits,
                   const int64_t* prior_keys, const int64_t* prior_counts, int64_t n_prior, int64_t* digits,
                   int64_t digit_stride, int64_t* run_keys, int64_t* run_counts, int64_t* stats, void* workspace,
                   size_t workspace_bytes, void* stream);

/*
 * Gumbel-softmax quantiser level, training mode (modules/quantize.py:108-130,144; distributions/gumbel.py:8-18) -- the
 * [N, K] tables of the reference (dist, noise, logits, weights and their autograd copies) never exist in memory:
 *   dist_k = |x|^2 + |c_k|^2 - 2 x.c_k;  ids = argmin_k dist_k;  g_k = -log(-log(u_k + 1e-20) + 1e-20);
 *   w = softmax((-dist + g) / temperature);  emb_out = w @ codebook;  loss = (1 + beta) |x - emb_out|^2 per row.
 * Noise: `uniforms` [N, K] (the reference's torch.rand draw; parity tests) or, when NULL, counter-based Philox4x32-10
 *   uniforms from (seed, offset) -- the backward regenerates the same draw from the same pair (one call consumes
 *   32 * ceil(K / 128) counters per row starting at `offset`).
 * Forward writes emb_out [N, D], lse [N] (log-sum-exp of the logits, consumed by the backward) and, when non-NULL,
 *   ids [N] int64 and loss [N].
 * Backward: g_emb [N, D] (may be NULL = 0), g_loss [N] (may be NULL = 0) -> g_x [N, D] (overwritten) and g_codebook [K, D]
 *   (ACCUMULATED into: the caller zeroes it).  Gradients are those of the reference's autograd graph: through the softmax
 *   weights and the distance table to x and the codebook, through w @ codebook to the codebook, and the two halves of
 *   QuantizeLoss (modules/loss.py:41-44).
 * Served shapes: D in {16, 32, 64}, K <= 256 (hv_gumbel_supported); others return HV_ERR_UNSUPPORTED.
 * hv_gumbel_uniforms writes the [N, K] uniforms the two kernels generate for (seed, offset): recording a step's draw, and
 *   the test that the Philox path equals the explicit-noise path.
 * The *_devrng entries are their counterparts with the pair in device memory: rng points at two uint64 {seed, offset},
 *   read by the kernels when they run, so a CUDA graph can draw a fresh seed on the device before every replay (the forward
 *   and backward of one replay read the same pair).  A pair gives the same draw as the host scalars of the same values.
 *   Argument errors return before any CUDA call (a NULL rng with n > 0: HV_ERR_NULL); n = 0 is a no-op; like the host-seed
 *   entries they allocate nothing and do not synchronise with the host.
 */
int hv_gumbel_supported(int d, int k);
int hv_gumbel_uniforms(int64_t n, int k, uint64_t seed, uint64_t offset, float* uniforms, void* stream);
int hv_gumbel_forward(const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                      const float* uniforms, uint64_t seed, uint64_t offset, float* emb_out, int64_t* ids, float* loss,
                      float* lse, void* stream);
int hv_gumbel_backward(const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                       const float* uniforms, uint64_t seed, uint64_t offset, const float* emb_out, const float* lse,
                       const float* g_emb, const float* g_loss, float* g_x, float* g_codebook, void* stream);
int hv_gumbel_uniforms_devrng(int64_t n, int k, const uint64_t* rng, float* uniforms, void* stream);
int hv_gumbel_forward_devrng(const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                             const float* uniforms, const uint64_t* rng, float* emb_out, int64_t* ids, float* loss, float* lse,
                             void* stream);
int hv_gumbel_backward_devrng(const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                              const float* uniforms, const uint64_t* rng, const float* emb_out, const float* lse,
                              const float* g_emb, const float* g_loss, float* g_x, float* g_codebook, void* stream);

/*
 * Fused encoder MLP in front of the quantiser: z = [l2norm](W_L silu(... silu(W_1 x))) -- the bias-free Linear + SiLU
 * stack of modules/encoder.py:23-36 as called by HRqVae.encode (modules/h_rqvae.py:599) in eval / bulk-assignment passes
 * (modules/tokenizer/h_semids.py:127).  One kernel: the chain of GEMMs runs on tcgen05 with the hidden activations kept
 * in tensor memory.  Operands are rounded to fp16 (TF32-grade significand: the precision of the reference's own GPU path,
 * modules/h_rqvae.py:21) with round to nearest even and saturation to +-65504; fp16 subnormals are kept.  Products
 * accumulate in fp32 and SiLU is evaluated in fp32; each hidden activation is then rounded to fp16 in the same way, as the
 * next GEMM's operand.  The output layer and the normalisation stay in fp32.
 *   dims        [n_layers + 1] HOST array: input, hidden..., output widths.  Served: {768, 512, 256, 128, 32}; any other
 *               shape returns HV_ERR_UNSUPPORTED / a zero workspace size (the caller keeps its cuBLAS path).
 *   weights     HOST array of n_layers DEVICE pointers, layer l = nn.Linear.weight [dims[l+1], dims[l]] fp32 row-major
 *   workspace   hv_encoder_workspace_bytes(): the fp16 weight image hv_encoder_pack_weights writes once per set of weights
 *   normalize   1: rows of z are L2-normalised (F.normalize, eps 1e-12; MLP(normalize=True))
 *   precise_silu  0: x*sigmoid(x) as h + h*tanh(h), h = x/2 (one MUFU op per element); 1: ex2 + rcp form
 *   z           [N, dims[n_layers]] fp32
 */
size_t hv_encoder_workspace_bytes(int n_layers, const int* dims);
int hv_encoder_pack_weights(const float* const* weights, int n_layers, const int* dims, void* workspace, size_t workspace_bytes,
                            void* stream);
int hv_encoder_forward(const float* x, int64_t n, int n_layers, const int* dims, const void* workspace, size_t workspace_bytes,
                       int normalize, int precise_silu, float* z, void* stream);
/*
 * The same pass for items stored in half precision: x_f16 [N, dims[0]] fp16 row-major (a catalogue kept as fp16 moves half
 * the bytes over PCIe and out of HBM; the reference keeps its item embeddings as a float tensor it slices per batch,
 * modules/tokenizer/h_semids.py:120-127).  hv_encoder_forward rounds fp32 items to fp16 (round to nearest even, saturating
 * to +-65504) before the first GEMM, so items that are the rounded fp32 items give bit-identical z.  That holds for every
 * item with |x| < 65520, where the fp32-to-fp16 conversion (x.half()) is finite.  From 65520 on, x.half() is inf while
 * hv_encoder_forward saturates the entry to +-65504; x.clamp(-65504, 65504).half() gives the fp32 entry's z there too.
 */
int hv_encoder_forward_f16(const void* x_f16, int64_t n, int n_layers, const int* dims, const void* workspace, size_t workspace_bytes,
                           int normalize, int precise_silu, float* z, void* stream);

/*
 * Eval-mode tag heads: per level i the TagPredictor of modules/h_rqvae.py:69-99 (reference h_rqvae.py:108-227) on
 * concat(emb_0 .. emb_i), reduced to argmax and softmax confidence as predict_tags does (reference h_rqvae.py:674-738).
 * The attention gate runs in fp32 on CUDA cores; every Linear after it is a tcgen05 GEMM with fp16 operands (the
 * encoder's numerics), fp32 accumulation, fp32 LayerNorm statistics / softmax / argmax (first index on ties).  Inference
 * only: dropout is the identity and LayerNorm uses its affine parameters.
 *   n_levels, d, first_hidden, class_counts, use_norm   the HRqVae shape: level i has E = d (i+1) inputs, hidden width
 *               H = first_hidden / 2 (i+1), inner width int(0.9 H), class_counts[i] (HOST array) classes; use_norm = 1 when
 *               the heads were built with use_batch_norm=True (nn.LayerNorm), 0 for nn.Identity.  Served: n_levels <= 8,
 *               E <= 128, padded widths <= 4096; otherwise HV_ERR_UNSUPPORTED / a zero size (the caller keeps PyTorch).
 * hv_tag_heads_workspace_bytes  scratch bytes hv_tag_heads_forward needs for `rows` rows (it works on sub-chunks of at
 *               most 18,944 rows, so the size stops growing there); *image_bytes (nullable) receives the image size.
 * hv_tag_heads_pack  params = HOST array of DEVICE fp32 pointers, level by level in TagPredictor.parameters() order
 *               (34 per level with LayerNorm, 22 without); writes the image once per set of weights.
 * hv_tag_heads_forward
 *   emb         level embeddings, element (l, r, c) at emb[l * emb_level_stride + r * emb_row_stride + c] (fp32)
 *   pred_out    int64, level i of row r at pred_out[r * pred_row_stride + i * pred_level_stride] (e.g. the tag columns of
 *               an id table); conf_out (nullable) fp32 the same way
 *   logits_out  nullable HOST array of n_levels nullable DEVICE pointers: fp32 [n, class_counts[i]] logits of level i
 * Nothing else of pred_out / conf_out is written.
 */
size_t hv_tag_heads_workspace_bytes(int n_levels, int d, int first_hidden, const int* class_counts, int use_norm, int64_t rows,
                                    size_t* image_bytes);
int hv_tag_heads_pack(const float* const* params, int n_params, int n_levels, int d, int first_hidden, const int* class_counts,
                      int use_norm, void* image, size_t image_bytes, void* stream);
int hv_tag_heads_forward(const float* emb, int64_t emb_level_stride, int64_t emb_row_stride, int64_t n, int n_levels, int d,
                         int first_hidden, const int* class_counts, int use_norm, const void* image, size_t image_bytes,
                         int64_t* pred_out, int64_t pred_row_stride, int64_t pred_level_stride, float* conf_out,
                         int64_t conf_row_stride, int64_t conf_level_stride, float* const* logits_out, void* workspace,
                         size_t workspace_bytes, void* stream);

/*
 * Data-parallel exchange of a small fp32 buffer (the codebook gradient, train_hidvae.py's DDP all-reduce) as ONE kernel
 * over NVLink / NVSwitch peer memory: every rank pushes its contribution into an inbox slot on every peer, flags it,
 * waits for its peers' flags and sums the slots in rank order (bit-identical results on every rank).
 *   n           floats, multiple of 4
 *   inbox_ptrs  device array [world] of the ranks' inbox bases as mapped in THIS process (symmetric allocation of
 *               2 * world * n floats per rank); flag_ptrs likewise for 2 * world * hv_peer_allreduce_chunks(n) uint32 flags
 *               (zero before the first call); seq: hv_peer_allreduce_chunks(n) + 1 private uint32 words (zero before the
 *               first call): the call counters and one sticky STATUS word.  Every rank must make the same sequence of
 *               calls, and consecutive calls on one set of inboxes must be ordered (one stream, or an event between them).
 *               CUDA-graph capturable.
 * A rank that does not show up within the timeout (default 10 s of wall time; hv_peer_allreduce_set_timeout_ms, 0 = wait for
 * ever) does not trap the kernel: the wait is abandoned, the status word (seq[chunks]) is set and the call's result is
 * invalid.  The caller copies that word to the host when it synchronises and passes it to hv_peer_allreduce_status
 * (HV_OK, or HV_ERR_CUDA with the missing rank / chunk).
 */
int hv_peer_allreduce_chunks(int64_t n);
void hv_peer_allreduce_set_timeout_ms(int64_t ms);
int hv_peer_allreduce_status(uint32_t status_word, int* missing_rank, int* chunk);
int hv_peer_allreduce(const float* src, float* dst, int64_t n, const uint64_t* inbox_ptrs, const uint64_t* flag_ptrs,
                      uint32_t* seq, int rank, int world, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HIDVAE_B200_H_ */
