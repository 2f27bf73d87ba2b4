/*
 * ganrev.h -- C ABI of libganrev_cuda.so, the B200-native (sm_100a) replacement for
 * the arithmetic under aleju/gan-reverser's apply_r.lua.
 *
 * The reference has no plugin / FFI interface of its own: apply_r.lua calls Torch7
 * objects directly.  The boundary is therefore the set of Lua calls apply_r.lua makes;
 * each entry point below names the reference call site (file:line in
 * aleju/gan-reverser) it stands behind.  INTEGRATION.md shows the LuaJIT-FFI binding.
 *
 * Conventions
 *  - All host tensors are contiguous row-major; float32 unless stated; images NCHW
 *    (exactly what FloatTensor:data() yields).  Ids are 0-based (the Lua shim adds 1).
 *  - Every call returns GANREV_OK (0) or an error code; ganrev_last_error() gives the
 *    message.  No exceptions, no abort(), and NO CPU FALLBACK: without an sm_100
 *    device ganrev_create() fails.
 *  - The caller owns every host buffer; the library owns all device memory.  Calls are
 *    synchronous: outputs are valid on return.  A ctx is driven by one host thread.
 *  - Dropout is never drawn inside the library: R's input mask is an explicit argument
 *    (uint8, 1 = keep) with the reference's semantics x*mask, no 1/(1-p) rescale
 *    (models.lua:399-406).
 *  - Resident buffers: every forward leaves its result on the device (G -> IMAGES,
 *    R slot s -> ATTRS_s, fix -> FIXED).  A NULL *input* pointer means "use the
 *    resident buffer"; a NULL *output* pointer means "keep it resident, do not copy
 *    back" (1M 32x32 fp32 faces are 4.1 GB; returning them costs more than making them).
 *
 * Weight blob (ganrev_load_G / ganrev_load_R): every parameter, float32, concatenated in
 * models.lua module order.  Conv weight [Cout][Cin][3][3] then bias [Cout]; Linear weight
 * [out][in] then bias [out]; each BatchNorm as gamma, beta, running_mean, running_var
 * ([C] each), eps = 1e-5.
 *   G (models.lua:115-132): Linear(nd -> 512*H/4*W/4), BN, Conv 512->256, BN,
 *                           Conv 256->128, BN, Conv 128->C.
 *   R (models.lua:409-451): 6 x (Conv, BN) with channels C->64->64->64->128->128->128,
 *                           Linear(128*H/4*W/4 -> 512), BN, Linear(512 -> nd).
 *
 * New work beyond the reference is marked as such: multi-GPU sharding and the refinement of recovered noise
 * vectors by gradient descent through G (ganrev_refine_l2).
 *
 * One geometry per context: G, R and R_fixer of apply_r.lua share {C, H, W, noiseDim}
 * (apply_r.lua:65-79) and the resident buffers are sized by it.  Loading a model with a
 * DIFFERENT geometry unloads the models of the old geometry and empties every resident
 * buffer, so nothing sized for the old geometry can be read or written afterwards.
 */
#ifndef GANREV_H
#define GANREV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GANREV_OK      0
#define GANREV_EINVAL  1   /* bad argument / unsupported geometry */
#define GANREV_ECUDA   2   /* CUDA runtime or kernel error */
#define GANREV_ENODEV  3   /* no sm_100 device */
#define GANREV_ESTATE  4   /* model / db / buffer not loaded */
#define GANREV_ENCCL   5   /* NCCL unavailable or failed */
#define GANREV_ENOMEM  6

/* resident device buffers (see "Resident buffers" above) */
#define GANREV_BUF_NOISE   0   /* [rows x nd]        float32 */
#define GANREV_BUF_IMAGES  1   /* [rows x C x H x W] float32 */
#define GANREV_BUF_ATTRS0  2   /* [rows x nd]        float32, output of R slot 0 */
#define GANREV_BUF_ATTRS1  3   /* [rows x nd]        float32, output of R slot 1 (fixer) */
#define GANREV_BUF_FIXED   4   /* [rows x C x H x W] float32, G(R_fixer(images)) */
#define GANREV_BUF_MASK    5   /* [rows x C x H x W] uint8 */
#define GANREV_BUF_COUNT   6

typedef struct ganrev_ctx ganrev_ctx;

int         ganrev_version(void);
/* One context = one GPU (one process per GPU under torchrun / one Lua state per GPU).
 * Replaces cutorch.setDevice (apply_r.lua:52-56). */
int         ganrev_create(ganrev_ctx** out, int device);
void        ganrev_destroy(ganrev_ctx* ctx);
const char* ganrev_last_error(const ganrev_ctx* ctx);   /* valid until the next call on ctx */

/* ---- multi-GPU (new work; the reference is single-device) ------------------------
 * Rank 0 makes a unique id, the launcher (torch.distributed / MPI / a file) hands it
 * to every rank, every rank calls ganrev_comm_init.  NCCL is dlopen()ed on first use.
 * After init the database of ganrev_db_set is one row-shard of a global database:
 * search merges per-rank top-k with one allgather, kmeans sums centroid accumulators
 * with one allreduce per iteration.  G / R need no communication. */
int ganrev_comm_unique_id(ganrev_ctx* ctx, void* out, size_t cap, size_t* len);
int ganrev_comm_init(ganrev_ctx* ctx, int world, int rank, const void* uid, size_t len);

/* ---- models ---------------------------------------------------------------------
 * MODELS.create_G(dimensions, noiseDim, cuda)   models.lua:201-203 -> create_G3 :104-143
 * MODELS.create_R(dimensions, noiseDim, noiseMethod, fixer, cuda)  models.lua:385-464
 * slot 0 = R (apply_r.lua:92-94), slot 1 = R_fixer (apply_r.lua:97-104).
 * tanh_out = (noiseMethod ~= "normal")  models.lua:452-454. */
int ganrev_load_G(ganrev_ctx* ctx, int C, int H, int W, int noise_dim,
                  const float* blob, size_t n_floats);
int ganrev_load_R(ganrev_ctx* ctx, int slot, int C, int H, int W, int noise_dim, int tanh_out,
                  const float* blob, size_t n_floats);

/* NN_UTILS.forwardBatched(MODEL_G, noise, batchSize)   utils/nn_utils.lua:5-33,
 * apply_r.lua:136,146,349.  noise [N x nd] -> images [N x C x H x W] in [0,1]. */
int ganrev_forward_G(ganrev_ctx* ctx, const float* noise, int64_t N, float* images);
/* NN_UTILS.forwardBatched(MODEL_R / MODEL_R_FIXER, images, batchSize)  apply_r.lua:152-153.
 * mask may be NULL (no input dropout).  images [N x C x H x W] -> attrs [N x nd]. */
int ganrev_forward_R(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask,
                     int64_t N, float* attrs);
/* fixFaces / detectAnomalies inner loop, batched: attrs = R_slot(images, mask);
 * fixed = G(attrs); l2[i] = torch.dist(images[i], fixed[i]).  apply_r.lua:328-332,349,361-366.
 * attrs, fixed, l2 may each be NULL. */
int ganrev_fix_l2(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask, int64_t N,
                  float* attrs, float* fixed, double* l2);
/* torch.dist(a[i], b[i]) for N pairs of px-element vectors (apply_r.lua:366). */
int ganrev_l2(ganrev_ctx* ctx, const float* a, const float* b, int64_t N, int px, double* l2);
/* SURVEY 8(f) rank 3 -- findClosestNeighboursOf   sample.lua:128-148: for each of Q query images [Q x px] the
 * row of `set` [N x px] (NULL = the first N resident IMAGES) with the smallest torch.dist, first strict minimum
 * in row order (row 0 is always taken first, so a NaN there sticks, as in the Lua loop).  ids [Q] 0-based
 * (-1 when N == 0), dist [Q] (+inf when N == 0).  After ganrev_comm_init each rank passes ITS row shard of the set
 * (shards in rank order); ids are then global rows and every rank returns the same answer (one allgather of Q records). */
int ganrev_nearest_l2(ganrev_ctx* ctx, const float* queries, int Q, const float* set, int64_t N, int px,
                      int64_t* ids, double* dist);
/* apply_r.lua:370-378: sims = 1 - l2; thr = ascending sims[floor(n_calc*quantile)] (1-based);
 * flags[i] = sims[i] <= thr, i < n_show.  thr may be NULL.  l2 == NULL reuses the distances the last ganrev_fix_l2 /
 * ganrev_refine_l2 / ganrev_l2 call left on the device (GANREV_ESTATE if it left fewer than n_calc).  After ganrev_comm_init l2 / n_calc /
 * n_show describe this rank's shard (n_calc may be 0): the order statistic is taken over all ranks' n_calc values by a
 * device radix select with one 256-bin allreduce per pass; flags are this rank's first n_show. */
int ganrev_anomaly_flags(ganrev_ctx* ctx, const double* l2, int64_t n_calc, int64_t n_show,
                         double quantile, uint8_t* flags, double* thr);

/* ---- resident buffers ----------------------------------------------------------- */
int ganrev_buffer_put(ganrev_ctx* ctx, int which, const void* host, int64_t rows);
int ganrev_buffer_get(ganrev_ctx* ctx, int which, void* host, int64_t row0, int64_t rows);

/* ---- recovered-vector database --------------------------------------------------
 * vecs [N x d] becomes this rank's row shard.  vecs == NULL: the first N resident ATTRS0 rows ARE the shard -- the
 * database aliases that buffer (the recovered vectors stay where R left them, no copy); overwriting ATTRS0 afterwards
 * (ganrev_forward_R / ganrev_fix_l2 with slot 0, ganrev_buffer_put) un-sets the database. */
int ganrev_db_set(ganrev_ctx* ctx, const float* vecs, int64_t N, int d);
/* cosineSimilarity(v1, v2)   apply_r.lua:396-400 (nn.CosineDistance). */
int ganrev_cosine(ganrev_ctx* ctx, const float* a, const float* b, int d, float* out);
/* createSimilaritySearchImages inner loops   apply_r.lua:267-282: for each query the k
 * best rows by (cosine desc, id asc), NaN last.  ids [Q x k] global 0-based row ids
 * (-1 past the end of the database), scores [Q x k].  k <= 128. */
int ganrev_search_cosine(ganrev_ctx* ctx, const float* queries, int Q, int k,
                         int64_t* ids, float* scores);
/* The same search with the queries given as database rows ("search by example"): apply_r.lua's
 * needles are rows i*100 of the searched tensor itself (apply_r.lua:268-272).  rows [Q] are global
 * 0-based row ids; the query vectors never leave the device (across ranks they are assembled with
 * one integer max-allreduce). */
int ganrev_search_rows(ganrev_ctx* ctx, const int64_t* rows, int Q, int k, int64_t* ids, float* scores);
/* unsup.kmeans(x, k, niter)   apply_r.lua:198.  init_centroids [k x d] is explicit
 * (unsup draws N(0,1) rows and normalises them; the shim does that and passes them in).
 * total_counts [k] = counts summed over iterations; last_labels [N local rows] or NULL. */
int ganrev_kmeans(ganrev_ctx* ctx, int k, int niter, const float* init_centroids,
                  float* centroids, float* total_counts, int32_t* last_labels);
/* createClusterImages assignment loop   apply_r.lua:206-218: per row the cluster with the
 * MINIMUM cosine (strict <, lowest index on ties) and that cosine. */
int ganrev_assign_cosine_min(ganrev_ctx* ctx, const float* centroids, int k,
                             int32_t* cluster, float* cosv);
/* apply_r.lua:222-243: per cluster keep <= m members by (cos desc, id asc) and average
 * their images (images NULL = resident IMAGES; px = C*H*W).  member_ids [k x m] (-1
 * padded), member_counts [k], mean_images [k x px] (NULL to skip).  m <= 128.
 * Uses the result of the last ganrev_assign_cosine_min.  After ganrev_comm_init the database and `images` are this rank's
 * row shards: member ids are global rows, merged like the search (one allgather of k*m keys, one allreduce of k counts);
 * the kept images are assembled across ranks with an integer allreduce and every rank returns the same lists and means. */
int ganrev_cluster_members(ganrev_ctx* ctx, int k, int m, const float* images, int px,
                           int64_t* member_ids, int32_t* member_counts, float* mean_images);

/* ---- R training step (train_r.lua:138-170; SURVEY.md 8f rank 4) ------------------------------------------------
 * One optimisation step of R on a batch generated by the loaded G: images = G(noise) in eval mode (train_r.lua:140-141),
 * R_default (models.lua:389-464) forward in TRAINING mode (batch-norm batch statistics, running statistics updated with
 * momentum 0.1), nn.MSECriterion against the noise, backward, L1 / L2 penalties and gradient clamp (train_r.lua:150-163),
 * optim.adam.  Dropout is never drawn inside the library: `masks` is the concatenation of the uint8 keep-masks (1 = keep)
 *   [fixer only: B x C x H x W (nn.Dropout(0.5, true), v1: no rescale)] | B x 64 x H x W | B x 64 x H x W | B x 64 x H/2 x W/2 |
 *   B x 128 x H/2 x W/2 | B x 128 x H/2 x W/2 | B x 128 (nn.SpatialDropout(0.25): per sample and channel) | B x 512,
 * in module order (nn.Dropout() v2: kept values are scaled by 2).  State (fp32 parameters in weight-blob layout, Adam moments,
 * step count) lives in the context: train_R_init takes the same blob as ganrev_load_R; train_R_state returns the blob
 * (what = 0, ready for ganrev_load_R), the last step's gradients after penalties and clamp (1), or Adam's m / v (2 / 3).
 * hyper7 = {learning rate, beta1, beta2, epsilon, L1, L2, clamp (0 = off)}; optim.adam's defaults are {1e-3, 0.9, 0.999, 1e-8},
 * train_r.lua's {.., 0, 1e-4, 1}.  loss2[0] = the criterion's output, loss2[1] = with the penalties (feval's f). */
int ganrev_train_R_init(ganrev_ctx* ctx, int C, int H, int W, int noise_dim, int tanh_out, int fixer, const float* blob, size_t n_floats);
int ganrev_train_R_step(ganrev_ctx* ctx, const float* noise, int B, const uint8_t* masks, size_t mask_bytes, const float* hyper7, double* loss2);
int ganrev_train_R_state(ganrev_ctx* ctx, int what, float* out, size_t n_floats);

/* ---- noise-vector refinement (new work; the reference stops at R's single pass, apply_r.lua:152-153) --------------
 * For each image x_i, `iters` steps of Adam (optim.adam's update, as ganrev_train_R_step applies it) on
 *   f(z) = ||G(z) - x_i||^2 + prior * ||z||^2,  then, if zclamp > 0, |z| <= zclamp elementwise after every step.
 * hyper6 = {lr, beta1, beta2, eps, prior, zclamp}.  images NULL = resident IMAGES; z0 NULL = the first N rows of resident
 * ATTRS_slot (GANREV_ESTATE if it holds fewer).  The refined vectors are left in ATTRS_slot (slot 0: un-sets an aliasing
 * database, as ganrev_fix_l2 does), G(z_final) in FIXED, and l2[i] = torch.dist(x_i, G(z_final)) stays on the device for
 * ganrev_anomaly_flags(l2 = NULL); fixed and l2 are exactly ganrev_forward_G(z_final) + ganrev_l2, and iters = 0 is the fix
 * path applied to z0.  attrs / fixed / l2 may be NULL.  GANREV_EINVAL for iters < 0, lr <= 0 or prior < 0.  Deterministic,
 * independent of the chunk size and of which other images share the call.  The gradient is G's backward pass on the tensor
 * cores, built on the first call (not at ganrev_load_G).  Image-sharded: after ganrev_comm_init every rank refines its own
 * rows, and the call makes no collective. */
int ganrev_refine_l2(ganrev_ctx* ctx, int slot, const float* images, const float* z0, int64_t N, int iters,
                     const float* hyper6, float* attrs, float* fixed, double* l2);
/* Tests: grad [N x nd] = the gradient of f at z and f [N], one forward + backward (no optimiser step). */
int ganrev_debug_refine_grad(ganrev_ctx* ctx, const float* images, const float* z, int64_t N, float prior,
                             float* grad, double* f);
/* Tests: one forward + backward pass of G as ganrev_refine_l2 runs it, stopped after `stage`, whose buffer is copied to out
 * (rows in input order, every chunk): 0 h0 [N][H/4][W/4][512] bf16, 1 h1 [N][H/2][W/2][256] bf16, 2 h2 [N][H][W][128] bf16,
 * 3 y [N][C][H][W] f32, 4 e2 [N][H][W][128] bf16, 5 e1 [N][H/2][W/2][256] bf16, 6 e0 [N][H/4][W/4][512] bf16, 7 glin [N][nd] f32
 * (glin + 2 prior z is ganrev_debug_refine_grad's gradient).  GANREV_EINVAL for another stage or an out_bytes that does not match. */
int ganrev_debug_refine_stage(ganrev_ctx* ctx, const float* images, const float* z, int64_t N, int stage, void* out,
                              size_t out_bytes);
/* Tests: G's forward pass as ganrev_forward_G runs it, chunk by chunk, stopped after layer `stage`, whose buffer is copied to out
 * (rows in input order): 0 lin [N][H/4][W/4][512] bf16, 1 c1 [N][H/2][W/2][256] bf16, 2 c2 [N][H][W][128] bf16 (GANREV_ESTATE when
 * the last conv's tap products are fused into conv2: h2 is never stored then), 3 taps [N][9C][H][W] f32 (plane tap*C + co),
 * 4 y [N][C][H][W] f32.  GANREV_EINVAL for another stage or an out_bytes that does not match. */
int ganrev_debug_G_stage(ganrev_ctx* ctx, const float* noise, int64_t N, int stage, void* out, size_t out_bytes);
/* Tests: the same for R of `slot` (mask as ganrev_forward_R): 0..5 conv1..conv6 bf16 NHWC ([N][H][W][64], [N][H][W][64],
 * [N][H/2][W/2][64] pooled, [N][H/2][W/2][128], [N][H/2][W/2][128], [N][H/4][W/4][128] pooled), 6 l1 [N][512] bf16, 7 out [N][nd] f32. */
int ganrev_debug_R_stage(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask, int64_t N, int stage, void* out,
                         size_t out_bytes);

/* ---- measurement hooks (bench.py) ----------------------------------------------- */
void*    ganrev_stream(ganrev_ctx* ctx);                 /* cudaStream_t all work runs on */
int      ganrev_sync(ganrev_ctx* ctx);
uint64_t ganrev_launch_count(const ganrev_ctx* ctx);     /* kernels launched so far */
/* Per-kernel CUDA-event timing on the library's stream. */
int ganrev_profile_enable(ganrev_ctx* ctx, int on);
int ganrev_profile_reset(ganrev_ctx* ctx);
int ganrev_profile_count(ganrev_ctx* ctx);
int ganrev_profile_get(ganrev_ctx* ctx, int idx, const char** name, uint64_t* launches,
                       double* total_ms, double* flops, double* bytes);
/* bench.py: a synthetic N(0,1) [N x d] database generated on the device (counter-based on seed and GLOBAL element index:
 * global_row0 = this shard's first global row) and adopted as by ganrev_db_set; the measured fp32 FMA roof of this GPU. */
int ganrev_debug_db_synthetic(ganrev_ctx* ctx, int64_t N, int d, uint64_t seed, int64_t global_row0);
int ganrev_debug_fma_peak(ganrev_ctx* ctx, double* tflops);
/* Tests: the tensor-core filter's approximate cosine of every (query, row) pair of a small database, out [Q x N], and the
 * error bound eps(d) the filter assumes (search_tc.cuh); how many searches the tensor-core path served [0] / handed to the
 * fmaf-chain kernels after raising a flag [1]. */
int ganrev_debug_tc_scores(ganrev_ctx* ctx, const float* queries, int Q, float* out, float* eps_out);
int ganrev_debug_tc_counters(ganrev_ctx* ctx, uint64_t* out2);
/* Tests / bench: counters of the TMA -> tf32 filter pipeline (stream_tc.cuh) since the last call, then reset: [0] (row, needle /
 * centroid) pairs that needed an exact chain on top of the filter, [1] rows handed to the every-chain list kernel, [2] the
 * largest observed |approximate - exact| over the assumed bound (float bits; only measured under "dbg" bit 18), [3] launches. */
int ganrev_debug_tfs_stats(ganrev_ctx* ctx, uint64_t* out4);
/* Debug: clock64 timeline of CTA 0 of the named tensor-core layer (roles x events, [8][256]). */
int ganrev_debug_trace_arm(ganrev_ctx* ctx, const char* layer);
int ganrev_debug_trace_read(ganrev_ctx* ctx, int64_t* out);
/* Tuning / debugging knobs (exact outputs are unaffected; conv_impl 1 differs within the conv tolerance; dbg invalidates results):
 *   "chunk"     images per pipeline chunk; 0 = default = 8192 32x32 faces' worth of pixels
 *   "conv_impl" 0 = tcgen05 implicit GEMM (default), 1 = plain CUDA-core kernels kept for on-device A/B checks
 *   "cta_pairs" bit mask of the conv layers that run as tcgen05 cta_group::2 CTA pairs (default all; read at ganrev_load_*: bit 4 also
 *               selects it for the refinement's conv2^T / conv1^T, built later from the value ganrev_load_G saw)
 *   "fuse_conv3" 1 = C == 1: the tap products of G's last conv come out of conv2's epilogue (default), 2 = also C == 3 (measured
 *               slower), 0 = separate 1x1 tensor-core pass over the stored activation; read at ganrev_load_G
 *   "xpose2"    1 = second store-transpose buffer per epilogue warp for G's Linear (default), 2 = every plain bf16 layer, 0 = none;
 *               read at ganrev_load_*.  "tma_hybrid" 1 = first chunk of an epilogue round by st.global, second by TMA store (default 0)
 *   "ups_cycles" MMA cycles a conv pipeline stage should carry (units per stage; default 512, G's first Up+Conv uses >= 1024); read at load time
 *   "pdl"       1 = conv layers launched with programmatic stream serialization (griddepcontrol: the next layer's prologue overlaps
 *               this layer's tail; measured +0.4 %, within noise), 0 = plain stream order (default)
 *   "tma_store" 1 = TMA bulk tensor stores in the conv epilogue of the plain layers (default), 2 = also the pooled layers, 0 = st.global everywhere
 *   "search_tc" 1 = many-query searches (Q >= 48, >= 8192 rows per rank) run as tensor-core candidate filter + exact re-score (default;
 *               results are bit-identical), 0 = fmaf-chain kernels only
 *   "stream_tc" 1 = searches with <= 32 needles, kmeans with k <= 32 and the cosine-min assignment (d % 4 == 0) run as TMA -> tf32
 *               tcgen05 filter + exact chains for the candidates / near-ties only (default; results are bit-identical), 0 = fmaf-chain kernels
 *   "label_tc"  1 = kmeans / cosine-min labelling for k <= 32, d % 4 == 0, d <= 128 on the tensor cores, exact chains only for near-ties
 *               (results are bit-identical; measured no faster than the register-tiled kernels yet), 0 = fmaf-chain kernels (default)
 *   "kmeans_tc" 1 = kmeans labelling for k > 32 on the tensor cores with exact chains only for near-ties (default; bit-identical), 0 = off
 *   "rtile"     1 = register-tiled kmeans / cosine-min kernels for 9 <= k <= 32 (default), 0 = one-thread-per-row streaming kernels
 *   "dbg"       timing experiments: bit 0 skip A loads, 1 skip B loads, 2 skip epilogue, 3 skip MMAs, 4 skip stores (results invalid) */
int ganrev_set_option(ganrev_ctx* ctx, const char* name, int64_t value);

#ifdef __cplusplus
}
#endif
#endif
