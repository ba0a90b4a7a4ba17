/*
 * ac_b200.h -- C ABI of libac_b200.so: the B200-native (sm_100a) embedding-to-distance path of
 * KevinWangHP/Anomaly-Clustering.
 *
 * The reference is 100 % Python: it has no FFI for this path, the "interface" is the Python call
 * surface of Anomaly-Clustering/models/patchcore/{patchcore,common,utils}.py and examples/main.py.
 * Each entry point below names the reference lines it replaces.  A maintainer binds these with
 * ctypes (see INTEGRATION.md); anomaly_clustering_b200/_lib.py is exactly that binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns every buffer,
 *     including the workspace; the library allocates no device memory and keeps no global state
 *     except a small mutex-protected host cache of launch plans (pure functions of the shapes);
 *   - every call is asynchronous and ordered on `stream` (a cudaStream_t); no hidden synchronisation;
 *   - return value: 0 on success, a negative AC_ERR_* code otherwise (never throws, never aborts);
 *   - there is NO CPU fallback: on anything that is not compute capability 10.x the calls fail with
 *     AC_ERR_DEVICE.
 */
#ifndef AC_B200_H
#define AC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AC_OK 0
#define AC_ERR_INVALID (-1)     /* bad argument (null pointer, non-positive size, ...)            */
#define AC_ERR_UNSUPPORTED (-2) /* shape outside what the kernels implement (stated per function) */
#define AC_ERR_DEVICE (-3)      /* current device is not sm_100 (B200)                            */
#define AC_ERR_CUDA (-4)        /* a CUDA runtime / driver call failed (see ac_last_cuda_error)   */
#define AC_ERR_WORKSPACE (-5)   /* workspace too small                                            */

/* operand element types (for the tensor-core operands and ac_row_norms) */
#define AC_DT_F32 0
#define AC_DT_F16 1
#define AC_DT_BF16 2

/* precision modes of ac_min_dist */
#define AC_PREC_F16 0    /* tcgen05 kind::f16, fp16 operands, fp32 accumulate (1 MMA pass)          */
#define AC_PREC_BF16 1   /* tcgen05 kind::f16, bf16 operands                                        */
#define AC_PREC_F16X3 2  /* split fp16 hi+lo, hi*hi + lo*hi + hi*lo in one accumulator (3 passes)   */
#define AC_PREC_BF16X3 3 /* split bf16 hi+lo, 3 passes                                              */
#define AC_PREC_F32 4    /* exact fp32 SIMT kernel, sum (x-y)^2, no tensor cores                    */

/* reduce modes of ac_reduce_weights */
#define AC_REDUCE_MEAN 0 /* unsupervised: mean over bank images (self excluded)  utils.py:227 */
#define AC_REDUCE_MIN 1  /* supervised:   min over bank images                   utils.py:236 */
#define AC_REDUCE_MIN_UPDATE 2 /* supervised, grown bank: min of w (read) and of the given bank images */

typedef void* ac_stream_t; /* cudaStream_t */

/* One hooked backbone feature map, read IN PLACE through strides (elements, not bytes):
 * CNN maps [B,C,H,W] contiguous: sb=C*H*W, sc=H*W, sh=W, sw=1.
 * ViT block outputs [B,1+P,C] (models/patchcore/patchcore.py:377-383 drops CLS and permutes):
 *   ptr = tokens + C (skips CLS), sb=(1+P)*C, sc=1, sh=W*C, sw=C -- no permuted copy is made. */
typedef struct {
  const float* ptr;
  int32_t C, H, W;
  int64_t sb, sc, sh, sw;
} ac_layer_t;

/* ---- library / device ------------------------------------------------------------------------ */
int ac_version(void);
const char* ac_strerror(int code);
/* 0 if device `dev` is compute capability 10.x, AC_ERR_DEVICE otherwise. */
int ac_device_ok(int dev);
/* cudaError_t of the last failing CUDA call made by this library on this thread (0 if none). */
int ac_last_cuda_error(void);
/* Pipeline watchdog of the tensor-core kernels (ac_min_dist*): a role that waits > ~10 s on an mbarrier records which
 * wait it was in host-mapped memory and traps, so the launch fails instead of hanging the GPU; the sticky CUDA error
 * surfaces at the caller's next synchronisation.  Returns that code (0 = never fired; 1 producer waits for a free stage,
 * 2 MMA issuer waits for a TMEM buffer, 3 MMA issuer waits for operands, 4 epilogue waits for an accumulator,
 * 5 / 6 unit queue) and clears it.  Readable after the trap because the flag lives in pinned host memory. */
int ac_last_watchdog(void);

/* ---- stage 1: feature maps -> patch embeddings Z ----------------------------------------------
 * Replaces AnomalyClusteringCore._embed after the backbone (models/patchcore/patchcore.py:368-431):
 * whole-map LayerNorm (:384-385), PatchMaker.patchify (:439-465), cross-layer bilinear resize
 * (:398-421), Preprocessing/MeanMapper (models/patchcore/common.py:145-170), Aggregator (:173-183),
 * in one fused kernel (+ a per-image statistics pre-pass).  No im2col tensor is materialised.
 *
 *   layers_host : HOST array of L descriptors
 *   Z           : [B*P, D] fp32 or NULL         P = patch grid of layer 0
 *   Zhi, Zlo    : [B*P, D] op_dtype (AC_DT_F16/AC_DT_BF16) or NULL: hi = round(Z), lo = round(Z-hi),
 *                 the tensor-core operands of ac_min_dist
 *   layernorm   : 1 = AnomalyClusteringCore._embed, 0 = PatchCore._embed (patchcore.py:92-146)
 * Workspace: ac_embed_workspace_bytes(layers_host, L, B, patchsize, stride, Dp, D) (statistics partials,
 * chunk table, and -- only for CNN-layout or resampled layers -- channel-contiguous / coarse-grid scratch).
 * ws must be 16-byte aligned, else AC_ERR_INVALID.  Z, Zhi and Zlo may have any element alignment: an output whose
 * base pointer is 16-byte aligned is written with 16-byte vector stores where the row pitch allows, any other with
 * scalar stores, and the bits written are the same either way. */
size_t ac_embed_workspace_bytes(const ac_layer_t* layers_host, int L, int B, int patchsize, int stride, int Dp,
                                int D);
int ac_embed(const ac_layer_t* layers_host, int L, int B, int patchsize, int stride, int Dp, int D,
             int layernorm, float eps, float* Z, void* Zhi, void* Zlo, int op_dtype, void* ws,
             size_t ws_bytes, ac_stream_t stream);
/* Same, and n2 [B*P] (may be NULL) receives the squared norms of the operand rows (hi, or hi + lo) that
 * ac_min_dist needs -- emitted by the embed kernel itself when the single-pass fused form applies (all layers
 * channel-contiguous, of one shape, 16-byte aligned: ViT tokens), by ac_row_norms otherwise.  Needs Zhi. */
int ac_embed_ex(const ac_layer_t* layers_host, int L, int B, int patchsize, int stride, int Dp, int D,
                int layernorm, float eps, float* Z, void* Zhi, void* Zlo, int op_dtype, float* n2, void* ws,
                size_t ws_bytes, ac_stream_t stream);

/* 16-bit backbone feature maps (a backbone run in bf16 or fp16): the same as ac_embed_ex / ac_embed_workspace_bytes
 * with every layer's ptr read as feat_dtype elements (AC_DT_F32, AC_DT_F16 or AC_DT_BF16, one type for all layers);
 * strides stay in elements.  Each 16-bit value is widened to fp32 as it is loaded and the LayerNorm and everything
 * after it run in fp32, so every output is BIT-IDENTICAL to the fp32 call on the upcast maps with the same strides and
 * the same element offsets.  (The forms that stage rows with bulk copies need 16-byte aligned rows: C % 8 == 0 for
 * 16-bit maps; the statistics pre-pass picks its vector loads from the element offset of each image, offset % 4 == 0.)
 * The workspace of a 16-bit call also holds an fp32 channel-contiguous copy of each map for the per-layer forms.
 * An unknown feat_dtype: AC_ERR_INVALID (workspace: 0). */
size_t ac_embed_workspace_bytes_dt(const ac_layer_t* layers_host, int L, int feat_dtype, int B, int patchsize, int stride,
                                   int Dp, int D);
int ac_embed_dt(const ac_layer_t* layers_host, int L, int feat_dtype, int B, int patchsize, int stride, int Dp, int D,
                int layernorm, float eps, float* Z, void* Zhi, void* Zlo, int op_dtype, float* n2, void* ws,
                size_t ws_bytes, ac_stream_t stream);

/* PatchMaker.patchify standalone (models/patchcore/patchcore.py:439-465):
 * x [B,C,H,W] contiguous -> out [B, h*w, C, k, k]; grid_host[2] receives (h, w). */
int ac_patchify(const float* x, int B, int C, int H, int W, int patchsize, int stride, float* out,
                int* grid_host, ac_stream_t stream);

/* F.adaptive_avg_pool1d over the last axis: in [rows, Lin] -> out [rows, Lout].
 * MeanMapper.forward (common.py:168-170) and Aggregator.forward (common.py:178-183). */
int ac_adaptive_pool1d(const float* in, int64_t rows, int Lin, int Lout, float* out,
                       ac_stream_t stream);

/* hi = round_to(dtype, x), lo = round_to(dtype, x - hi)  (lo may be NULL).  n elements. */
int ac_split_operand(const float* x, int64_t n, void* hi, void* lo, int dtype, ac_stream_t stream);

/* n2[r] = sum_d A[r,d]^2 in fp32; A is [rows, D] of `dtype`; if A2 != NULL the row is A + A2
 * (hi + lo operands). */
int ac_row_norms(const void* A, const void* A2, int dtype, int64_t rows, int D, float* n2,
                 ac_stream_t stream);

/* ---- stage 2: patch-versus-bank nearest neighbour ----------------------------------------------
 * Replaces the torch.cdist + torch.min(dim=1) loops of Weight_Distance_Unsupervised / _Supervised
 * (models/patchcore/utils.py:222-237):
 *   dmin[j*Mq + r] = min over the P rows q of bank image j of || Q[r] - Bank[j*P+q] ||_2
 * computed as sqrt(max(0, |q|^2 + |b|^2 - 2 q.b)) with the dot products on the tcgen05 tensor cores
 * (TMA-fed, fp32 accumulation in TMEM) and the per-bank-image row-min fused into the epilogue: the
 * [Mq, nb_img*P] distance matrix never reaches HBM.  AC_PREC_F32 runs an exact SIMT kernel instead.
 *
 *   Qhi/Qlo [Mq, D], Bhi/Blo [nb_img*P, D] : operands of the dtype implied by `precision`
 *             (fp32 for AC_PREC_F32; lo only for the X3 modes, else NULL)
 *   Qn2 [Mq], Bn2 [nb_img*P] : fp32 squared norms of the operands (ac_row_norms), unused for F32
 *   dmin [nb_img, Mq] fp32
 * Tensor-core modes need D % 8 == 0 (TMA row pitch), else AC_ERR_UNSUPPORTED.
 * Workspace: ac_min_dist_workspace_bytes(). */
size_t ac_min_dist_workspace_bytes(int64_t Mq, int nb_img, int P, int D, int precision);
int ac_min_dist(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, const void* Bhi,
                const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision,
                float* dmin, void* ws, size_t ws_bytes, ac_stream_t stream);

/* w[r] = mean_j dmin[j, r] over bank images j != q_self[r / Pq]   (AC_REDUCE_MEAN, utils.py:227)
 *      = min_j  dmin[j, r]                                           (AC_REDUCE_MIN,  utils.py:236)
 *      = min(w[r], min_j dmin[j, r])                                 (AC_REDUCE_MIN_UPDATE)
 * q_self: [ceil(Mq/Pq)] int32 bank-image index of each query image, -1 or NULL = none.
 * AC_REDUCE_MIN_UPDATE reads w as a running minimum: a supervised bank that gains images passes the distances to the new
 * images only (dmin [K, Mq]) and gets the minimum over the whole bank, bit-identical to AC_REDUCE_MIN over all of it
 * because a min of fp32 values does not depend on the order it is taken in.  q_self and groups mean what they mean for
 * AC_REDUCE_MIN.  Any other mode is AC_ERR_INVALID. */
int ac_reduce_weights(const float* dmin, int64_t Mq, int nb_img, int Pq, const int32_t* q_self,
                      int mode, float* w, ac_stream_t stream);

/* Symmetric form of the unsupervised case (SURVEY.md section 8f row 4): the queries are images
 * [q_img0, q_img0 + Mq/P) OF the bank (Q = B + q_img0*P*D), and torch.cdist(Z[i], Z[j]) is the transpose
 * of torch.cdist(Z[j], Z[i]) (utils.py:226), so every unordered image pair {i, j} is multiplied ONCE: by the
 * query image that "owns" it (j within the next floor((N-1)/2) images after i in circular order).  The owner's
 * tile yields both
 *   rowmin_d2[j*Mq + r]              = min_c |q_r - b_(j,c)|^2     for query rows r of image i   (plain stores), and
 *   colmin_d2[(i-q_img0)*nb_img*P + j*P + c] = min_{r in image i} |q_r - b_(j,c)|^2             (atomicMin),
 * i.e. the distance of patch (j,c) to its nearest patch of image i.  Values are SQUARED distances; entries of
 * pairs that are not owned are undefined (rowmin) / huge (colmin).  With a single rank (Mq = nb_img*P) colmin is
 * already laid out as [bank image, query row]; sharded runs exchange column blocks (all-to-all) first.
 * Only bank images in the circular window [bank_begin, bank_begin + bank_count) are visited (bank_count = nb_img:
 * all), so a sharded run can multiply against its local shard while the remote shards are still in flight and
 * finish with a second call; init_colmin = 1 resets colmin first (first call of a sequence).
 * Tensor-core precisions only; needs P >= 32 and Mq % P == 0, else AC_ERR_UNSUPPORTED (use ac_min_dist). */
int ac_min_dist_sym(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                    const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                    int bank_count, int init_colmin, float* rowmin_d2, float* colmin_d2, void* ws, size_t ws_bytes,
                    ac_stream_t stream);

/* w[r] = mean over bank images j != i(r) of sqrt(owned(i,j) ? rowmin_d2[j,r] : colmin_d2[j,r]); both arrays
 * [nb_img, Mq], i(r) = q_img0 + r / Pq.  Replaces utils.py:227 for the symmetric form. */
int ac_reduce_weights_sym(const float* rowmin_d2, const float* colmin_d2, int64_t Mq, int nb_img, int Pq, int q_img0,
                          float* w, ac_stream_t stream);

/* ---- stage 2, precision mode "f16r": tensor-core search + exact re-evaluation -----------------------
 * The tensor-core distance carries the fp32 accumulation error of K = D products of magnitude |q||b| (about 3e-3
 * absolute at D = 4096, |x| ~ 31), too much for softmax(w / tau) once tau < 1 (utils.py:253), while the ARG-min
 * is far more robust than the value.  The *_arg variants additionally record which bank row won:
 *   argmin[j*Mq + r]  (ac_min_dist_arg)      row inside bank image j nearest to query row r
 *   rowarg[j*Mq + r]  (ac_min_dist_sym_arg)  same, for the pairs the query image owns
 *   colkey[(i-q_img0)*nb_img*P + j*P + c]    (fp32 bits of min d2 << 32) | row inside query image i that is nearest
 *                                            to bank patch (j,c)  -- the 64-bit counterpart of colmin_d2
 * (sharded runs exchange colkey column blocks exactly like colmin_d2), and ac_refine_min_dist recomputes
 *   dmin[j*Mq + r] = || q_r - b_(j, arg) ||_2 = sqrt(sum_k (q_r[k] - b[k])^2)
 * in fp32 without the |x|^2+|y|^2-2xy cancellation: the query row from Zq (fp32, if not NULL) else from its
 * operand copy Qhi (+ Qlo), the bank row from the operand copy Bhi (+ Blo).  sym = 1: query image i = q_img0 + r/P,
 * arg from rowarg where i owns the pair {i,j} else from the low half of colkey[j*Mq + r] (layout [bank image, query row],
 * i.e. after the column-block exchange); the own image gets 0.  sym = 0: arg from rowarg everywhere; q_self
 * ([ceil(Mq/Pq)] bank index of each query image, or NULL) names pairs to skip.  Bn2 (the bank operands' squared norms,
 * as for ac_min_dist; may be NULL) lets a pair cost one FFMA per element.  Feed dmin to ac_reduce_weights.
 * Costs one gathered 2*D-byte row per (query row, bank image): ~1/3 of the one-pass GEMM time at config 2.
 * Needs D % 8 == 0 and D <= 12800, else AC_ERR_UNSUPPORTED (use the X3 modes).  Zq, Qhi, Qlo, Bhi and Blo (those given)
 * must be 16-byte aligned (it reads them as 16-byte vectors), else AC_ERR_INVALID. */
int ac_min_dist_arg(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, const void* Bhi, const void* Blo,
                    const float* Bn2, int nb_img, int P, int D, int precision, float* dmin, int32_t* argmin, void* ws,
                    size_t ws_bytes, ac_stream_t stream);

/* ac_min_dist / ac_min_dist_arg (argmin may be NULL) for a bank that is still ARRIVING (sharded supervised runs; see
 * ac_min_dist_sym_ready): bank_ready [nb_img] int32 arrival flags in device memory (NULL = resident), first_bank_image = where the
 * walk over the bank images starts (the first resident one; the others are visited in increasing order, wrapping around). */
int ac_min_dist_ready(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, const void* Bhi, const void* Blo,
                      const float* Bn2, int nb_img, int P, int D, int precision, float* dmin, int32_t* argmin,
                      const int32_t* bank_ready, int first_bank_image, void* ws, size_t ws_bytes, ac_stream_t stream);
int ac_min_dist_sym_arg(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                        const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                        int bank_count, int init_colkey, float* rowmin_d2, int32_t* rowarg, uint64_t* colkey, void* ws,
                        size_t ws_bytes, ac_stream_t stream);
int ac_refine_min_dist(const float* Zq, const void* Qhi, const void* Qlo, int64_t Mq, const void* Bhi, const void* Blo,
                       int op_dtype, int nb_img, int P, int D, const int32_t* rowarg, const uint64_t* colkey, int sym,
                       int q_img0, const int32_t* q_self, int Pq, const int32_t* groups, const float* Bn2, float* dmin,
                       ac_stream_t stream);

/* ---- per-category banks in one launch sequence -------------------------------------------------------
 * The reference runs one make_category_data per category, each with its own bank (examples/main.py:353).  The _ex
 * forms take the images of SEVERAL categories back to back: groups[2*j], groups[2*j+1] (device int32 [nb_img, 2]) =
 * first image and image count of the category of image j; image pairs exist only inside a category, the ownership
 * rule of the symmetric form is applied inside it, and the reductions run over the image's own category.
 * groups = NULL is one category (= the plain entry points).  ac_min_dist_sym_ex is the general symmetric entry point:
 * float column minima (colmin_d2) when rowarg == colkey == NULL, else the arg-recording form (colmin_d2 unused).
 * ac_refine_min_dist takes the same `groups` (sym = 1 only).  ac_reduce_weights_ex needs q_self when groups is given. */
int ac_min_dist_sym_ex(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                       const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                       int bank_count, int init, float* rowmin_d2, float* colmin_d2, int32_t* rowarg, uint64_t* colkey,
                       const int32_t* groups, void* ws, size_t ws_bytes, ac_stream_t stream);

/* The same launch for a bank that is still ARRIVING (sharded runs: remote shards are pulled by the copy engines while the kernel
 * runs): bank_ready [nb_img] int32 in device memory, bank_ready[j] != 0 once the operand rows and norms of bank image j have
 * landed (written by whatever stream performs the transfer, after it); the kernel's loader waits for the flag of a bank image
 * before its first load of it (watchdog code 7 if it never comes).  NULL = ac_min_dist_sym_ex.  One launch then covers the
 * local and all remote bank images instead of one launch per landed window. */
int ac_min_dist_sym_ready(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                          const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                          int bank_count, int init, float* rowmin_d2, float* colmin_d2, int32_t* rowarg, uint64_t* colkey,
                          const int32_t* groups, const int32_t* bank_ready, void* ws, size_t ws_bytes, ac_stream_t stream);
int ac_reduce_weights_sym_ex(const float* rowmin_d2, const float* colmin_d2, int64_t Mq, int nb_img, int Pq, int q_img0,
                             const int32_t* groups, float* w, ac_stream_t stream);

/* ---- growing an unsupervised category ---------------------------------------------------------------
 * w[r] of Weight_Distance_Unsupervised (utils.py:222-227) is a MEAN over the other images of one per-image minimum each, so when
 * M images join N_old images only the M*N_old + M*(M-1)/2 new image pairs need the distance pass.  The bank is the
 * nb_img = N_old + M images stored contiguously (new ones last), the query window is the new images (q_img0 = n_old,
 * Mq = M*P), and ownership is
 *   new image i, old image j:  i owns {i, j};
 *   two new images:            pair_owned among the new images (the rule of ac_min_dist_sym with N = M);
 *   two old images:            never visited.
 * n_old = 0 is exactly ac_min_dist_sym_ex (the same units, the same bits).  Outputs and every other argument as
 * ac_min_dist_sym_ex: rowmin_d2 [nb_img, Mq], colmin_d2 (or colkey) [M, nb_img*P], rowarg / colkey for the refined precisions.
 * groups must be NULL (AC_ERR_UNSUPPORTED); q_img0 != n_old or Mq != (nb_img - n_old)*P: AC_ERR_INVALID. */
int ac_min_dist_sym_grow(const void* Qhi, const void* Qlo, const float* Qn2, int64_t Mq, int q_img0, const void* Bhi,
                         const void* Blo, const float* Bn2, int nb_img, int P, int D, int precision, int bank_begin,
                         int bank_count, int init, float* rowmin_d2, float* colmin_d2, int32_t* rowarg, uint64_t* colkey,
                         const int32_t* groups, int n_old, void* ws, size_t ws_bytes, ac_stream_t stream);
/* Exact fp32 re-evaluation (as ac_refine_min_dist) of the NEW pairs of one growth launch only: the new rows against every other
 * image, arg from rowarg where the new image owns the pair, else from colkey; the old rows against the new images, arg from
 * colkey.  Z [nb_img*P, D] fp32 is the whole category (each row's own Z); Bhi / Blo / Bn2 its operands as for the launch.
 * drow [nb_img, M*P] receives the distances of the pairs the new row's image owns, dcol [M, nb_img*P] those of the pairs a
 * new image j owns (row R of the category at dcol[(j - n_old)*nb_img*P + R]); entries of other pairs are left untouched. */
int ac_refine_min_dist_grow(const float* Z, const void* Bhi, const void* Blo, int op_dtype, int n_old, int nb_img, int P, int D,
                            const int32_t* rowarg, const uint64_t* colkey, const float* Bn2, float* drow, float* dcol,
                            ac_stream_t stream);
/* Running sums of the category: S [nb_img*P] fp64, S[R] += d(R, j) over the new pairs of row R (old rows: the M new images;
 * new rows: every other image), partner images in increasing order; then w[R] = float(S[R] / (nb_img - 1)) for every row.
 * Rows of new images start from 0, rows of old ones from S as left by the previous update.  rowv / colv in the layouts of
 * drow / dcol above: squared = 1 for the squared minima of ac_min_dist_sym_grow, 0 for the distances of
 * ac_refine_min_dist_grow.  The order of addition is fixed by the data, so the result does not depend on the launch geometry.
 * Only the entries of the rule's table are read for each pair (the other one may hold anything, NaN included).  A category of
 * one image (nb_img = 1, n_old = 0) has no partner: S = 0 and w = NaN. */
int ac_accumulate_weights_grow(const float* rowv, const float* colv, int squared, int n_old, int nb_img, int P, double* S,
                               float* w, ac_stream_t stream);
int ac_reduce_weights_ex(const float* dmin, int64_t Mq, int nb_img, int Pq, const int32_t* q_self, const int32_t* groups,
                         int mode, float* w, ac_stream_t stream);

/* ---- stage 3 -----------------------------------------------------------------------------------
 * alpha[t, i, :] = softmax_p(w[i, :] / tau_t) in float64, max-subtracted (identical to
 * Matrix_Alpha_* wherever the reference's exp does not overflow, utils.py:246-255); tau == 0 gives
 * one-hot (the reference's math.isclose(tau, 0)): one-hot-on-max with ties split equally (:248-250).
 * alpha64 [T,N,P] double and/or alpha32 [T,N,P] float (either may be NULL). taus_host: HOST array. */
int ac_alpha(const float* w, int N, int P, const double* taus_host, int T, double* alpha64,
             float* alpha32, ac_stream_t stream);

/* X[i, :] = sum_p alpha[i,p] * Z[i,p,:]   (torch.bmm line, examples/main.py:294-296).  Any alignment of Z and X: the
 * vector loads need D % 4 == 0 and 16-byte aligned Z and X, other calls take a scalar loop with the same result bits. */
int ac_weighted_embed(const float* alpha, const float* Z, int N, int P, int D, float* X,
                      ac_stream_t stream);

/* The same for T temperatures in ONE pass over Z (a tau sweep calls the bmm line once per tau, examples/main.py:294-296 inside the
 * loop of :353): alpha [T, N, P], X [T, N, D]; bit-identical to T calls of ac_weighted_embed. */
int ac_weighted_embed_multi(const float* alpha, const float* Z, int T, int N, int P, int D, float* X, ac_stream_t stream);

/* X without Z (SURVEY.md section 8f row 4): Z is a fixed linear map of the LayerNorm'd feature maps, so
 * X[i] = sum_p alpha[i,p] Z[i,p] = Pool(A_i) with A_i[c,ki,kj] = sum_p alpha[i,p] * LN_i[c, y_p+ki-1, x_p+kj-1]:
 * a 3x3 correlation of the alpha map with every channel, then the MeanMapper / Aggregator windows once per
 * image.  Same result as ac_embed + ac_weighted_embed (examples/main.py:266-296) while fp32 Z is never stored.
 * alpha [B, P] fp32, X [B, D] fp32.  Needs patchsize 3, stride 1, every layer on the layer-0 grid and Aggregator
 * windows that do not straddle layers, and a (h0 + 2) x (w0 + 2) fp32 alpha tile of at most 200 KB (h0 = w0 <= 224),
 * else AC_ERR_UNSUPPORTED (use ac_embed + ac_weighted_embed).  ws must be 16-byte aligned, else AC_ERR_INVALID. */
size_t ac_weighted_embed_from_features_workspace_bytes(const ac_layer_t* layers_host, int L, int B, int patchsize);
int ac_weighted_embed_from_features(const ac_layer_t* layers_host, int L, int B, int patchsize, int stride, int Dp,
                                    int D, int layernorm, float eps, const float* alpha, float* X, void* ws,
                                    size_t ws_bytes, ac_stream_t stream);
/* The same for feature maps of element type feat_dtype (see ac_embed_dt): X is bit-identical to the fp32 call on the
 * upcast maps with the same strides and element offsets. */
size_t ac_weighted_embed_from_features_workspace_bytes_dt(const ac_layer_t* layers_host, int L, int feat_dtype, int B,
                                                          int patchsize);
int ac_weighted_embed_from_features_dt(const ac_layer_t* layers_host, int L, int feat_dtype, int B, int patchsize,
                                       int stride, int Dp, int D, int layernorm, float eps, const float* alpha, float* X,
                                       void* ws, size_t ws_bytes, ac_stream_t stream);

/* Multi-GPU plumbing (no counterpart in the reference, which is single-device: examples/main.py:38): up to 16 strided 2-D blocks
 * (rows x row_bytes, row_bytes a multiple of 4, own row strides in bytes) copied in ONE launch.  Sources / destinations may be
 * peer mappings (symmetric memory over NVLink); the sharded path collects the column minima of its query rows with it.
 * All array arguments are HOST arrays of length n. */
int ac_copy_blocks(int n, const void* const* src_host, const int64_t* src_stride_bytes_host, void* const* dst_host,
                   const int64_t* dst_stride_bytes_host, const int32_t* rows_host, const int64_t* row_bytes_host,
                   ac_stream_t stream);

/* Dmat[i,j] = || X[i] - X[j] ||_2, the Euclidean matrix Ward linkage consumes
 * (examples/test.py:193-195 -> scipy pdist).  Dmat [N,N] fp32, exactly symmetric, zero diagonal.  Any alignment of X
 * (vector loads only when X is 16-byte aligned; the result bits do not depend on it). */
int ac_pairwise_l2(const float* X, int N, int D, float* Dmat, ac_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AC_B200_H */
