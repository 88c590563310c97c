/* libdss_b200 -- C ABI of the B200-native deep-spectral hot path.
 *
 * The reference (lukemelas/deep-spectral-segmentation) has no FFI/plugin interface: the hot path is two Python
 * callables, extract_features (extract/extract.py:21-116) and _extract_eig (extract/extract.py:119-244), that call
 * torch / scipy / pymatting directly. This header declares the entry points a ctypes binding in those two
 * functions uses instead of the library calls; each one cites the reference lines it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes. Every data pointer is a DEVICE pointer owned by the caller unless
 *     the name ends in _host. The library never synchronises the device and never frees caller memory; all work
 *     is enqueued on the caller's stream (a cudaStream_t passed as void*).
 *   - Scratch memory comes from the caller: query dss_*_workspace_bytes, pass (ws, ws_bytes). Workspaces must be
 *     256-byte aligned. A dss_vit_t handle owns only its packed weights and cached positional embeddings.
 *   - Return value: DSS_OK (0) or a negative dss_status; dss_last_error() gives a thread-local message.
 *     Asynchronous numerical outcomes (eigensolver convergence) are reported through device-side info arrays.
 *   - Row-major, C-contiguous tensors; shapes are written [outer, ..., inner].
 */
#ifndef DSS_B200_H
#define DSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dss_stream_t; /* cudaStream_t */

typedef enum {
  DSS_OK = 0,
  DSS_ERR_BAD_ARG = -1,
  DSS_ERR_CUDA = -2,
  DSS_ERR_WORKSPACE = -3,
  DSS_ERR_UNSUPPORTED = -4
} dss_status;

const char* dss_last_error(void);
int dss_version(void);            /* 100 * major + minor */
int dss_device_sm_count(void);    /* SM count of the current device (148 on B200), <0 on error */

/* Launch accounting: number of kernels this library has launched in this process. */
long long dss_kernel_launch_count(void);
/* Per-kernel-class device timing for roofline reports: while enabled, every kernel launch is bracketed by CUDA
 * events on its stream. dss_profile_enable(1) starts a fresh recording, dss_profile_read synchronises the recorded
 * events and returns the number of classes written to `out` (<0 on error). Not for use inside timed regions. */
typedef struct { const char* name; long long launches; double total_ms; } dss_profile_entry;
void dss_profile_enable(int on);
int dss_profile_read(dss_profile_entry* out, int max_entries);

/* ------------------------------------------------------------------------------------------------------------
 * DINO ViT feature extractor  (replaces utils.get_model + model.get_intermediate_layers + the qkv hook,
 * extract/extract_utils.py:40-50, extract/extract.py:49-53,82-98)
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct dss_vit dss_vit_t;

typedef struct {
  int patch;     /* 16 or 8 */
  int dim;       /* 384 (ViT-S) or 768 (ViT-B); head dim must be 64 */
  int depth;     /* 12 */
  int heads;     /* 6 / 12 */
  int mlp_ratio; /* 4 */
  int grid0;     /* side of the training positional grid: 224 / patch */
  float ln_eps;  /* 1e-6 */
} dss_vit_config;

/* fp32 device pointers in the upstream state_dict layout (torch Linear weight = [out, in]) */
typedef struct {
  const float *ln1_w, *ln1_b;   /* [d] */
  const float *qkv_w, *qkv_b;   /* [3d, d], [3d] */
  const float *proj_w, *proj_b; /* [d, d], [d] */
  const float *ln2_w, *ln2_b;   /* [d] */
  const float *fc1_w, *fc1_b;   /* [4d, d], [4d] */
  const float *fc2_w, *fc2_b;   /* [d, 4d], [d] */
} dss_vit_block_weights;

typedef struct {
  const float* patch_w;   /* [d, 3, P, P] conv weight */
  const float* patch_b;   /* [d] */
  const float* cls_token; /* [d] */
  const float* pos_embed; /* [1 + grid0*grid0, d] */
  const dss_vit_block_weights* blocks; /* host array of `depth` entries */
  const float *norm_w, *norm_b; /* [d] final LayerNorm; may be NULL (only dss_vit_forward_cls needs them) */
} dss_vit_weights;

int dss_vit_create(const dss_vit_config* cfg, dss_vit_t** out);
void dss_vit_destroy(dss_vit_t* h);
/* Packs the weights into the library's fp16 operand layout (synchronises `stream` before returning). */
int dss_vit_load_weights(dss_vit_t* h, const dss_vit_weights* w, dss_stream_t stream);

size_t dss_vit_workspace_bytes(const dss_vit_t* h, int B, int H, int W);

/* images_u8 [B, H, W, 3] RGB bytes (what cv2.imread+BGR2RGB yields, extract_utils.py:30-31). The library applies
 * ToTensor + Normalize(ImageNet) (extract_utils.py:53-59) and the top-left crop to patch multiples
 * (extract.py:82-88) on the fly, runs blocks [0, which_block) fully and block `which_block` up to its K projection
 * and writes k_out [B, N, d] fp32 == output_dict['k'] (extract.py:98), N = (H/P)*(W/P).
 * which_block may be negative (python indexing, default -1). */
int dss_vit_forward_k(dss_vit_t* h, const uint8_t* images_u8, int B, int H, int W, int which_block, float* k_out,
                      void* ws, size_t ws_bytes, dss_stream_t stream);

/* Debug/parity hook: residual stream x [B, T, d] fp32 after `n_blocks` full blocks (T = N + 1, CLS first). */
int dss_vit_forward_tokens(dss_vit_t* h, const uint8_t* images_u8, int B, int H, int W, int n_blocks, float* x_out,
                           void* ws, size_t ws_bytes, dss_stream_t stream);

/* The model's own forward (upstream VisionTransformer.forward: all blocks, final LayerNorm, CLS token), which the
 * reference calls on bounding-box crops (extract/extract.py:537-541, extract_bbox_features): cls_out [B, d] fp32. */
int dss_vit_forward_cls(dss_vit_t* h, const uint8_t* images_u8, int B, int H, int W, float* cls_out, void* ws,
                        size_t ws_bytes, dss_stream_t stream);

/* Interpolated positional embedding [T, d] fp32 for an (Hp x Wp) patch grid, as upstream
 * VisionTransformer.interpolate_pos_encoding computes it (bicubic, scale (Hp+0.1)/grid0). Copied to out (device). */
int dss_vit_pos_embed(dss_vit_t* h, int Hp, int Wp, float* out, dss_stream_t stream);
/* The same interpolation on HOST buffers (pure CPU, no CUDA call): pos_embed_host [1+grid0^2, d] -> out_host
 * [1+Hp*Wp, d]. This is the routine the handle runs once per distinct image shape. */
int dss_pos_embed_interp_host(const float* pos_embed_host, int grid0, int d, int Hp, int Wp, float* out_host);

/* ------------------------------------------------------------------------------------------------------------
 * Low-level operators (unit-test surface of the ViT kernels). fp16 operands are IEEE binary16.
 * ------------------------------------------------------------------------------------------------------------ */
typedef enum {
  DSS_EPI_BIAS_F16 = 0,      /* out f16 [M, N] = acc + bias                                   */
  DSS_EPI_BIAS_GELU_F16 = 1, /* out f16 [M, N] = gelu_erf(acc + bias)                         */
  DSS_EPI_BIAS_RESID_F32 = 2,/* out f32 [M, N] += acc + bias   (in-place residual)            */
  DSS_EPI_BIAS_F32 = 3,      /* out f32 [M, N] = acc + bias                                   */
  DSS_EPI_PATCH_F32 = 4,     /* out f32 row (m/rin)*rout + m%rin + 1 = acc + bias + aux[m%rin + 1, :]  (patch embed) */
  DSS_EPI_DROPCLS_F32 = 5    /* out f32 row (m/rin)*rout + m%rin - 1 = acc + bias, rows with m%rin == 0 skipped */
} dss_epilogue;

/* out = epilogue(A[M,K] (f16) * Wt[N,K]^T (f16) + bias[N]) on tcgen05 tensor cores (TMA-fed, TMEM accumulator).
 * K % 8 == 0, N % 32 == 0, lda == K, ldw == K. aux/rin/rout only for the row-remapping epilogues. */
int dss_op_gemm_f16(const void* A, const void* Wt, const float* bias, void* out, int M, int N, int K, int epilogue,
                    const float* aux, int rin, int rout, dss_stream_t stream);
/* Same contract on CUDA cores (slow, fp32 FMA): in-GPU checker for the tensor-core kernel, used by tests only. */
int dss_op_gemm_f16_simt(const void* A, const void* Wt, const float* bias, void* out, int M, int N, int K,
                         int epilogue, const float* aux, int rin, int rout, dss_stream_t stream);
/* LayerNorm fused into the GEMM's A-operand producer (the qkv / fc1 layers of ViT-S; K must be 384):
 * out f16 [M, N] = (gelu ? gelu_erf : id)(LayerNorm(x f32 [M, K]; gamma, beta, eps) @ Wt f16 [N, K]^T + bias); N % 128 == 0 */
int dss_op_gemm_ln_f16(const float* x, const float* gamma, const float* beta, const void* Wt, const float* bias,
                       void* out, int M, int N, int K, float eps, int gelu, dss_stream_t stream);
/* y f16 [M, d] = LayerNorm(x f32 [M, d]) * gamma + beta, d in {384, 768} */
int dss_op_layernorm_f16(const float* x, const float* gamma, const float* beta, void* y, int M, int d, float eps,
                         dss_stream_t stream);
/* qkv f16 [B, T, 3*d] (q | k | v, heads of 64 inside each) -> out f16 [B, T, d] = softmax(q k^T / 8) v */
int dss_op_attention_f16(const void* qkv, void* out, int B, int T, int heads, dss_stream_t stream);
/* same contract on tcgen05 (TMA-fed QK^T and PV UMMAs, S and O in TMEM); the ViT forward uses this one */
int dss_op_attention_tc_f16(const void* qkv, void* out, int B, int T, int heads, dss_stream_t stream);
/* images_u8 [B,H,W,3] -> patches f16 [B*N, 3*P*P], column order (c, py, px), normalised */
int dss_op_im2col_f16(const uint8_t* images_u8, void* patches, int B, int H, int W, int P, dss_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Affinity + graph Laplacian eigensolver (replaces extract/extract.py:148,191-195,207-235,237-240)
 * ------------------------------------------------------------------------------------------------------------ */
enum { DSS_AFF_NORMALIZE = 1, DSS_AFF_THRESHOLD_AT_ZERO = 2, DSS_AFF_NO_MAX_SCALE = 4 };

size_t dss_affinity_workspace_bytes(int B, int N, int d);
/* feats [B, N, d] fp32 -> Wmat [B, N, ldw] fp32 (row pitch ldw >= N, ldw % 4 == 0, pad columns written as 0):
 *   F^ = F / max(||F||, 1e-12) rowwise (if NORMALIZE)                      extract.py:148
 *   W  = F^ F^T ; W *= (W > 0) (if THRESHOLD) ; W /= max(W)                extract.py:191-194
 *        (NO_MAX_SCALE skips the division: the 'affinity' / 'affinity_svd' branches, extract.py:160-172)
 *   W += color_counts * color_lambda  (if color_counts != NULL)            extract.py:213,221
 *   degree[b, i] = sum_j W[b, i, j]   (if degree != NULL)                  extract_utils.py:217 (row_sum)
 * color_counts [B, N, N] uint8 is the dense KNN colour affinity of dss_knn_color_counts.
 * W is symmetric: only the tiles on or above the diagonal are computed on the tensor cores and each is stored twice
 * (W[i,j] and W[j,i] are the same bits). The row sums are accumulated in the same epilogue (fixed summation order,
 * bit-reproducible) so that the eigensolver does not need another pass over W; pass the result to
 * dss_eigsh_laplacian. A colour term added AFTER this call (dss_rw_affinity_add) updates `degree` itself. */
int dss_affinity(const float* feats, int B, int N, int d, int flags, const uint8_t* color_counts, float color_lambda,
                 float* Wmat, int ldw, float* degree, void* ws, size_t ws_bytes, dss_stream_t stream);

/* Colour KNN affinity (extract_utils.py:151-188): rgb [B, Hl*Wl, 3] fp32 in [0,1] (the /255 low-res image of
 * extract.py:199-204). Two exact-KNN passes (k=20, w=2.0) and (k=10, w=0.1) over points (r,g,b,w*x,w*y),
 * x,y = linspace(0,1); counts[i,j] += 1 and counts[j,i] += 1 per directed neighbour pair (self included), i.e.
 * the dense form of the reference's duplicate-summing csr_matrix. counts [B, N, N] uint8 is overwritten; the buffer
 * must be 4-byte aligned and its capacity rounded up to a multiple of 4 bytes (bytes are updated with 32-bit atomics;
 * any N, odd included). */
size_t dss_knn_workspace_bytes(int B, int N);
int dss_knn_color_counts(const float* rgb, int B, int Hl, int Wl, uint8_t* counts, void* ws, size_t ws_bytes,
                         dss_stream_t stream);

/* Eigensolver. Wmat [B, N, ldw] symmetric, non-negative (row pitch ldw as written by dss_affinity). Only the upper
 * triangle (j >= i) of every matrix is read. degree [B, N] = row sums of W as written by dss_affinity, or NULL (the
 * solver then computes them with one more pass over W).
 *   lapnorm != 0: K smallest pairs of (D - W) v = lambda D v, D = diag(rowsum W) (entries < 1e-12 -> 1,
 *                 extract_utils.py:217-218); eigenvectors D-orthonormal            extract.py:225-229
 *   lapnorm == 0: K smallest pairs of (D - W) v = lambda v, unit 2-norm vectors    extract.py:230-234
 * Outputs: evals [B, K] ascending, evecs [B, K, N] with the reference's sign rule applied (extract.py:237-240),
 * info [B, 4] int32 = {lanczos steps, converged(1/0), 0, 0}, resid [B, K] fp32 residual estimates (may be NULL).
 * Method: Lanczos with full re-orthogonalisation on D^-1/2 W D^-1/2 (null vector deflated analytically), Ritz
 * values by Sturm bisection in fp64. tol <= 0 selects 1e-6; max_steps <= 0 selects min(N-1, 320). */
size_t dss_eigsh_workspace_bytes(int B, int N, int K, int max_steps);
int dss_eigsh_laplacian(const float* Wmat, const float* degree, int ldw, int B, int N, int K, int lapnorm, float tol,
                        int max_steps, float* evals, float* evecs, int* info, float* resid, void* ws, size_t ws_bytes,
                        dss_stream_t stream);

/* K algebraically largest eigenpairs of the symmetric matrices Amat [B, N, lda], descending, unit 2-norm vectors,
 * reference sign rule applied. Serves which_matrix='affinity' (eigsh(W, which='LM', k=K), extract.py:166-172; for a
 * non-negative affinity the largest-magnitude eigenvalues are the largest positive ones -- info[b,2] is set to 1 if a
 * negative eigenvalue of larger magnitude exists) and 'affinity_svd' (left singular vectors of F^ = eigenvectors of
 * F^ F^T, extract.py:160-163). Same workspace / info / resid conventions as dss_eigsh_laplacian. */
int dss_eigsh_topk(const float* Amat, int lda, int B, int N, int K, float tol, int max_steps, float* evals,
                   float* evecs, int* info, float* resid, void* ws, size_t ws_bytes, dss_stream_t stream);

/* Random-walk colour affinity (which_color_matrix='rw', extract_utils.py:191-204 -> pymatting _rw_laplacian with
 * radius 1): Wmat[b, i, j] += float32(sum over the 3x3 clamped neighbourhood offsets that land on j of
 * exp(-coef * ||z_i - z_j||^2)) * color_lambda, z = rgb_u8 / 255 in float64; the same amount is added to degree[b, i]
 * (may be NULL). rgb_u8 [B, Hl*Wl, 3] is the low-resolution image of extract.py:199-204 BEFORE the /255.
 * pymatting hard-codes coef = 900 (its sigma argument is unused); pass 1/sigma^2 for the textbook kernel. */
int dss_rw_affinity_add(const uint8_t* rgb_u8, int B, int Hl, int Wl, float color_lambda, double coef, float* Wmat,
                        int ldw, float* degree, dss_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Segmentations from the eigenvectors (replace extract/extract.py:283-349 and :364-390), fused after the eigensolve
 * ------------------------------------------------------------------------------------------------------------ */
/* mask[b, n] = 255 if evecs[b, which, n] > threshold else 0   (the 'L' image the reference saves; which = 1) */
int dss_segment_threshold(const float* evecs, int B, int K, int N, int which, float threshold, uint8_t* mask,
                          dss_stream_t stream);
/* Batched K-means (k-means++ seeding, Lloyd, scikit-learn's stopping rules: tol * mean feature variance on the centre
 * shift, strict label convergence, max_iter; empty clusters are re-seeded with the farthest point). One CTA per image.
 * Point n of image b has coordinates points[b * image_stride + n * point_stride + j * dim_stride], j < dims -- the
 * eigenvector embedding evecs[b, 1 + j, n] is (K*N, 1, N) from &evecs[b=0, 1, 0]; raw features [B, N, d] are (N*d, d, 1).
 * n_clusters [B] int32 (device) gives k per image (the reference's adaptive mode), capped by max_clusters <= 64.
 * If infer_bg_index, labels are taken on a grid_h x grid_w grid (grid_h * grid_w == N) and the label with the largest
 * border share is swapped with 0 (extract_utils.py:124-135). labels [B, N] uint8; info [B, 2] = {iterations,
 * converged}; inertia [B] (may be NULL). seed: counter-based generator keyed by (seed, image_keys[b]) -- image_keys [B]
 * int32 (device; e.g. the `indices` field of the feature files) makes an image's clustering independent of the batch it
 * is processed in; NULL uses the position in the batch. (The reference's clustering is unseeded.) */
int dss_segment_kmeans(const float* points, long long image_stride, long long point_stride, long long dim_stride, int B,
                       int N, int dims, const int* n_clusters, const int* image_keys, int max_clusters, int grid_h,
                       int grid_w, int infer_bg_index, unsigned int seed, int max_iter, float tol, uint8_t* labels,
                       int* info, float* inertia, dss_stream_t stream);

/* Bilinear up-sampling of patch features (align_corners=False, as F.interpolate at extract.py:185-188):
 * feats [B, Hp*Wp, d] fp32 -> out [B, Hl*Wl, d] fp32. Used when image_downsample_factor != patch size. */
int dss_upsample_bilinear(const float* feats, int B, int Hp, int Wp, int d, int Hl, int Wl, float* out,
                          dss_stream_t stream);
/* Row-wise L2 normalisation x / max(||x||, 1e-12) (F.normalize, extract.py:148): feats [rows, d] -> out [rows, d]. */
int dss_normalize_rows(const float* feats, int rows, int d, float* out, dss_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DSS_B200_H */
