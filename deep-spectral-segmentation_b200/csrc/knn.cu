// Colour KNN affinity (reference extract/extract_utils.py:151-188, which calls pymatting.util.kdtree.knn).
//
// For every low-resolution pixel i the reference finds its k nearest pixels (itself included) in the 5-D space
// (r, g, b, w*x, w*y), twice: (k=20, w=2.0) and (k=10, w=0.1), and builds csr_matrix((1, (ij, ji))) with
// ij = [i.., j..], ji = [j.., i..]; duplicates are summed, so each directed neighbour pair (i -> j) adds 1 to
// W[i,j] and 1 to W[j,i]. This kernel does an exact brute-force KNN (N <= 6400 points: a KD-tree buys nothing on a
// GPU) and accumulates the same dense matrix as uint8 counts (max value 4).
//
// One warp per query point; the image's points sit in shared memory (SoA). Neighbours are extracted in
// increasing (squared distance, index) order by k successive warp-wide arg-min sweeps; squared distances are
// accumulated in fp32 dimension by dimension without FMA contraction so that ties/orderings are reproducible
// bit-for-bit by the CPU oracle (oracle/eigs_ref.py:knn_exact).
#include "common.cuh"

namespace dss {

constexpr int KNN_WARPS = 8;

__device__ __forceinline__ float sqdist5(const float* __restrict__ pts, int N, int j, const float (&q)[5]) {
  float d2 = 0.f;
#pragma unroll
  for (int c = 0; c < 5; ++c) {
    const float diff = __fsub_rn(q[c], pts[c * N + j]);
    d2 = __fadd_rn(d2, __fmul_rn(diff, diff));
  }
  return d2;
}

__global__ void __launch_bounds__(KNN_WARPS * 32)
knn_counts_kernel(const float* __restrict__ rgb, uint32_t* __restrict__ counts_words, int N, int Hl, int Wl, int k,
                  double weight) {
  extern __shared__ float pts[];  // [5][N]
  const int b = blockIdx.y;
  const float* src = rgb + (size_t)b * N * 3;
  const double sx = Wl > 1 ? 1.0 / (double)(Wl - 1) : 0.0;  // np.linspace(0, 1, w) step
  const double sy = Hl > 1 ? 1.0 / (double)(Hl - 1) : 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const int col = i % Wl, row = i / Wl;
    pts[0 * N + i] = src[i * 3 + 0];
    pts[1 * N + i] = src[i * 3 + 1];
    pts[2 * N + i] = src[i * 3 + 2];
    const double x = (col == Wl - 1 && Wl > 1) ? 1.0 : (double)col * sx;
    const double y = (row == Hl - 1 && Hl > 1) ? 1.0 : (double)row * sy;
    pts[3 * N + i] = (float)(weight * x);
    pts[4 * N + i] = (float)(weight * y);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * KNN_WARPS + warp;
  if (qi >= N) return;
  float q[5];
#pragma unroll
  for (int c = 0; c < 5; ++c) q[c] = pts[c * N + qi];
  // bytes are addressed over the WHOLE [B, N, N] buffer (only its base is 4-byte aligned), so odd N -- e.g. the 23 x 31
  // grid of a 375 x 500 VOC image -- needs no row padding: byte e lives in word e >> 2 at bit offset 8 * (e & 3)
  const size_t img_off = (size_t)b * N * N;
  uint32_t* cw = counts_words;
  // last selected key (d2, idx); start below everything
  float last_d = -1.f;
  int last_j = -1;
  for (int r = 0; r < k; ++r) {
    float best_d = INFINITY;
    int best_j = 0x7fffffff;
    for (int j = lane; j < N; j += 32) {
      const float d2 = sqdist5(pts, N, j, q);
      const bool after = (d2 > last_d) || (d2 == last_d && j > last_j);
      const bool better = (d2 < best_d) || (d2 == best_d && j < best_j);
      if (after && better) { best_d = d2; best_j = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, best_d, o);
      const int oj = __shfl_xor_sync(0xffffffffu, best_j, o);
      if (od < best_d || (od == best_d && oj < best_j)) { best_d = od; best_j = oj; }
    }
    last_d = best_d;
    last_j = best_j;
    if (lane == 0 && best_j < N) {
      const size_t e0 = img_off + (size_t)qi * N + best_j, e1 = img_off + (size_t)best_j * N + qi;
      atomicAdd(cw + (e0 >> 2), 1u << (8 * (e0 & 3)));
      atomicAdd(cw + (e1 >> 2), 1u << (8 * (e1 & 3)));
    }
  }
}

}  // namespace dss

using namespace dss;

extern "C" size_t dss_knn_workspace_bytes(int B, int N) {
  (void)B; (void)N;
  return 256;  // no scratch needed; kept for ABI symmetry
}

extern "C" int dss_knn_color_counts(const float* rgb, int B, int Hl, int Wl, uint8_t* counts, void* ws,
                                    size_t ws_bytes, dss_stream_t stream) {
  (void)ws; (void)ws_bytes;
  DSS_REQUIRE(rgb && counts, "knn: null pointer");
  DSS_REQUIRE(B > 0 && Hl > 0 && Wl > 0, "knn: empty problem");
  const int N = Hl * Wl;
  DSS_REQUIRE(N >= 20, "knn: need at least 20 points (k=20 neighbours), got %d", N);
  DSS_REQUIRE((reinterpret_cast<uintptr_t>(counts) & 3) == 0, "knn: counts must be 4-byte aligned");
  const size_t smem = (size_t)5 * N * sizeof(float);
  DSS_REQUIRE(smem <= 200 * 1024, "knn: N=%d points do not fit in shared memory", N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DSS_CHECK_CUDA(cudaMemsetAsync(counts, 0, (size_t)B * N * N, st));
  DSS_CHECK_CUDA(allow_dynamic_smem(knn_counts_kernel, (int)smem));
  dim3 grid(cdiv(N, KNN_WARPS), B);
  const int ks[2] = {20, 10};
  const double ws_[2] = {2.0, 0.1};
  for (int pass = 0; pass < 2; ++pass) {
    LaunchScope scope(st, KC_KNN);
    knn_counts_kernel<<<grid, KNN_WARPS * 32, smem, st>>>(rgb, reinterpret_cast<uint32_t*>(counts), N, Hl, Wl, ks[pass],
                                                          ws_[pass]);
    DSS_CHECK_CUDA(cudaGetLastError());
  }
  return DSS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Random-walk colour affinity (reference extract/extract_utils.py:191-204 -> pymatting.laplacian.rw_laplacian.
// _rw_laplacian(image, sigma, radius=1)): for every pixel i and every offset (dy, dx) in [-1, 1]^2 the CLAMPED
// neighbour j gets the weight exp(-coef * ||z_i - z_j||^2) (float64, z = rgb / 255); csr_matrix sums duplicates, which
// border clamping produces (a corner pixel lists itself four times). The reference then densifies to float32, scales by
// image_color_lambda and adds it to the feature affinity (extract.py:216,221). The matrix has <= 9 entries per row,
// so this kernel adds them in place to the dense W the affinity GEMM wrote -- one thread per pixel owns row i (its
// duplicates are merged in float64 first, exactly like the csr constructor) -- and adds the row's total to `degree`.
namespace dss {

__global__ void __launch_bounds__(128)
rw_affinity_add_kernel(const uint8_t* __restrict__ rgb, int Hl, int Wl, float lambda, double coef, float* __restrict__ W,
                       int ldw, float* __restrict__ degree) {
  const int N = Hl * Wl;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (i >= N) return;
  const uint8_t* img = rgb + (size_t)b * N * 3;
  const int y = i / Wl, x = i % Wl;
  const double zi[3] = {img[i * 3] / 255.0, img[i * 3 + 1] / 255.0, img[i * 3 + 2] / 255.0};
  int js[9];
  double ws[9];
  int cnt = 0;
  for (int dy = -1; dy <= 1; ++dy)
    for (int dx = -1; dx <= 1; ++dx) {
      const int x2 = max(0, min(Wl - 1, x + dx)), y2 = max(0, min(Hl - 1, y + dy));
      const int j = x2 + y2 * Wl;
      double d2 = 0.0;
      for (int c = 0; c < 3; ++c) {
        const double diff = zi[c] - img[j * 3 + c] / 255.0;
        d2 += diff * diff;
      }
      const double nrm = sqrt(d2);                 // np.linalg.norm(zi - zj) ** 2
      const double w = exp(-coef * (nrm * nrm));
      int k = 0;
      for (; k < cnt; ++k)
        if (js[k] == j) break;
      if (k < cnt) ws[k] += w;                     // duplicate (i, j): summed, as scipy's csr constructor does
      else { js[cnt] = j; ws[cnt] = w; ++cnt; }
    }
  float* row = W + ((size_t)b * N + i) * ldw;
  float dsum = 0.f;
  for (int k = 0; k < cnt; ++k) {
    const float add = static_cast<float>(ws[k]) * lambda;   // W_color.astype(float32) * image_color_lambda
    row[js[k]] += add;                                       // W_feat + ...
    dsum += add;
  }
  if (degree) degree[(size_t)b * N + i] += dsum;
}

}  // namespace dss

extern "C" int dss_rw_affinity_add(const uint8_t* rgb_u8, int B, int Hl, int Wl, float color_lambda, double coef,
                                   float* Wmat, int ldw, float* degree, dss_stream_t stream) {
  DSS_REQUIRE(rgb_u8 && Wmat, "rw_affinity: null pointer");
  DSS_REQUIRE(B > 0 && Hl > 0 && Wl > 0, "rw_affinity: empty problem");
  DSS_REQUIRE(ldw >= Hl * Wl, "rw_affinity: ldw < N");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LaunchScope scope(st, KC_KNN);
  rw_affinity_add_kernel<<<dim3(cdiv(Hl * Wl, 128), B), 128, 0, st>>>(rgb_u8, Hl, Wl, color_lambda, coef, Wmat, ldw, degree);
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}
