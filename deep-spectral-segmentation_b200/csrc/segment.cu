// First consumers of the eigenvectors (reference extract/extract.py:283-411), fused after the eigensolve so that the
// eigenvectors do not have to leave the GPU:
//   single-region: eigenvector 1 > threshold on the patch grid                       (extract.py:364-390)
//   multi-region : K-means on the non-constant eigenvectors (or on the raw features, kmeans_baseline), the label that
//                  owns most of the border becomes 0                                 (extract.py:283-349,
//                                                                                     extract_utils.py:124-135)
// The reference clusters with scikit-learn's KMeans (k-means++ seeding from numpy's global RNG, Lloyd iterations,
// tol = 1e-4, max_iter = 300, n_init = 1). Its labels depend on that RNG stream, so only the PARTITION is comparable:
// this kernel runs the same algorithm (greedy k-means++ with 2 + log k local trials, Lloyd with the same stopping rule
// and empty-cluster relocation) with a counter-based generator seeded by (seed, image), one CTA per image, points read
// in place from the eigenvector / feature tensors through two strides.
#include <math.h>

#include "common.cuh"

namespace dss {

constexpr int SEG_THREADS = 256;
constexpr int SEG_WARPS = SEG_THREADS / 32;
constexpr int SEG_MAX_CLUSTERS = 64;

__global__ void __launch_bounds__(256)
threshold_mask_kernel(const float* __restrict__ evecs, int K, int N, int which, float threshold,
                      uint8_t* __restrict__ mask, int B) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * N) return;
  const int b = (int)(i / N), n = (int)(i % N);
  // (eigenvector > threshold) as the 8-bit image PIL's convert('L') makes of a boolean array: 0 / 255
  mask[i] = evecs[((long long)b * K + which) * N + n] > threshold ? 255 : 0;
}

__device__ __forceinline__ size_t align_up_dev(size_t x, size_t a) { return (x + a - 1) / a * a; }

__device__ __forceinline__ uint32_t seg_hash(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t x = a * 0x9E3779B1u ^ (b + 0x7F4A7C15u) * 0x85EBCA77u ^ (c + 0x165667B1u) * 0xC2B2AE3Du;
  x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ double seg_uniform(uint32_t seed, uint32_t img, uint32_t ctr) {
  return (double)(seg_hash(seed, img, ctr) >> 8) * (1.0 / 16777216.0);   // [0, 1)
}

struct KmeansParams {
  const float* pts;         // point n of image b, coordinate j: pts[b * img_stride + n * pt_stride + j * dim_stride]
  long long img_stride, pt_stride, dim_stride;
  const int* n_clusters;    // [B]
  const int* image_keys;    // [B] or null: per-image key of the random generator (null: position in the batch)
  uint8_t* labels;          // [B, N]
  int* info;                // [B, 2] = {Lloyd iterations, 1 if converged}
  float* inertia;           // [B] or null
  int B, N, dims, max_k, Hs, Ws, infer_bg, max_iter;
  float tol;
  uint32_t seed;
};

// block-wide sum / arg-max helpers over SEG_THREADS threads
__device__ __forceinline__ double seg_block_sum(double v, double* red, int tid) {
  v = warp_sum(v);
  __syncthreads();
  if ((tid & 31) == 0) red[tid >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < SEG_WARPS; ++i) s += red[i];
  return s;
}

// squared distance of point n to centre c (centres in shared memory, row-major [k][dims])
__device__ __forceinline__ float seg_dist2(const float* __restrict__ p, long long dstride, const float* __restrict__ cen,
                                           int dims) {
  float s0 = 0.f, s1 = 0.f;
  int j = 0;
  for (; j + 1 < dims; j += 2) {
    const float a = p[(long long)j * dstride] - cen[j], b = p[(long long)(j + 1) * dstride] - cen[j + 1];
    s0 = fmaf(a, a, s0); s1 = fmaf(b, b, s1);
  }
  if (j < dims) { const float a = p[(long long)j * dstride] - cen[j]; s0 = fmaf(a, a, s0); }
  return s0 + s1;
}

__global__ void __launch_bounds__(SEG_THREADS)
kmeans_segment_kernel(KmeansParams p) {
  extern __shared__ __align__(16) uint8_t seg_smem[];
  const int N = p.N, dims = p.dims, tid = threadIdx.x;
  // shared layout: centres [max_k][dims] f32 | sums [max_k][dims] f64 | counts [max_k] i32 | mind2 [N] f32 |
  //                lab [N] u8 | scratch
  float* cen = reinterpret_cast<float*>(seg_smem);
  double* sums = reinterpret_cast<double*>(seg_smem + align_up_dev((size_t)p.max_k * dims * 4, 16));
  int* counts = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(sums) + (size_t)p.max_k * dims * 8);
  float* mind2 = reinterpret_cast<float*>(counts + SEG_MAX_CLUSTERS);
  uint8_t* lab = reinterpret_cast<uint8_t*>(mind2 + N);
  __shared__ double red[SEG_WARPS];
  __shared__ double s_val[SEG_WARPS];
  __shared__ int s_idx[SEG_WARPS];
  __shared__ int s_pick, s_changed;
  __shared__ double s_best;

  for (int img = blockIdx.x; img < p.B; img += gridDim.x) {
    const float* pts = p.pts + (long long)img * p.img_stride;
    int k = p.n_clusters[img];
    k = k < 1 ? 1 : (k > p.max_k ? p.max_k : k);
    if (k > N) k = N;
    const uint32_t key = p.image_keys ? (uint32_t)p.image_keys[img] : (uint32_t)img;
    __syncthreads();

    // ---- variance of the data (sklearn: tol * mean of the per-feature variances)
    double vsum = 0.0;
    for (int j = 0; j < dims; ++j) {
      double s = 0.0, s2 = 0.0;
      for (int n = tid; n < N; n += SEG_THREADS) {
        const double v = pts[(long long)n * p.pt_stride + (long long)j * p.dim_stride];
        s += v; s2 += v * v;
      }
      s = seg_block_sum(s, red, tid);
      s2 = seg_block_sum(s2, red, tid);
      const double mean = s / N;
      vsum += s2 / N - mean * mean;
    }
    const double tol_abs = (double)p.tol * (vsum / dims);

    // ---- k-means++ seeding (sklearn _kmeans_plusplus: first centre uniform, then 2 + log k candidates drawn with
    // probability proportional to the current squared distance; the candidate with the smallest potential wins)
    uint32_t ctr = 0;
    const int first = min(N - 1, (int)(seg_uniform(p.seed, key, ctr++) * N));
    for (int j = tid; j < dims; j += SEG_THREADS) cen[j] = pts[(long long)first * p.pt_stride + (long long)j * p.dim_stride];
    __syncthreads();
    double pot = 0.0;
    for (int n = tid; n < N; n += SEG_THREADS) {
      const float d2 = seg_dist2(pts + (long long)n * p.pt_stride, p.dim_stride, cen, dims);
      mind2[n] = d2;
      pot += d2;
    }
    pot = seg_block_sum(pot, red, tid);
    const int trials = 2 + (int)log((double)k);
    for (int c = 1; c < k; ++c) {
      int best_cand = -1;
      double best_pot = 0.0;
      for (int t = 0; t < trials; ++t) {
        // sample an index with probability mind2 / pot: thread 0 walks the cumulative sum (N <= a few thousand)
        const double target = seg_uniform(p.seed, key, ctr++) * pot;
        if (tid == 0) {
          double acc = 0.0;
          int pick = N - 1;
          for (int n = 0; n < N; ++n) {
            acc += mind2[n];
            if (acc > target) { pick = n; break; }
          }
          s_pick = pick;
        }
        __syncthreads();
        const int cand = s_pick;
        float* cc = cen + (size_t)c * dims;   // slot c doubles as the candidate buffer
        __syncthreads();
        for (int j = tid; j < dims; j += SEG_THREADS) cc[j] = pts[(long long)cand * p.pt_stride + (long long)j * p.dim_stride];
        __syncthreads();
        double np_ = 0.0;
        for (int n = tid; n < N; n += SEG_THREADS)
          np_ += fminf(mind2[n], seg_dist2(pts + (long long)n * p.pt_stride, p.dim_stride, cc, dims));
        np_ = seg_block_sum(np_, red, tid);
        if (best_cand < 0 || np_ < best_pot) { best_cand = cand; best_pot = np_; }
      }
      float* cc = cen + (size_t)c * dims;
      __syncthreads();
      for (int j = tid; j < dims; j += SEG_THREADS) cc[j] = pts[(long long)best_cand * p.pt_stride + (long long)j * p.dim_stride];
      __syncthreads();
      for (int n = tid; n < N; n += SEG_THREADS)
        mind2[n] = fminf(mind2[n], seg_dist2(pts + (long long)n * p.pt_stride, p.dim_stride, cc, dims));
      pot = best_pot;
      __syncthreads();
    }

    // ---- Lloyd iterations
    for (int n = tid; n < N; n += SEG_THREADS) lab[n] = 255;
    int iters = 0, converged = 0;
    double inertia = 0.0;
    for (int it = 0; it < p.max_iter; ++it) {
      // E step: nearest centre (ties -> lower index), label changes counted
      for (int i = tid; i < k * dims; i += SEG_THREADS) sums[i] = 0.0;
      if (tid < SEG_MAX_CLUSTERS) counts[tid] = 0;
      if (tid == 0) s_changed = 0;
      __syncthreads();
      int changed = 0;
      double in_part = 0.0;
      for (int n = tid; n < N; n += SEG_THREADS) {
        const float* pn = pts + (long long)n * p.pt_stride;
        float bd = INFINITY;
        int bc = 0;
        for (int c = 0; c < k; ++c) {
          const float d2 = seg_dist2(pn, p.dim_stride, cen + (size_t)c * dims, dims);
          if (d2 < bd) { bd = d2; bc = c; }
        }
        changed += lab[n] != bc;
        lab[n] = (uint8_t)bc;
        mind2[n] = bd;
        in_part += bd;
        // M step accumulation in fp64 (the sum of fp32 values in fp64 is order independent to ~1e-16 relative)
        atomicAdd(&counts[bc], 1);
        for (int j = 0; j < dims; ++j) atomicAdd(&sums[(size_t)bc * dims + j], (double)pn[(long long)j * p.dim_stride]);
      }
      inertia = seg_block_sum(in_part, red, tid);
      if (changed) atomicAdd(&s_changed, changed);
      __syncthreads();
      iters = it + 1;
      if (s_changed == 0) { converged = 1; break; }   // strict convergence: labels did not change
      // empty clusters take the point that is farthest from its centre (sklearn _relocate_empty_clusters)
      for (int c = 0; c < k; ++c) {
        if (counts[c] != 0) continue;   // block-uniform (shared memory, read after the barrier)
        double bv = -1.0;
        int bi = 0;
        for (int n = tid; n < N; n += SEG_THREADS)
          if ((double)mind2[n] > bv) { bv = mind2[n]; bi = n; }
        for (int o = 16; o > 0; o >>= 1) {
          const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
        __syncthreads();
        if (tid == 0) {
          for (int w = 1; w < SEG_WARPS; ++w)
            if (s_val[w] > s_val[0] || (s_val[w] == s_val[0] && s_idx[w] < s_idx[0])) { s_val[0] = s_val[w]; s_idx[0] = s_idx[w]; }
          const int far = s_idx[0], old = lab[far];
          const float* pf = pts + (long long)far * p.pt_stride;
          for (int j = 0; j < dims; ++j) {
            const double v = pf[(long long)j * p.dim_stride];
            sums[(size_t)old * dims + j] -= v;
            sums[(size_t)c * dims + j] = v;
          }
          counts[old] -= 1;
          counts[c] = 1;
          lab[far] = (uint8_t)c;
          mind2[far] = 0.f;
        }
        __syncthreads();
      }
      // M step: new centres, squared shift
      double shift = 0.0;
      for (int i = tid; i < k * dims; i += SEG_THREADS) {
        const int c = i / dims;
        const float nc = counts[c] > 0 ? (float)(sums[i] / (double)counts[c]) : cen[i];
        const double dlt = (double)nc - (double)cen[i];
        shift += dlt * dlt;
        cen[i] = nc;
      }
      shift = seg_block_sum(shift, red, tid);
      if (shift <= tol_abs) {   // sklearn: centre shift below tol -> stop, then one more E step fixes the labels
        for (int n = tid; n < N; n += SEG_THREADS) {
          const float* pn = pts + (long long)n * p.pt_stride;
          float bd = INFINITY;
          int bc = 0;
          for (int c = 0; c < k; ++c) {
            const float d2 = seg_dist2(pn, p.dim_stride, cen + (size_t)c * dims, dims);
            if (d2 < bd) { bd = d2; bc = c; }
          }
          lab[n] = (uint8_t)bc;
        }
        converged = 1;
        __syncthreads();
        break;
      }
    }

    // ---- background rule (extract.py:337-345, extract_utils.py:124-135): the label with the largest share of the
    // 2 (H + W) border cells (corners counted twice, ties -> smallest label) is swapped with label 0
    if (p.infer_bg && p.Hs * p.Ws == N) {
      if (tid < SEG_MAX_CLUSTERS) counts[tid] = 0;
      __syncthreads();
      for (int i = tid; i < 2 * (p.Hs + p.Ws); i += SEG_THREADS) {
        int n;
        if (i < p.Hs) n = i * p.Ws;                                   // segmap[:, 0]
        else if (i < 2 * p.Hs) n = (i - p.Hs) * p.Ws + p.Ws - 1;      // segmap[:, -1]
        else if (i < 2 * p.Hs + p.Ws) n = i - 2 * p.Hs;               // segmap[0, :]
        else n = (p.Hs - 1) * p.Ws + (i - 2 * p.Hs - p.Ws);           // segmap[-1, :]
        atomicAdd(&counts[lab[n]], 1);
      }
      __syncthreads();
      int bg = 0;
      for (int c = 1; c < k; ++c)
        if (counts[c] > counts[bg]) bg = c;
      // labels that do not occur at all are not in np.unique(segmap); they have count 0 and can only win when every
      // count is 0, which cannot happen (the border is not empty)
      for (int n = tid; n < N; n += SEG_THREADS) {
        const int l = lab[n];
        lab[n] = (uint8_t)(l == bg ? 0 : (l == 0 ? bg : l));
      }
      __syncthreads();
    }
    for (int n = tid; n < N; n += SEG_THREADS) p.labels[(long long)img * N + n] = lab[n];
    if (tid == 0) {
      p.info[img * 2 + 0] = iters;
      p.info[img * 2 + 1] = converged;
      if (p.inertia) p.inertia[img] = (float)inertia;
    }
    __syncthreads();
  }
}

}  // namespace dss

using namespace dss;

extern "C" int dss_segment_threshold(const float* evecs, int B, int K, int N, int which, float threshold, uint8_t* mask,
                                     dss_stream_t stream) {
  DSS_REQUIRE(evecs && mask, "segment_threshold: null pointer");
  DSS_REQUIRE(B > 0 && N > 0 && which >= 0 && which < K, "segment_threshold: bad shape / eigenvector index (K=%d which=%d)",
              K, which);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LaunchScope scope(st, KC_MISC);
  const long long total = (long long)B * N;
  threshold_mask_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(evecs, K, N, which, threshold, mask, B);
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}

extern "C" int dss_segment_kmeans(const float* points, long long image_stride, long long point_stride, long long dim_stride,
                                  int B, int N, int dims, const int* n_clusters, const int* image_keys, int max_clusters,
                                  int grid_h, int grid_w, int infer_bg_index, unsigned int seed, int max_iter, float tol,
                                  uint8_t* labels, int* info, float* inertia, dss_stream_t stream) {
  DSS_REQUIRE(points && n_clusters && labels && info, "segment_kmeans: null pointer");
  DSS_REQUIRE(B > 0 && N > 0 && dims > 0, "segment_kmeans: empty problem");
  DSS_REQUIRE(max_clusters >= 1 && max_clusters <= SEG_MAX_CLUSTERS, "segment_kmeans: 1 <= max_clusters <= %d",
              SEG_MAX_CLUSTERS);
  DSS_REQUIRE(!infer_bg_index || grid_h * grid_w == N, "segment_kmeans: grid %dx%d does not match %d points", grid_h,
              grid_w, N);
  KmeansParams p;
  p.pts = points; p.img_stride = image_stride; p.pt_stride = point_stride; p.dim_stride = dim_stride;
  p.n_clusters = n_clusters; p.image_keys = image_keys; p.labels = labels; p.info = info; p.inertia = inertia;
  p.B = B; p.N = N; p.dims = dims; p.max_k = max_clusters; p.Hs = grid_h; p.Ws = grid_w; p.infer_bg = infer_bg_index;
  p.max_iter = max_iter > 0 ? max_iter : 300;
  p.tol = tol >= 0.f ? tol : 1e-4f;
  p.seed = seed;
  const size_t smem = align_up((size_t)max_clusters * dims * 4, 16) + (size_t)max_clusters * dims * 8 +
                      SEG_MAX_CLUSTERS * 4 + (size_t)N * 4 + align_up((size_t)N, 16) + 64;
  DSS_REQUIRE(smem <= 200 * 1024, "segment_kmeans: %d clusters x %d dims x %d points need %zu B of shared memory", max_clusters,
              dims, N, smem);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DSS_CHECK_CUDA(allow_dynamic_smem(kmeans_segment_kernel, (int)smem));
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  const int grid = B < 2 * sms ? B : 2 * sms;
  LaunchScope scope(st, KC_MISC);
  kmeans_segment_kernel<<<grid, SEG_THREADS, smem, st>>>(p);
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}
