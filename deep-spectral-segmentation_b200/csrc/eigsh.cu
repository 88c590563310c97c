// Smallest-K eigenpairs of the graph Laplacian pencil (D - W) v = lambda D v   (reference extract/extract.py:222-240,
// which calls scipy.sparse.linalg.eigsh(D - W, k=K, sigma=0, which='LM', M=D): dense LU + ARPACK shift-invert).
//
// B200 design: no factorisation. With S = D^-1/2 W D^-1/2 the pencil's smallest eigenvalues are 1 - (largest
// eigenvalues of S) and v = D^-1/2 u. The top eigenpair of S is known in closed form (u0 = D^1/2 1 / sqrt(sum D),
// mu0 = 1) and is deflated analytically; the next K-1 come from Lanczos with full re-orthogonalisation (two
// classical Gram-Schmidt passes) -- ~16-50 symmetric mat-vecs per image instead of an N^3 LU.
//
// One persistent CTA per image: the whole iteration (mat-vec, re-orthogonalisation, Ritz extraction, convergence
// test) runs inside one kernel with block-level barriers only; images are independent, so a batch fills the GPU
// with one CTA per SM and nothing ever synchronises across CTAs. The mat-vec is the only HBM stream of the
// kernel and W is symmetric, so only its UPPER TRIANGLE is read: row r contributes W[r, c >= r] x[c] to y[r] (warp
// reduction) and W[r, c > r] x[r] to y[c] (per-lane column accumulators in registers, combined across warps through
// shared memory once per mat-vec) -- 2 N^2 bytes per step instead of 4 N^2. The degree D = W 1 comes from the
// affinity kernel's epilogue (dss_affinity) when the caller passes it; otherwise one extra pass computes it.
// The Lanczos basis lives in a per-CTA global scratch (L2), the working vectors in shared memory. Ritz values of the tridiagonal matrix come from a 32-way
// Sturm multisection in fp64 (one warp per eigenvalue), Ritz vectors from a twisted factorisation.
#include <math.h>

#include "common.cuh"

namespace dss {

constexpr int EIG_THREADS = 512;
constexpr int EIG_WARPS = EIG_THREADS / 32;
constexpr int EIG_MAX_K = 64;

constexpr int EIG_STRIP_CH = 4;                    // float4 column chunks per lane and strip
constexpr int EIG_STRIP = 32 * 4 * EIG_STRIP_CH;   // 512 columns per strip

struct EigParams {
  const float* W;     // [B, N, ldw]
  const float* deg;   // [B, N] row sums of W (from the affinity epilogue) or null: computed here
  float* evals;       // [B, K]
  float* evecs;       // [B, K, N]
  int* info;          // [B, 4]
  float* resid;       // [B, K] or null
  float* basis;       // per-CTA scratch: [(mmax+1), Npad]
  double* tri;        // per-CTA scratch: [2, Kw, mmax]   (Ritz vectors of T, temp)
  int B, N, ldw, Npad, K, mmax;
  int mode;           // 0: normalised Laplacian pencil, 1: unnormalised Laplacian, 2: plain top-K of the matrix itself
  float tol;
};

template <int NW>
__device__ __forceinline__ double block_sum(double v, double* red, int tid) {
  v = warp_sum(v);
  __syncthreads();  // protect red from the previous use
  if ((tid & 31) == 0) red[tid >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < NW; ++i) s += red[i];
  return s;
}

__device__ __forceinline__ float hash_uniform(uint32_t i, uint32_t seed) {
  uint32_t x = i * 2654435761u ^ (seed * 0x9E3779B9u + 0x85EBCA6Bu);
  x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
  return (float)(x >> 8) * (2.0f / 16777216.0f) - 1.0f;
}

// dot of a global (or shared) vector with the shared vector w, whole warp, float4 path when Npad-aligned
__device__ __forceinline__ float warp_dot(const float* __restrict__ a, const float* __restrict__ w, int N, int lane) {
  float s0 = 0.f, s1 = 0.f;
  const int n4 = N >> 2;
  const float4* a4 = reinterpret_cast<const float4*>(a);
  const float4* w4 = reinterpret_cast<const float4*>(w);
  for (int i = lane; i < n4; i += 32) {
    const float4 x = a4[i], y = w4[i];
    s0 = fmaf(x.x, y.x, s0); s1 = fmaf(x.y, y.y, s1);
    s0 = fmaf(x.z, y.z, s0); s1 = fmaf(x.w, y.w, s1);
  }
  for (int i = (n4 << 2) + lane; i < N; i += 32) s0 = fmaf(a[i], w[i], s0);
  return warp_sum(s0 + s1);
}

// number of eigenvalues of the n x n tridiagonal (alpha, beta) that are < x
__device__ __forceinline__ int sturm_count(const double* alpha, const double* beta2, int n, double x) {
  int cnt = 0;
  double q = alpha[0] - x;
  if (q == 0.0) q = -1e-300;
  cnt += q < 0.0;
  for (int i = 1; i < n; ++i) {
    q = (alpha[i] - x) - beta2[i - 1] / q;
    if (q == 0.0) q = -1e-300;
    cnt += q < 0.0;
  }
  return cnt;
}

__host__ __device__ inline size_t eig_double_bytes(int mmax) {
  size_t nd = (size_t)3 * mmax + 2 * (EIG_MAX_K + 1) + EIG_WARPS;
  nd = (nd + 1) & ~(size_t)1;
  return nd * sizeof(double);
}

// R = rows per warp and pass of the mat-vec (R independent 128-bit loads in flight per lane), MINB = CTAs per SM the
// register budget is sized for. The library launches <4, 1, EIG_THREADS>: one CTA per SM, 128 registers, all 16 loads
// of a row group's column blocks in flight per lane. (Measured on the 296-image step at N = 900: <2, 2, 512>, two
// images per SM at 64 registers, 2.27 ms vs 1.94 ms; <4, 2, 256> equal, and 3 % slower on the VOC mix.)
template <int R, int MINB, int NT>
__global__ void __launch_bounds__(NT, MINB)
lanczos_laplacian_kernel(EigParams p) {
  constexpr int NW = NT / 32;                          // warps of this instantiation (the layout keeps room for NW)
  constexpr int PRE = (MINB == 2 && NT == NT) ? 2 : EIG_STRIP_CH;   // column blocks whose loads are in flight together
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int N = p.N, Npad = p.Npad, mmax = p.mmax, K = p.K, ldw = p.ldw;
  const bool lapn = p.mode == 0, plain = p.mode == 2;
  const int Kw = plain ? p.K : p.K - 1;   // Ritz pairs wanted from Lanczos (the Laplacian's null vector is analytic)
  const int off = plain ? 0 : 1;          // output slot of the first Lanczos pair
  // shared layout
  double* alpha = reinterpret_cast<double*>(smem_raw);      // [mmax]
  double* beta = alpha + mmax;                               // [mmax]   beta[j] = ||w_j|| (couples j, j+1)
  double* beta2 = beta + mmax;                               // [mmax]
  double* theta = beta2 + mmax;                              // [EIG_MAX_K + 1] (the wanted pairs + the guard pair)
  double* red = theta + EIG_MAX_K + 1;                       // [EIG_WARPS]
  double* resid_s = red + EIG_WARPS;                         // [EIG_MAX_K + 1]
  // float arrays start 16-byte aligned (float4 access): the double block is padded to an even count
  float* xs = reinterpret_cast<float*>(smem_raw + eig_double_bytes(mmax));  // [Npad] scaled mat-vec input
  float* wv = xs + Npad;                                     // [Npad] working vector
  float* vcur = wv + Npad;                                   // [Npad] current Lanczos vector
  float* dsc = vcur + Npad;                                  // [Npad] D^-1/2 (lapnorm) or D (unnormalised)
  float* u0 = dsc + Npad;                                    // [Npad] deflated null vector (unit 2-norm)
  float* ycol = u0 + Npad;                                   // [Npad] column part of the symmetric mat-vec
  const int stripw = Npad < EIG_STRIP ? Npad : EIG_STRIP;
  float* colbuf = ycol + Npad;                               // [NW][stripw] per-warp column accumulators
  float* coef = colbuf + (size_t)EIG_WARPS * stripw;         // [mmax + 2]
  __shared__ int s_flag;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* basis = p.basis + (size_t)blockIdx.x * (size_t)(mmax + 1) * Npad;
  double* triS = p.tri + (size_t)blockIdx.x * 2 * (size_t)(Kw + 1) * mmax;  // [Kw + 1][mmax] Ritz vectors of T
  double* triB = triS + (size_t)(Kw + 1) * mmax;                            // [Kw + 1][mmax] temp

  for (int img = blockIdx.x; img < p.B; img += gridDim.x) {
    const float* W = p.W + (size_t)img * N * ldw;
    __syncthreads();
    // ---- degree D = W 1  (row_sum, extract_utils.py:217), clamp < 1e-12 -> 1 (:218)
    if (plain) {              // plain top-K mode: no degree
      for (int i = tid; i < N; i += NT) wv[i] = 1.0f;
    } else if (p.deg != nullptr) {   // accumulated by the affinity epilogue: no pass over W
      for (int i = tid; i < N; i += NT) wv[i] = __ldg(p.deg + (size_t)img * N + i);
    } else {
      for (int r = warp; r < N; r += NW) {
        const float4* row = reinterpret_cast<const float4*>(W + (size_t)r * ldw);
        float s0 = 0.f, s1 = 0.f;
        for (int i = lane; i < (Npad >> 2); i += 32) {  // pad columns [N, Npad) are zero
          const float4 v = __ldg(row + i);
          s0 += v.x + v.y; s1 += v.z + v.w;
        }
        const float s = warp_sum(s0 + s1);
        if (lane == 0) wv[r] = s;
      }
    }
    __syncthreads();
    double part = 0.0;
    for (int i = tid; i < Npad; i += NT) {
      float dg = 0.f;
      if (i < N) {
        dg = wv[i];
        if (dg < 1e-12f) dg = 1.0f;   // get_diagonal's threshold (extract_utils.py:218)
        part += (double)dg;
      }
      wv[i] = dg;
    }
    const double sumD = block_sum<NW>(part, red, tid);
    for (int i = tid; i < Npad; i += NT) {
      const float dg = wv[i];
      if (i < N) {
        if (lapn) {
          dsc[i] = (float)(1.0 / sqrt((double)dg));
          u0[i] = (float)(sqrt((double)dg) / sqrt(sumD));
        } else if (plain) {
          dsc[i] = 1.0f;   // operator = the matrix itself, nothing is deflated
          u0[i] = 0.f;
        } else {
          dsc[i] = dg;
          u0[i] = (float)(1.0 / sqrt((double)N));
        }
      } else {
        dsc[i] = 0.f; u0[i] = 0.f;
      }
      xs[i] = 0.f; vcur[i] = 0.f;
    }
    __syncthreads();

    int n = 0;          // Lanczos steps done
    int converged = (Kw <= 0);
    bool have_theta = false;
    if (Kw > 0) {
      // ---- start vector: deterministic pseudo-random, orthogonal to u0
      for (int i = tid; i < Npad; i += NT) wv[i] = (i < N) ? hash_uniform((uint32_t)i, 0x1234567u) : 0.f;
      __syncthreads();
      for (int pass = 0; pass < 2; ++pass) {
        double d = 0.0;
        for (int i = tid; i < N; i += NT) d += (double)wv[i] * (double)u0[i];
        const float c = (float)block_sum<NW>(d, red, tid);
        for (int i = tid; i < N; i += NT) wv[i] = fmaf(-c, u0[i], wv[i]);
        __syncthreads();
      }
      {
        double d = 0.0;
        for (int i = tid; i < N; i += NT) d += (double)wv[i] * (double)wv[i];
        const float inv = (float)(1.0 / sqrt(block_sum<NW>(d, red, tid)));
        for (int i = tid; i < Npad; i += NT) {
          const float v = (i < N) ? wv[i] * inv : 0.f;
          vcur[i] = v;
          basis[i] = v;
        }
      }
      __syncthreads();

      double anorm = 1.0;
      for (int j = 0; j < mmax; ++j) {
        // ---- mat-vec  w = S v  (lapnorm)   or   w = (W - D) v  (unnormalised: top of -(D-W)), upper triangle of W only
        for (int i = tid; i < Npad; i += NT) {
          xs[i] = lapn ? dsc[i] * vcur[i] : vcur[i];
          wv[i] = 0.f;   // row part, accumulated strip by strip by the warp that owns the row
        }
        __syncthreads();
        for (int s0 = 0; s0 < Npad; s0 += EIG_STRIP) {
          const int s1 = min(Npad, s0 + EIG_STRIP);          // columns [s0, s1) of this strip
          float4 colacc[EIG_STRIP_CH];
#pragma unroll
          for (int k = 0; k < EIG_STRIP_CH; ++k) colacc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
          const float4* x4 = reinterpret_cast<const float4*>(xs);
          const float4* W4 = reinterpret_cast<const float4*>(W);
          // R consecutive rows per warp and pass (r % R == 0, so their diagonal elements share one 4-column chunk)
          for (int r = warp * R; r < N && r < s1; r += NW * R) {
            // 32-bit chunk offsets from the image's base (N * ldw < 2^31): one IMAD.WIDE per load instead of a 64-bit
            // row pointer that the 64-register budget forces the compiler to rebuild in every block
            const float4* rowp[R];
            float xr[R], acc[R];
#pragma unroll
            for (int q = 0; q < R; ++q) {
              const bool ok = r + q < N;
              rowp[q] = W4 + (((ok ? r + q : N - 1) * ldw) >> 2);
              // opaque to the optimiser: without this the row pointer is re-derived from (image, row, ldw) inside every
              // one of the unrolled blocks below (~25 integer instructions per pair of loads)
              asm volatile("" : "+l"(rowp[q]));
              xr[q] = ok ? xs[r + q] : 0.f;
              acc[q] = 0.f;
            }
            const int chd = r >> 2;                          // chunk that holds the diagonal elements of these rows
            // warp-uniform range of k blocks (32 chunks each) that intersect columns [max(r, s0), s1): the blocks left
            // of the diagonal are skipped as a whole, and the per-element masks of the diagonal chunk are only evaluated
            // in the one block that contains it (round 2, first version: ncu showed 1.2 G warp instructions per launch,
            // 14 % of them FFMA -- the predicated mask / address arithmetic of all eight blocks was issued for every row)
            const int cb = s0 >> 2, nch = s1 >> 2;
            const int k_first = chd > cb ? (chd - cb) >> 5 : 0;
            const int k_end = ((s1 - s0) + 127) >> 7;
            // Groups of PRE blocks: all of a group's loads (PRE x R independent 128-bit loads per lane) are issued before
            // any of them is consumed -- with one block at a time the warps stalled on the first FFMA of every block
            // (55 % of the stall samples) at 46 % of the DRAM peak: not enough bytes in flight.
#pragma unroll
            for (int k0 = 0; k0 < EIG_STRIP_CH; k0 += PRE) {
              if (k0 + PRE <= k_first || k0 >= k_end) continue;   // (uniform) nothing of this group right of the diagonal
              float4 u[PRE][R];
              bool act[PRE];
#pragma unroll
              for (int kk = 0; kk < PRE; ++kk) {
                const int k = k0 + kk;
                const int ch = cb + lane + 32 * k;           // this lane's chunk of block k: columns 4 ch .. 4 ch + 3
                act[kk] = k >= k_first && k < k_end && ch >= chd && ch < nch;
#pragma unroll
                for (int q = 0; q < R; ++q) u[kk][q] = act[kk] ? __ldg(rowp[q] + ch) : make_float4(0.f, 0.f, 0.f, 0.f);
              }
#pragma unroll
              for (int kk = 0; kk < PRE; ++kk) {
                const int k = k0 + kk;
                if (k < k_first || k >= k_end) continue;     // (uniform)
                const int ch = cb + lane + 32 * k;
                if (!act[kk]) continue;
                const float4 x = x4[ch];
                if (k == k_first && ch == chd) {             // the chunk that holds the diagonal elements of these rows
#pragma unroll
                  for (int q = 0; q < R; ++q) {
                    // row part: drop the elements left of the diagonal; column part: drop the diagonal as well
                    const int dq = (r + q) & 3;
                    float4 a = u[kk][q];
                    if (dq > 0) a.x = 0.f;
                    if (dq > 1) a.y = 0.f;
                    if (dq > 2) a.z = 0.f;
                    float4 c = a;
                    if (dq == 0) c.x = 0.f;
                    if (dq == 1) c.y = 0.f;
                    if (dq == 2) c.z = 0.f;
                    if (dq == 3) c.w = 0.f;
                    acc[q] = fmaf(a.x, x.x, acc[q]); acc[q] = fmaf(a.y, x.y, acc[q]);
                    acc[q] = fmaf(a.z, x.z, acc[q]); acc[q] = fmaf(a.w, x.w, acc[q]);
                    colacc[k].x = fmaf(c.x, xr[q], colacc[k].x); colacc[k].y = fmaf(c.y, xr[q], colacc[k].y);
                    colacc[k].z = fmaf(c.z, xr[q], colacc[k].z); colacc[k].w = fmaf(c.w, xr[q], colacc[k].w);
                  }
                } else {
#pragma unroll
                  for (int q = 0; q < R; ++q) {
                    const float4 a = u[kk][q];
                    acc[q] = fmaf(a.x, x.x, acc[q]); acc[q] = fmaf(a.y, x.y, acc[q]);
                    acc[q] = fmaf(a.z, x.z, acc[q]); acc[q] = fmaf(a.w, x.w, acc[q]);
                    colacc[k].x = fmaf(a.x, xr[q], colacc[k].x); colacc[k].y = fmaf(a.y, xr[q], colacc[k].y);
                    colacc[k].z = fmaf(a.z, xr[q], colacc[k].z); colacc[k].w = fmaf(a.w, xr[q], colacc[k].w);
                  }
                }
              }
            }
#pragma unroll
            for (int q = 0; q < R; ++q) {
              const float sa = warp_sum(acc[q]);
              if (lane == 0 && r + q < N) wv[r + q] += sa;   // row r is owned by this warp in every strip
            }
          }
          // column part of the strip: per-warp accumulators -> shared memory -> summed in warp order (deterministic)
          float4* cb = reinterpret_cast<float4*>(colbuf + (size_t)warp * stripw);
#pragma unroll
          for (int k = 0; k < EIG_STRIP_CH; ++k) {
            const int cl = lane + 32 * k;                    // chunk inside the strip
            if (4 * cl < s1 - s0) cb[cl] = colacc[k];
          }
          __syncthreads();
          for (int c = tid; c < s1 - s0; c += NT) {
            float sc = 0.f;
#pragma unroll
            for (int w2 = 0; w2 < NW; ++w2) sc += colbuf[(size_t)w2 * stripw + c];
            ycol[s0 + c] = sc;
          }
          __syncthreads();
        }
        for (int i = tid; i < Npad; i += NT) {
          const float sa = wv[i] + ycol[i];
          wv[i] = (i < N) ? (lapn ? dsc[i] * sa : (plain ? sa : sa - dsc[i] * xs[i])) : 0.f;
        }
        __syncthreads();
        // ---- full re-orthogonalisation (CGS2) against u0, v_0..v_j ; alpha_j = sum of the v_j coefficients
        double aj = 0.0;
        for (int pass = 0; pass < 2; ++pass) {
          for (int i = warp; i < j + 2; i += NW) {
            const float* a = (i == 0) ? u0 : ((i - 1 == j) ? vcur : basis + (size_t)(i - 1) * Npad);
            const float c = warp_dot(a, wv, N, lane);
            if (lane == 0) coef[i] = c;
          }
          __syncthreads();
          aj += (double)coef[j + 1];
          for (int i = tid; i < N; i += NT) {
            float acc = coef[0] * u0[i];
            for (int t = 0; t < j; ++t) acc = fmaf(coef[t + 1], basis[(size_t)t * Npad + i], acc);
            acc = fmaf(coef[j + 1], vcur[i], acc);
            wv[i] -= acc;
          }
          __syncthreads();
        }
        double d = 0.0;
        for (int i = tid; i < N; i += NT) d += (double)wv[i] * (double)wv[i];
        const double bj = sqrt(block_sum<NW>(d, red, tid));
        if (tid == 0) {
          alpha[j] = aj;
          beta[j] = bj;
          beta2[j] = bj * bj;
        }
        n = j + 1;
        anorm = fmax(anorm, fabs(aj) + bj);
        const bool breakdown = !(bj > 1e-7 * anorm);   // invariant subspace: all Ritz pairs are exact
        if (!breakdown) {
          const float inv = (float)(1.0 / bj);
          float* vn = basis + (size_t)(j + 1) * Npad;
          for (int i = tid; i < Npad; i += NT) {
            const float v = (i < N) ? wv[i] * inv : 0.f;
            vcur[i] = v;
            vn[i] = v;
          }
        }
        __syncthreads();

        // ---- convergence test on the K-1 largest Ritz pairs of T_n
        const int n0 = max(Kw + 4, 12);
        const int every = (n <= 64) ? 4 : 8;
        const bool check = breakdown || n == mmax || n >= N - 1 || (n >= n0 && ((n - n0) % every) == 0);
        const int kk = min(Kw, n);  // Ritz pairs that exist
        // + one GUARD pair (the next Ritz value): the wanted pairs having small residuals does not exclude an eigenvalue
        // of a tight cluster that has not emerged from the Krylov space yet; such an eigenvalue shows up as a poorly
        // converged next Ritz value whose residual interval reaches into the wanted range (found with K = 32 on a
        // spectrum with 1e-4 gaps: 81 steps, all residuals < tol, eigenvalue 32 off by 5e-3)
        const int kg = min(Kw + 1, n);
        if (check) {
          // Gershgorin bounds (every warp computes them redundantly: n <= mmax small)
          double gl = 1e300, gh = -1e300;
          for (int i = lane; i < n; i += 32) {
            const double off = (i > 0 ? beta[i - 1] : 0.0) + (i < n - 1 ? beta[i] : 0.0);
            gl = fmin(gl, alpha[i] - off);
            gh = fmax(gh, alpha[i] + off);
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            gl = fmin(gl, __shfl_xor_sync(0xffffffffu, gl, o));
            gh = fmax(gh, __shfl_xor_sync(0xffffffffu, gh, o));
          }
          const double span = fmax(gh - gl, 1e-30);
          gl -= 1e-3 * span; gh += 1e-3 * span;
          for (int k = warp; k < kg; k += NW) {
            // k-th largest eigenvalue = ascending index t = n-1-k ; lambda_t >= x  <=>  count(x) <= t
            const int t = n - 1 - k;
            double lo = gl, hi = gh;
            for (int round = 0; round < 11; ++round) {
              const double step = (hi - lo) / 33.0;
              const double x = lo + step * (double)(lane + 1);
              const int c = sturm_count(alpha, beta2, n, x);
              const unsigned mask = __ballot_sync(0xffffffffu, c <= t);
              const int np = __popc(mask);  // predicate is monotone: true for a prefix of lanes
              const double nlo = (np > 0) ? lo + step * (double)np : lo;
              const double nhi = (np < 32) ? lo + step * (double)(np + 1) : hi;
              lo = nlo; hi = nhi;
            }
            const double th = 0.5 * (lo + hi);
            // Ritz vector of T by twisted factorisation of T - th I (lane 0, sequential recurrences)
            double* zs = triS + (size_t)k * mmax;
            double* tb = triB + (size_t)k * mmax;
            if (lane == 0) {
              if (n == 1) {
                zs[0] = 1.0;
              } else {
                double dp = alpha[0] - th;
                for (int i = 0; i < n - 1; ++i) {
                  if (dp == 0.0) dp = 1e-300;
                  zs[i] = dp;
                  dp = (alpha[i + 1] - th) - beta2[i] / dp;
                }
                if (dp == 0.0) dp = 1e-300;
                zs[n - 1] = dp;
                double dm = alpha[n - 1] - th;
                double gmin = fabs(zs[n - 1] + dm - (alpha[n - 1] - th));
                int r = n - 1;
                if (dm == 0.0) dm = 1e-300;
                tb[n - 1] = dm;
                for (int i = n - 2; i >= 0; --i) {
                  dm = (alpha[i] - th) - beta2[i] / dm;
                  if (dm == 0.0) dm = 1e-300;
                  tb[i] = dm;
                  const double g = fabs(zs[i] + dm - (alpha[i] - th));
                  if (g < gmin) { gmin = g; r = i; }
                }
                // z_r = 1 ; upward z_i = -beta_i z_{i+1} / d+_i ; downward z_{i+1} = -beta_i z_i / d-_{i+1}
                double z = 1.0;
                const double dpr = zs[r];
                (void)dpr;
                zs[r] = 1.0;
                // upward needs d+_i for i < r which are still stored in zs[i]
                for (int i = r - 1; i >= 0; --i) {
                  z = -beta[i] * z / zs[i];
                  zs[i] = z;
                }
                z = 1.0;
                for (int i = r; i < n - 1; ++i) {
                  z = -beta[i] * z / tb[i + 1];
                  zs[i + 1] = z;
                }
              }
            }
            __syncwarp();
            double nn = 0.0;
            for (int i = lane; i < n; i += 32) nn += zs[i] * zs[i];
            nn = warp_sum(nn);
            const double inv = 1.0 / sqrt(nn);
            for (int i = lane; i < n; i += 32) zs[i] *= inv;
            __syncwarp();
            if (lane == 0) {
              theta[k] = th;
              resid_s[k] = fabs(beta[n - 1] * zs[n - 1]);
            }
          }
          __syncthreads();
          if (tid == 0) {
            int ok = 1;
            for (int k = 0; k < kk; ++k) ok &= (resid_s[k] <= (double)p.tol * anorm);
            ok &= (kk == Kw);
            if (kg > Kw && Kw > 0 && !breakdown && n < N - 1)   // guard: nothing hidden above the last wanted Ritz value
              ok &= (theta[Kw] + resid_s[Kw] <= theta[Kw - 1] + (double)p.tol * anorm);
            s_flag = ok;
          }
          __syncthreads();
          converged = s_flag;
          have_theta = true;
          if (converged || breakdown) break;
        }
      }
    }

    // plain mode serves which='LM': report if a negative eigenvalue is larger in magnitude than the K-th positive one
    int lm_differs = 0;
    if (plain && n > 0 && have_theta) {
      // number of Ritz values below -|theta_K|: any such eigenvalue would be selected by which='LM' instead
      lm_differs = sturm_count(alpha, beta2, n, -fabs(theta[min(Kw, n) - 1])) > 0 ? 1 : 0;
    }
    // ---- outputs: ascending eigenvalues, D-orthonormal (lapnorm) / unit (unnormalised) vectors, sign rule
    float* ev = p.evals + (size_t)img * K;
    float* evec = p.evecs + (size_t)img * K * N;
    {
      const float c0 = lapn ? (float)(1.0 / sqrt(sumD)) : (float)(1.0 / sqrt((double)N));
      if (!plain)
        for (int i = tid; i < N; i += NT) evec[i] = c0;
      if (tid == 0) {
        if (!plain) {
          ev[0] = 0.f;
          if (p.resid) p.resid[(size_t)img * K] = 0.f;
        }
        p.info[img * 4 + 0] = n;
        p.info[img * 4 + 1] = converged ? 1 : 0;
        p.info[img * 4 + 2] = lm_differs;
        p.info[img * 4 + 3] = 0;
      }
    }
    const int have = min(Kw, n);  // Ritz pairs available
    for (int k = 0; k < Kw; ++k) {
      float* out = evec + (size_t)(k + off) * N;
      if (k >= have) {  // degenerate request (K-1 > steps possible): fill with NaN
        for (int i = tid; i < N; i += NT) out[i] = __int_as_float(0x7fc00000);
        if (tid == 0) ev[k + off] = __int_as_float(0x7fc00000);
        continue;
      }
      const double* zs = triS + (size_t)k * mmax;
      double d = 0.0;
      for (int i = tid; i < N; i += NT) {
        float acc = 0.f;
        for (int t = 0; t < n; ++t) acc = fmaf((float)zs[t], basis[(size_t)t * Npad + i], acc);
        wv[i] = acc;
        d += (double)acc * (double)acc;
      }
      const float inv = (float)(1.0 / sqrt(block_sum<NW>(d, red, tid)));
      int pos = 0;
      for (int i = tid; i < N; i += NT) {
        const float v = lapn ? wv[i] * inv * dsc[i] : wv[i] * inv;
        wv[i] = v;
        pos += v > 0.f;
      }
      const int npos = (int)(block_sum<NW>((double)pos, red, tid) + 0.5);
      // sign rule (extract.py:237-240): flip iff 0.5 < mean(v > 0) < 1.0
      const float sgn = (2 * npos > N && npos < N) ? -1.f : 1.f;
      for (int i = tid; i < N; i += NT) out[i] = sgn * wv[i];
      if (tid == 0) {
        ev[k + off] = lapn ? (float)(1.0 - theta[k]) : (plain ? (float)theta[k] : (float)(-theta[k]));
        if (p.resid) p.resid[(size_t)img * K + k + off] = (float)resid_s[k];
      }
      __syncthreads();
    }
  }
}

static size_t eig_smem_bytes(int Npad, int mmax) {
  const int stripw = Npad < EIG_STRIP ? Npad : EIG_STRIP;
  return eig_double_bytes(mmax) + (size_t)6 * Npad * sizeof(float) + (size_t)EIG_WARPS * stripw * sizeof(float) +
         (size_t)(mmax + 2) * sizeof(float) + 16;
}

static int eig_resolve(int N, int K, int max_steps) {
  int mmax = max_steps > 0 ? max_steps : 320;
  if (mmax > N - 1) mmax = N - 1;
  if (mmax < K) mmax = K;
  if (mmax < 1) mmax = 1;
  return mmax;
}

// one CTA per image, at most one per SM
static int eig_grid(int B) {
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  return B < sms ? B : sms;
}

}  // namespace dss

using namespace dss;

extern "C" size_t dss_eigsh_workspace_bytes(int B, int N, int K, int max_steps) {
  if (B <= 0 || N <= 0 || K <= 0) return 0;
  const int Npad = (N + 3) & ~3;
  const int mmax = eig_resolve(N, K, max_steps);
  const int grid = eig_grid(B);
  const size_t basis = align_up((size_t)grid * (mmax + 1) * Npad * sizeof(float), 256);
  const size_t tri = align_up((size_t)grid * 2 * (K + 1) * mmax * sizeof(double), 256);
  return basis + tri;
}

static int eigsh_launch(const float* Wmat, const float* deg, int ldw, int B, int N, int K, int mode, float tol, int max_steps,
                        float* evals, float* evecs, int* info, float* resid, void* ws, size_t ws_bytes,
                        dss_stream_t stream) {
  DSS_REQUIRE(Wmat && evals && evecs && info && ws, "eigsh: null pointer");
  DSS_REQUIRE(B > 0 && N > 1, "eigsh: empty problem B=%d N=%d", B, N);
  DSS_REQUIRE(K >= 1 && K <= EIG_MAX_K && K < N, "eigsh: need 1 <= K <= %d and K < N (K=%d N=%d)", EIG_MAX_K, K, N);
  DSS_REQUIRE(ldw >= N && ldw % 4 == 0, "eigsh: ldw must be >= N and a multiple of 4 (N=%d ldw=%d)", N, ldw);
  DSS_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0 && (reinterpret_cast<uintptr_t>(Wmat) & 15) == 0,
              "eigsh: workspace must be 256-byte aligned and W 16-byte aligned");
  const size_t need = dss_eigsh_workspace_bytes(B, N, K, max_steps);
  if (ws_bytes < need) {
    set_error("eigsh: workspace too small (%zu < %zu)", ws_bytes, need);
    return DSS_ERR_WORKSPACE;
  }
  EigParams p;
  p.W = Wmat; p.deg = deg; p.evals = evals; p.evecs = evecs; p.info = info; p.resid = resid;
  p.B = B; p.N = N; p.ldw = ldw; p.Npad = (N + 3) & ~3; p.K = K; p.mode = mode;
  p.mmax = eig_resolve(N, K, max_steps);
  p.tol = tol > 0.f ? tol : 1e-6f;
  const int grid = eig_grid(B);
  p.basis = reinterpret_cast<float*>(ws);
  p.tri = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(ws) +
                                    align_up((size_t)grid * (p.mmax + 1) * p.Npad * sizeof(float), 256));
  const size_t smem = eig_smem_bytes(p.Npad, p.mmax);
  if (smem > 227 * 1024) {
    set_error("eigsh: N=%d with max_steps=%d needs %zu B of shared memory (> 227 KB)", N, p.mmax, smem);
    return DSS_ERR_UNSUPPORTED;
  }
  DSS_CHECK_CUDA(allow_dynamic_smem(lanczos_laplacian_kernel<4, 1, EIG_THREADS>, (int)smem));
  LaunchScope scope(static_cast<cudaStream_t>(stream), KC_EIGSH);
  lanczos_laplacian_kernel<4, 1, EIG_THREADS><<<grid, EIG_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(p);
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}

extern "C" int dss_eigsh_laplacian(const float* Wmat, const float* degree, int ldw, int B, int N, int K, int lapnorm,
                                   float tol, int max_steps, float* evals, float* evecs, int* info, float* resid,
                                   void* ws, size_t ws_bytes, dss_stream_t stream) {
  return eigsh_launch(Wmat, degree, ldw, B, N, K, lapnorm ? 0 : 1, tol, max_steps, evals, evecs, info, resid, ws, ws_bytes,
                      stream);
}

extern "C" int dss_eigsh_topk(const float* Amat, int lda, int B, int N, int K, float tol, int max_steps, float* evals,
                              float* evecs, int* info, float* resid, void* ws, size_t ws_bytes, dss_stream_t stream) {
  return eigsh_launch(Amat, nullptr, lda, B, N, K, 2, tol, max_steps, evals, evecs, info, resid, ws, ws_bytes, stream);
}
