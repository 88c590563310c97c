// out = epilogue(A[M,K] * Wt[N,K]^T + bias) with fp16 operands, fp32 accumulation in Tensor Memory.
//
// Persistent kernel, one CTA per SM, 128x128 output tiles handed out round-robin (n fastest, so CTAs that run
// together share the A rows in L2 and the whole weight matrix stays L2-resident):
//   warp 0      : TMA producer   (cp.async.bulk.tensor 2D, 128B swizzle, 64-wide K slabs); the 4-stage ring keeps
//                 running across tile boundaries, so loads for the next tile are in flight during the epilogue
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer (UMMA 128x128x16, kind::f16) into one of TWO
//                 128-column accumulators, so the MMAs of tile i+1 overlap the epilogue of tile i
//   warps 2..9  : epilogue, two groups of 4 warps (one per TMEM lane quarter), each group owns 64 columns:
//                 tcgen05.ld 32 lanes x 32 columns -> +bias / exact-erf GELU -> fp32 staging chunk in smem ->
//                 row-contiguous (coalesced) global reads of the residual and writes of the result
// CTAs run as CLUSTERS OF TWO that work on vertically adjacent tiles (same n, m and m+1): each CTA fetches half of
// the weight tile and TMA-multicasts it into both CTAs' shared memory, which cuts the L2 -> SM operand traffic (the
// bound of this kernel) by 25-33 %. The slot-free signal (tcgen05.commit) is multicast to both CTAs as well.
// Both operands are K-major, which is the native layout of activations [rows, features] and of torch Linear
// weights [out, in]; no transposes anywhere.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

namespace dss {

constexpr int BM = 128, BK = 64, UMMA_K = 16;   // BK: one 128-byte swizzle atom of fp16 (one TMA box / 4 UMMAs)
constexpr int A_ATOM_BYTES = BM * BK * 2;
// swizzle atoms (64-deep K slabs) per pipeline stage. 128-wide tiles: 2 (128-deep stages halve the MMA warp's
// per-FLOP wait/elect/commit overhead: +12 % measured); 256-wide tiles: 1 (their UMMAs are already twice as long and
// only 2 x 96 KB stages would fit, which hides less load latency than 4 x 48 KB: 790 vs 828 TFLOP/s measured).
constexpr int slabs_per_stage(int bn) { return bn == 128 ? 2 : 1; }
constexpr int EPI_WARPS = 16;            // 4 TMEM lane quarters x 4 column slices
constexpr int GEMM_THREADS = 64 + EPI_WARPS * 32;
constexpr int MANUAL_EPI_WARPS = 8;      // the row-remapping / affinity epilogues use the first 8 epilogue warps
constexpr int STG_LD = 36;               // manual path staging chunk: 128 rows x 32 cols fp32, row pitch 36
constexpr int STG_BYTES = BM * STG_LD * 4;
constexpr int BOX_BYTES = BM * 128;      // TMA-store path staging box: 128 rows x 128 bytes (swizzled)

// epilogues whose output rows are the GEMM rows: written with TMA (the row-remapping ones keep the manual path)
constexpr int EPI_AFFINITY_F32 = 100;    // internal epilogue id (not in the public enum): batched patch-affinity tile
__host__ __device__ constexpr bool epi_uses_tma_store(int epi) {
  return epi == DSS_EPI_BIAS_F16 || epi == DSS_EPI_BIAS_GELU_F16 || epi == DSS_EPI_BIAS_RESID_F32 ||
         epi == DSS_EPI_BIAS_F32 || epi == EPI_AFFINITY_F32;
}
constexpr int default_stages(int bn, bool tma) { return tma ? (bn == 128 ? 3 : 4) : 2; }
// Shared-memory bandwidth is what bounds the kernel (DESIGN.md section 3): wide tiles and a deep ring are what matter.
// CG = 1: one CTA per output tile, the pair shares the weight tile by TMA multicast (each CTA still holds all of it).
// CG = 2: tcgen05.mma.cta_group::2, each CTA holds only ITS half of the weight tile, which halves the B operand traffic
// per FLOP; the smaller stages buy a deeper ring. Used for the long-K residual GEMM (fc2), see launch_tc.
template <int BN, bool TMA_OUT, int ST = default_stages(BN, TMA_OUT), int CG = 1> struct TileCfg {
  static constexpr int KS = slabs_per_stage(BN);
  static constexpr int A_TILE_BYTES = KS * A_ATOM_BYTES;
  static constexpr int B_ATOM_BYTES = BN * BK * 2 / CG;   // CG = 2: BN/2 rows per CTA
  static constexpr int B_TILE_BYTES = KS * B_ATOM_BYTES;
  static constexpr int STAGE_BYTES = A_TILE_BYTES + B_TILE_BYTES;   // [A atom 0 | A atom 1 | B atom 0 | B atom 1]
  static constexpr int STAGING_BYTES = TMA_OUT ? 2 * BOX_BYTES : 4 * STG_BYTES;
  static constexpr int MAX_STAGES = (232448 - 1024 - 1024 - 256 - STAGING_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = CG == 1 ? ST : (MAX_STAGES > 8 ? 8 : MAX_STAGES);
  static constexpr int TMEM_COLS = BN == 128 ? 256 : 512;   // two fp32 accumulators, power-of-two allocation
  // ring | staging | barriers | alignment slack
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + 256 + 1024;
};


struct EpiParams {
  void* out;
  const float* bias;
  const float* aux;
  int ldo;
  int rin, rout;
  // batched mode (gridDim.z = images): operand rows of image z start at z * batch_rows
  int batch_rows;
  // affinity epilogue
  const unsigned int* img_max;  // [images] float bits of max(W) per image
  const unsigned int* img_absmax;  // [images] float bits of max|f| when the features were pre-scaled by 2^-e (else null)
  const uint8_t* counts;        // [images, M, M] colour-KNN counts or null
  float lambda;
  int threshold;                // bit 0: relu threshold, bit 1: do not divide by max(W)
  int perm_blocks;              // B operand K-slab permutation for the split-fp16 Gram product (0 = none)
  // symmetric (affinity) mode: only tiles on or above the diagonal are computed; each strictly-upper tile is also
  // stored transposed, and per-tile row / column sums go to deg_part [images, 2 * 4 * tiles, ld_part] (degree fusion)
  int tri;
  float* deg_part;
  int ld_part;
};

// Row of the output buffer that GEMM row m maps to (or -1: skip).
template <int EPI>
__device__ __forceinline__ long long out_row(int m, const EpiParams& p) {
  if constexpr (EPI == DSS_EPI_PATCH_F32) {
    return (long long)(m / p.rin) * p.rout + (m % p.rin) + 1;
  } else if constexpr (EPI == DSS_EPI_DROPCLS_F32) {
    const int t = m % p.rin;
    return t == 0 ? -1 : (long long)(m / p.rin) * p.rout + t - 1;
  } else {
    return m;
  }
}

// Applies the epilogue to 32 consecutive columns [n, n+32) of one row and stores them.
// ---- coalesced epilogue, second phase: one warp owns one output row of the tile at a time, lane l owns columns
// n..n+3 (n = n0 + 4*l), so every global access of a warp is one contiguous 512 B (fp32) / 256 B (fp16) segment.
template <int EPI>
__device__ __forceinline__ void store_row4(float4 v, int m, int n, const EpiParams& p) {
  const long long r = out_row<EPI>(m, p);
  if (r < 0) return;
  if constexpr (EPI == DSS_EPI_BIAS_F16 || EPI == DSS_EPI_BIAS_GELU_F16) {
    uint2 q;
    q.x = pack_half2(v.x, v.y);
    q.y = pack_half2(v.z, v.w);
    *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.out) + r * p.ldo + n) = q;
  } else {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + r * p.ldo + n) = v;
  }
}

// ---- one thread = one row x 32 columns (used by the CUDA-core checker kernel only)
template <int EPI>
__device__ __forceinline__ void epilogue_store(const float (&v)[32], int m, int n, const EpiParams& p) {
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    float4 x = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    if constexpr (EPI == DSS_EPI_BIAS_GELU_F16) {
      x.x = gelu_erf(x.x); x.y = gelu_erf(x.y); x.z = gelu_erf(x.z); x.w = gelu_erf(x.w);
    }
    if constexpr (EPI == DSS_EPI_BIAS_RESID_F32) {
      const float4 y = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.out) + (long long)m * p.ldo + n + j);
      x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w;
    }
    if constexpr (EPI == DSS_EPI_PATCH_F32) {
      const float4 y = __ldg(reinterpret_cast<const float4*>(p.aux + (long long)((m % p.rin) + 1) * p.ldo + n + j));
      x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w;
    }
    store_row4<EPI>(x, m, n + j, p);
  }
}

struct TileCoord { int m0, n0, z; };
// work item t of a cluster = (image z, pair of vertically adjacent m-tiles, n-tile); CTA `rank` takes tile 2*pair+rank
template <int BN>
__device__ __forceinline__ TileCoord decode_tile(int t, int pairs_m, int tiles_n, int rank, int tri = 0) {
  if (tri) {
    // symmetric output (BN == BM): row pair p only visits n-tiles j >= 2p. Tile (2p+1, 2p) of the odd CTA lies below the
    // diagonal: it is computed (the pair runs in lock step on the shared B tile) but never stored.
    int per_img = 0;
    for (int p = 0; p < pairs_m; ++p) per_img += max(tiles_n - 2 * p, 0);
    const int z = t / per_img;
    int rem = t - z * per_img, p = 0;
    for (; p < pairs_m; ++p) {
      const int cnt = max(tiles_n - 2 * p, 0);
      if (rem < cnt) break;
      rem -= cnt;
    }
    return TileCoord{(2 * p + rank) * BM, (2 * p + rem) * BN, z};
  }
  const int per_img = pairs_m * tiles_n;
  const int z = t / per_img, rem = t - z * per_img;
  return TileCoord{((rem / tiles_n) * 2 + rank) * BM, (rem % tiles_n) * BN, z};
}

template <int EPI, int BN, int ST = default_stages(BN, epi_uses_tma_store(EPI)), int CG = 1>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_f16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                        const __grid_constant__ CUtensorMap tmC, int M, int N, int K, int pairs_m, int tiles_n,
                        int total_items, EpiParams p) {
  using Cfg = TileCfg<BN, epi_uses_tma_store(EPI), ST, CG>;
  constexpr int STAGES = Cfg::STAGES, STAGE_BYTES = Cfg::STAGE_BYTES, TMEM_COLS = Cfg::TMEM_COLS;
  constexpr int KS = Cfg::KS, A_TILE_BYTES = Cfg::A_TILE_BYTES;
  static_assert(CG == 1 || epi_uses_tma_store(EPI), "the CTA-pair MMA path is only wired to the TMA-store epilogues");
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024 B alignment (the swizzle pattern is a function of address bits [7,10))
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - raw);
  float* stage_base = reinterpret_cast<float*>(gbase + STAGES * STAGE_BYTES);
  const uint32_t bar_base = base + STAGES * STAGE_BYTES + Cfg::STAGING_BYTES;
  // barrier block: full[STAGES] | empty[STAGES] | tmem_full[2] | tmem_empty[2] | tmem_ptr(u32)
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int i) { return bar_base + 8u * (2 * STAGES + i); };
  auto tempty_bar = [&](int i) { return bar_base + 8u * (2 * STAGES + 2 + i); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_ptr_gen =
      reinterpret_cast<volatile uint32_t*>(gbase + STAGES * STAGE_BYTES + Cfg::STAGING_BYTES + 8 * (2 * STAGES + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = (K + KS * BK - 1) / (KS * BK);   // pipeline stages per tile (128-deep)
  const int rank = (int)cluster_ctarank();          // 0 / 1 inside the CTA pair
  const int cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if constexpr (epi_uses_tma_store(EPI)) tma_prefetch_desc(&tmC);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      // CG 1: released by the MMA warps of BOTH CTAs (each writes into the other's slot); CG 2: one multicast commit
      mbar_init(empty_bar(s), CG == 1 ? 2 : 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar(i), 1);
      // CG 2: the issuing (even) CTA collects the "accumulator drained" arrivals of both CTAs' epilogue warps
      mbar_init(tempty_bar(i), (epi_uses_tma_store(EPI) ? EPI_WARPS : MANUAL_EPI_WARPS) * CG);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    if constexpr (CG == 1) {
      tmem_alloc(tmem_ptr_addr, TMEM_COLS);
      tmem_relinquish();
    } else {
      tmem_alloc_cg2(tmem_ptr_addr, TMEM_COLS);
      tmem_relinquish_cg2();
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // both CTAs' barriers are initialised before any remote arrive / multicast can reach them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp == 0) {
    // The whole warp runs the loop with warp-uniform values (so addresses / coordinates stay in uniform registers and
    // the TMA issue needs no register-to-uniform "waterfall"); one elected lane issues.
    const uint32_t ubase = __shfl_sync(0xffffffffu, base, 0);
    int s = 0;
    uint32_t ph = 0;   // ring position, carried across tiles (no division in the loop)
    for (int t = cid; t < total_items; t += ncl) {
      const TileCoord tc = decode_tile<BN>(t, pairs_m, tiles_n, rank, p.tri);
      const int row_base = tc.z * p.batch_rows;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(bar_base + 8u * (STAGES + s), ph ^ 1u);
        const uint32_t sa = ubase + s * STAGE_BYTES;
        const uint32_t fb = bar_base + 8u * s;
        int ka[KS], kbB[KS];
#pragma unroll
        for (int a = 0; a < KS; ++a) {
          ka[a] = kb * KS + a;   // 64-deep slab index
          // split-fp16 Gram product: A = [hi | hi/64 | 64 lo], B = [hi | 64 lo | hi/64] are the same array read
          // with the last two groups of K slabs swapped
          kbB[a] = ka[a];
          if (p.perm_blocks > 0 && ka[a] >= p.perm_blocks && ka[a] < 3 * p.perm_blocks)
            kbB[a] = ka[a] < 2 * p.perm_blocks ? ka[a] + p.perm_blocks : ka[a] - p.perm_blocks;
        }
        if (elect_one()) {
          if constexpr (CG == 1) {
            mbar_arrive_expect_tx(fb, STAGE_BYTES);
#pragma unroll
            for (int a = 0; a < KS; ++a) {
              tma_load_2d(sa + a * A_ATOM_BYTES, &tmA, fb, ka[a] * BK, row_base + tc.m0);
              // this CTA's half of the weight slab (box 64 x BN/2 rows), delivered to both CTAs of the pair
              tma_load_2d_mc(sa + A_TILE_BYTES + a * Cfg::B_ATOM_BYTES + rank * (Cfg::B_ATOM_BYTES / 2), &tmB, fb,
                             kbB[a] * BK, row_base + tc.n0 + rank * (BN / 2), (uint16_t)0x3);
            }
          } else {
            // both CTAs' bytes are credited to the even CTA's barrier, which the issuing MMA warp waits on
            if (rank == 0) mbar_arrive_expect_tx(fb, 2 * STAGE_BYTES);
#pragma unroll
            for (int a = 0; a < KS; ++a) {
              tma_load_2d_cg2(sa + a * A_ATOM_BYTES, &tmA, fb, ka[a] * BK, row_base + tc.m0);
              tma_load_2d_cg2(sa + A_TILE_BYTES + a * Cfg::B_ATOM_BYTES, &tmB, fb, kbB[a] * BK,
                              row_base + tc.n0 + rank * (BN / 2));   // only THIS CTA's half of the weight slab
            }
          }
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1 && (CG == 1 || rank == 0)) {
    // MMA issuer: the whole warp waits on the barriers, one elected lane issues. Descriptors are computed from
    // warp-uniform values OUTSIDE the elected region: at 64-128 tensor cycles per UMMA the issue cost matters.
    // (CG 2: only the even CTA issues; one instruction drives both CTAs' tensor cores, M = 256.)
    constexpr uint32_t idesc = umma_idesc_f16(BM * CG, BN);
    const uint32_t ubase = __shfl_sync(0xffffffffu, base, 0);
    const uint32_t utmem = __shfl_sync(0xffffffffu, tmem_base, 0);
    int s = 0, lt = 0;
    uint32_t ph = 0;
    for (int t = cid; t < total_items; t += ncl, ++lt) {
      const int buf = lt & 1;
      const uint32_t aph = (lt >> 1) & 1;
      mbar_wait(tempty_bar(buf), aph ^ 1u);  // the epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t acc = utmem + buf * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(bar_base + 8u * s, ph);
        tc_fence_after();
        const uint32_t sa = ubase + s * STAGE_BYTES;
        // advancing K inside a 128 B swizzle atom = advancing the descriptor's start-address field by 32 B >> 4;
        // the second atom of the stage starts A_ATOM_BYTES / B_ATOM_BYTES further
        const uint64_t adesc = umma_desc_sw128(sa);
        const uint64_t bdesc = umma_desc_sw128(sa + A_TILE_BYTES);
        const uint32_t eb = bar_base + 8u * (STAGES + s);
        if (elect_one()) {
#pragma unroll
          for (int a = 0; a < KS; ++a)
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t ad = adesc + (uint64_t)(a * (A_ATOM_BYTES >> 4) + 2 * k);
              const uint64_t bd = bdesc + (uint64_t)(a * (Cfg::B_ATOM_BYTES >> 4) + 2 * k);
              if constexpr (CG == 1) umma_f16_ss(acc, ad, bd, idesc, (kb | a | k) != 0 ? 1u : 0u);
              else umma_f16_ss_cg2(acc, ad, bd, idesc, (kb | a | k) != 0 ? 1u : 0u);
            }
          // slot free once these MMAs have consumed it (CG 1: in this CTA, arriving in both; CG 2: in both CTAs)
          if constexpr (CG == 1) umma_commit_mc(eb, (uint16_t)0x3);
          else umma_commit_cg2_mc(eb, (uint16_t)0x3);
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
      if (elect_one()) {   // accumulator complete (CG 2: in both CTAs)
        if constexpr (CG == 1) umma_commit(tfull_bar(buf));
        else umma_commit_cg2_mc(tfull_bar(buf), (uint16_t)0x3);
      }
      __syncwarp();
    }
  } else if (warp >= 2) {
    // epilogue: group g owns columns [g*BN/2, (g+1)*BN/2) of the tile; a warp may only touch TMEM lanes [32*(warp%4), +32)
    const int ew = warp - 2;
    const int g = ew >> 2, wq = ew & 3;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    if constexpr (epi_uses_tma_store(EPI)) {
      // ---- All 16 epilogue warps cooperate on one 128-byte-wide output box at a time (32 fp32 or 64 fp16 columns):
      // warp (quarter q, slice sl) moves TMEM lanes [32q, 32q+32) x columns [sl*W, sl*W+W) -> registers -> +bias
      // (-> GELU) -> two 16-byte chunks of the 128 B-swizzled staging box; one thread then issues the TMA store.
      // The residual epilogue uses the TMA *reduce-add* (performed at the L2): x += acc + bias never reads x.
      constexpr bool OUT16 = (EPI == DSS_EPI_BIAS_F16 || EPI == DSS_EPI_BIAS_GELU_F16);
      constexpr int BOXC = OUT16 ? 64 : 32;          // columns per 128-byte-wide store box
      constexpr int W = BOXC / 4;                    // columns per warp slice (16 fp16 / 8 fp32 = 32 bytes)
      constexpr int NBOX = BN / BOXC;
      const int sl = ew >> 2;
      const bool issuer = (ew == 0) && (lane == 0);
      const uint32_t stage_u32 = base + STAGES * STAGE_BYTES;
      int lt = 0, cc = 0;
      [[maybe_unused]] float aff_rowsum = 0.f;       // affinity: this thread's row sum over the tile's columns
      [[maybe_unused]] float aff_mx = 1.f, aff_rmx = 1.f, aff_unscale = 1.f;
      for (int t = cid; t < total_items; t += ncl, ++lt) {
        const TileCoord tc = decode_tile<BN>(t, pairs_m, tiles_n, rank, p.tri);
        const int buf = lt & 1;
        const uint32_t aph = (lt >> 1) & 1;
        mbar_wait(tfull_bar(buf), aph);
        tc_fence_after();
        if constexpr (EPI == EPI_AFFINITY_F32) {
          if (p.tri && tc.m0 > tc.n0) {
            // the odd CTA's tile below the diagonal (computed only to keep the pair in lock step on the shared B tile):
            // nothing is read or stored, the accumulator goes straight back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(buf));
            continue;
          }
        }
#pragma unroll 1
        for (int b = 0; b < NBOX; ++b) {
          const int nc = tc.n0 + b * BOXC;           // first global column of the box
          const bool live = nc < N;
          float bias_r[W];                            // independent of the accumulator: issued before the TMEM wait
#pragma unroll
          for (int j = 0; j < W; j += 4) {
            float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bias != nullptr && live) bv = __ldg(reinterpret_cast<const float4*>(p.bias + nc + sl * W + j));
            bias_r[j] = bv.x; bias_r[j + 1] = bv.y; bias_r[j + 2] = bv.z; bias_r[j + 3] = bv.w;
          }
          uint32_t r[W];
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * BN + b * BOXC + sl * W;
          if constexpr (OUT16) tmem_ld_32x16(taddr, r); else tmem_ld_32x8(taddr, r);
          tmem_ld_wait();
          if (b == NBOX - 1) {  // this warp has read all of its TMEM: hand the accumulator back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if constexpr (CG == 1) mbar_arrive(tempty_bar(buf));
              else mbar_arrive_cluster(tempty_bar(buf), 0);   // the even CTA's MMA warp owns both accumulators' release
            }
          }
          float x[W];
#pragma unroll
          for (int e = 0; e < W; e += 2) {
            unpack_f32x2(add_f32x2(pack_f32x2(__uint_as_float(r[e]), __uint_as_float(r[e + 1])),
                                   pack_f32x2(bias_r[e], bias_r[e + 1])), x[e], x[e + 1]);
            if constexpr (EPI == DSS_EPI_BIAS_GELU_F16) gelu_erf_x2(x[e], x[e + 1], x[e], x[e + 1]);
          }
          if constexpr (EPI == EPI_AFFINITY_F32) {
            // W[z, m, n] = relu(acc) / max (+ lambda * counts); columns >= M (row-pitch padding) are zeros; rows >= M
            // are clipped by the per-image (3D) tensor map
            const int m = tc.m0 + row, n = nc + sl * W;
            if (b == 0) {   // per-tile constants (L2 round trips: not once per box)
              aff_mx = __uint_as_float(__ldg(p.img_max + tc.z));
              aff_rmx = __frcp_rn(aff_mx);
              // un-normalised features were pre-scaled by pre = 2^-ceil(log2 max|f|) (affinity.cu): the scale cancels
              // in W / max(W); when the division is skipped (which_matrix = 'affinity' / 'affinity_svd') it is undone
              aff_unscale = 1.0f;
              if ((p.threshold & 2) && p.img_absmax != nullptr) {
                const float am = __uint_as_float(__ldg(p.img_absmax + tc.z));
                if (am > 0.f) aff_unscale = exp2f(2.0f * ceilf(log2f(am)));
              }
              aff_rowsum = 0.f;
            }
            const float mx = aff_mx, rmx = aff_rmx, unscale = aff_unscale;
            const bool relu = p.threshold & 1, nodiv = p.threshold & 2;
            // y / mx without the compiler's IEEE division subroutine: its range check sends zero and tiny numerators --
            // most of a thresholded affinity -- down a ~100-instruction slow path (ncu: 84 % of this kernel's 617 M warp
            // instructions). mx is the largest Gram diagonal: exactly 1 for most normalised images (nothing to do), else
            // q = y r, one residual correction: q + (y - q mx) r -- the correctly rounded quotient for these operand
            // ranges (0 <= y <= ~mx, mx in the normal range).
            const bool scale = !nodiv && mx != 1.0f;
#pragma unroll
            for (int e = 0; e < W; ++e) {
              float y = x[e];
              if (relu) y = fmaxf(y, 0.f);                  // W * (W > 0)
              if (scale) {                                  // W / W.max()
                const float q0 = y * rmx;
                y = fmaf(fmaf(-q0, mx, y), rmx, q0);
              }
              if (nodiv) y *= unscale;
              x[e] = y;
            }
            // edge boxes only (last tile row / column of the image): the colour term and the bounds are per element
            const bool edge = nc + BOXC > M || tc.m0 + BM > M;   // (uniform)
            const bool rowok = !edge || m < M;
            if (p.counts != nullptr && rowok) {
              const uint8_t* cnt = p.counts + ((long long)tc.z * M + m) * M + n;
#pragma unroll
              for (int e = 0; e < W; ++e)
                if (!edge || n + e < M) x[e] += static_cast<float>(cnt[e]) * p.lambda;   // + W_color * lambda
            }
            if (edge) {
#pragma unroll
              for (int e = 0; e < W; ++e)
                if (n + e >= M) x[e] = 0.f;
            }
            if (p.tri) {
              // ---- symmetric mode. The matrix is exactly symmetric by construction (the same value is written to
              // (m, n) and (n, m)), only tiles on or above the diagonal do any work, and the degree D = W 1 that the
              // eigensolver starts from (extract_utils.py:207-220) is accumulated here instead of by another pass
              // over W: per-thread row sums and per-warp column sums go to fixed partial slots (deterministic order).
              // Tiles strictly above the diagonal: TMA store of the tile + mirrored direct stores. Diagonal tiles: the
              // two halves of the tile come out of differently ordered accumulations (the split-fp16 K groups are
              // swapped between the operands), so only the elements on or above the diagonal are stored -- each to
              // both positions -- and the TMA store is skipped: W[i, j] and W[j, i] are the same bits everywhere.
              // (The odd CTA's below-diagonal tile never gets here.)
              const bool upper = tc.m0 < tc.n0;
              float xm[W];
#pragma unroll
              for (int e = 0; e < W; ++e) {
                xm[e] = rowok ? x[e] : 0.f;
                aff_rowsum += xm[e];
              }
              float* part = p.deg_part + (long long)tc.z * (8 * tiles_n) * p.ld_part;
              float* Wz = reinterpret_cast<float*>(p.out) + (long long)tc.z * M * p.ldo;
              if (b == NBOX - 1 && rowok)   // row partial slot of (column tile j, slice sl)
                part[(long long)((tc.n0 / BN) * 4 + sl) * p.ld_part + m] = aff_rowsum;
              if (!upper) {                 // diagonal tile: direct stores only, no staging / TMA store for this box
                if (rowok) {
                  float* rowp = Wz + (long long)m * p.ldo + n;      // (m, n + e)
                  float* colp = Wz + (long long)n * p.ldo + m;      // (n + e, m)
#pragma unroll
                  for (int e = 0; e < W; ++e) {
                    if (n + e >= m && n + e < p.ldo) rowp[e] = x[e];                          // on / above the diagonal
                    if (n + e > m && n + e < M) colp[(long long)e * p.ldo] = x[e];            // its mirror image
                  }
                }
                continue;
              }
              // mirrored store W[z, n + e, m] = W[z, m, n + e]: lanes hold consecutive m -> 128 B per warp store
              if (!edge || m < p.ldo) {
                float* colp = Wz + (long long)n * p.ldo + m;
#pragma unroll
                for (int e = 0; e < W; ++e)
                  if (!edge || n + e < M) colp[(long long)e * p.ldo] = xm[e];
              }
              // column sums over this warp's 32 rows: segmented butterfly (8 -> 4 -> 2 -> 1 values per lane)
              float c4[4], c2[2], c1;
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float mine = (lane & 16) ? xm[e + 4] : xm[e], theirs = (lane & 16) ? xm[e] : xm[e + 4];
                c4[e] = mine + __shfl_xor_sync(0xffffffffu, theirs, 16);
              }
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const float mine = (lane & 8) ? c4[e + 2] : c4[e], theirs = (lane & 8) ? c4[e] : c4[e + 2];
                c2[e] = mine + __shfl_xor_sync(0xffffffffu, theirs, 8);
              }
              {
                const float mine = (lane & 4) ? c2[1] : c2[0], theirs = (lane & 4) ? c2[0] : c2[1];
                c1 = mine + __shfl_xor_sync(0xffffffffu, theirs, 4);
              }
              c1 += __shfl_xor_sync(0xffffffffu, c1, 2);
              c1 += __shfl_xor_sync(0xffffffffu, c1, 1);
              // lane l now holds the sum of column e = 4 * bit4 + 2 * bit3 + bit2 of l (all four lanes l & 3 agree)
              if ((lane & 3) == 0) {
                const int e = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
                // column partial slot of (row tile i = m0 / BM, lane quarter q); it belongs to matrix row n + e
                part[(long long)(4 * tiles_n + (tc.m0 / BM) * 4 + q) * p.ld_part + n + e] = c1;
              }
            }
          }
          // the staging box is free once the store issued two boxes ago has finished READING it
          if (issuer) tma_store_wait_read<1>();
          __syncwarp();   // named barriers are warp-aligned: reconverge after lane-conditional code
          asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
          const uint32_t sbuf = stage_u32 + (cc & 1) * BOX_BYTES;
          const uint32_t srow = sbuf + row * 128;
#pragma unroll
          for (int h = 0; h < 2; ++h) {   // two 16-byte chunks per thread
            const int j = sl * 2 + h;
            const uint32_t addr = srow + ((j ^ (row & 7)) << 4);
            if constexpr (OUT16) {
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(pack_half2(x[h * 8 + 0], x[h * 8 + 1])),
                           "r"(pack_half2(x[h * 8 + 2], x[h * 8 + 3])), "r"(pack_half2(x[h * 8 + 4], x[h * 8 + 5])),
                           "r"(pack_half2(x[h * 8 + 6], x[h * 8 + 7]))
                           : "memory");
            } else {
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(x[h * 4 + 0]), "f"(x[h * 4 + 1]),
                           "f"(x[h * 4 + 2]), "f"(x[h * 4 + 3])
                           : "memory");
            }
          }
          fence_proxy_async_smem();   // generic-proxy smem writes -> visible to the TMA (async proxy)
          __syncwarp();   // named barriers are warp-aligned: reconverge after lane-conditional code
          asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
          if (issuer) {
            if (live) {
              if constexpr (EPI == DSS_EPI_BIAS_RESID_F32)
                tma_reduce_add_2d(&tmC, sbuf, nc, tc.m0);
              else if constexpr (EPI == EPI_AFFINITY_F32)
                tma_store_3d(&tmC, sbuf, nc, tc.m0, tc.z);
              else
                tma_store_2d(&tmC, sbuf, nc, tc.m0);
            }
            tma_store_commit();
          }
          ++cc;   // (boxes that skip the staging buffers -- diagonal affinity tiles -- do not advance the buffer parity)
        }
      }
      if (issuer) tma_store_wait_all<0>();
    } else if (ew < MANUAL_EPI_WARPS) {
    constexpr int NCHUNK = BN / 64;            // 32-column chunks per group
    int lt = 0, cc = 0;  // cc: running chunk counter -> consecutive chunks always use alternate staging buffers
    for (int t = cid; t < total_items; t += ncl, ++lt) {
      const TileCoord tc = decode_tile<BN>(t, pairs_m, tiles_n, rank, p.tri);
      const int buf = lt & 1;
      const uint32_t aph = (lt >> 1) & 1;
      mbar_wait(tfull_bar(buf), aph);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < NCHUNK; ++c, ++cc) {
        const int col0 = g * (BN / 2) + c * 32;  // first column of this chunk inside the tile
        float* stg = stage_base + (g * 2 + (cc & 1)) * (STG_BYTES / 4);
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * BN + col0, r);
        tmem_ld_wait();
        if (c == NCHUNK - 1) {  // this warp has read all of its TMEM: hand the accumulator back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty_bar(buf));
        }
        const int nc = tc.n0 + col0;           // global column of the chunk
        // Phase 1: +bias (-> GELU) -> staging chunk (thread = row; pitch 36 floats -> conflict-free float4 writes)
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias != nullptr && nc < N) bv = __ldg(reinterpret_cast<const float4*>(p.bias + nc + j));
          float4 v;
          v.x = __uint_as_float(r[j + 0]) + bv.x;
          v.y = __uint_as_float(r[j + 1]) + bv.y;
          v.z = __uint_as_float(r[j + 2]) + bv.z;
          v.w = __uint_as_float(r[j + 3]) + bv.w;
          if constexpr (EPI == DSS_EPI_BIAS_GELU_F16) {
            v.x = gelu_erf(v.x); v.y = gelu_erf(v.y); v.z = gelu_erf(v.z); v.w = gelu_erf(v.w);
          }
          *reinterpret_cast<float4*>(stg + row * STG_LD + j) = v;
        }
        // group-local barrier (ids 1, 2). Double-buffered staging: one barrier per chunk is enough, because a
        // thread reaches the barrier of chunk c only after finishing phase 2 of the previous user of buffer c^1.
        __syncwarp();   // named barriers are warp-aligned: reconverge after lane-conditional code
        asm volatile("bar.sync %0, 128;" ::"r"(2 + g) : "memory");
        // Phase 2: 8 lanes x 16 B cover the 128 B of one row of the chunk, 4 rows per warp instruction
        if (nc < N) {
          const int cl = (lane & 7) * 4;
          float4 v[8], y[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = wq * 32 + i * 4 + (lane >> 3);
            const int m = tc.m0 + rr;
            v[i] = *reinterpret_cast<const float4*>(stg + rr * STG_LD + cl);
            y[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (m < M) {
              if constexpr (EPI == DSS_EPI_BIAS_RESID_F32)
                y[i] = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.out) + (long long)m * p.ldo + nc + cl);
              if constexpr (EPI == DSS_EPI_PATCH_F32)
                y[i] = __ldg(reinterpret_cast<const float4*>(p.aux + (long long)((m % p.rin) + 1) * p.ldo + nc + cl));
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = wq * 32 + i * 4 + (lane >> 3);
            const int m = tc.m0 + rr;
            if (m >= M) continue;
            float4 x = v[i];
            x.x += y[i].x; x.y += y[i].y; x.z += y[i].z; x.w += y[i].w;
            store_row4<EPI>(x, m, nc + cl, p);
          }
        }
      }
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer may still multicast / arrive into this CTA's shared memory until it is done too
  if (warp == 1) {
    if constexpr (CG == 1) tmem_dealloc(tmem_base, TMEM_COLS);
    else tmem_dealloc_cg2(tmem_base, TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// CUDA-core checker with the same epilogues (tests only).
template <int EPI>
__global__ void gemm_f16_simt_kernel(const __half* __restrict__ A, const __half* __restrict__ Wt, int M, int N, int K,
                                     EpiParams p) {
  // one thread = one row x 32 columns
  const int m = blockIdx.y * blockDim.y + threadIdx.y;
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) * 32;
  if (m >= M || n >= N) return;
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = 0.f;
  for (int k = 0; k < K; ++k) {
    const float a = __half2float(A[(size_t)m * K + k]);
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaf(a, __half2float(Wt[(size_t)(n + j) * K + k]), v[j]);
  }
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] += p.bias[n + j];
  epilogue_store<EPI>(v, m, n, p);
}

// ---------------------------------------------------------------------------------------------------------------
// Host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess || !ptr) {
    set_error("cuTensorMapEncodeTiled not available from the CUDA driver");
    return nullptr;
  }
  fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  return fn;
}

// Tile width used for an N-column GEMM (B operand = weights [N, K]): 256 if it divides N, else 128.
int gemm_tile_n(int N) {
  // widest tile that divides N: operand bytes per FLOP (shared-memory bandwidth, the binding resource) fall with BN
  return N % 256 == 0 ? 256 : (N % 192 == 0 ? 192 : 128);
}

// 2D fp16 row-major [rows, cols] tensor, box = 64 columns x box_rows rows, 128 B swizzle, zero fill out of bounds.
int make_tmap_f16(CUtensorMap* tm, const void* ptr, int rows, int cols, int box_rows) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return DSS_ERR_CUDA;
  DSS_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA operand must be 16-byte aligned");
  DSS_REQUIRE(cols % 8 == 0, "TMA operand row pitch must be a multiple of 16 bytes (cols=%d)", cols);
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)cols * 2};
  DSS_REQUIRE(box_rows > 0 && box_rows <= 256, "TMA box rows must be in [1, 256]");
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%d cols=%d)", (int)r, rows, cols);
    return DSS_ERR_CUDA;
  }
  return DSS_OK;
}

// Output tensor map for the TMA-store epilogues: row-major [rows, cols] of fp16 (box 64 x 128) or fp32 (box 32 x 128),
// i.e. 128-byte-wide boxes with the 128 B swizzle.
int make_tmap_out(CUtensorMap* tm, const void* ptr, int rows, int cols, int is_f32) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return DSS_ERR_CUDA;
  DSS_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA output must be 16-byte aligned");
  const int esz = is_f32 ? 4 : 2;
  DSS_REQUIRE((cols * esz) % 16 == 0, "TMA output row pitch must be a multiple of 16 bytes (cols=%d)", cols);
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)cols * esz};
  cuuint32_t box[2] = {(cuuint32_t)(is_f32 ? 32 : 64), (cuuint32_t)BM};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                   const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (output) failed with CUresult %d (rows=%d cols=%d)", (int)r, rows, cols);
    return DSS_ERR_CUDA;
  }
  return DSS_OK;
}

// Per-image fp32 output [images, rows, ld] for the affinity epilogue: 3D map, box 32 columns x 128 rows x 1 image
int make_tmap_out3d_f32(CUtensorMap* tm, const void* ptr, int images, int rows, int ld) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return DSS_ERR_CUDA;
  DSS_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && ld % 4 == 0, "affinity output must be 16-byte aligned / pitched");
  cuuint64_t gdim[3] = {(cuuint64_t)ld, (cuuint64_t)rows, (cuuint64_t)images};
  cuuint64_t gstride[2] = {(cuuint64_t)ld * 4, (cuuint64_t)rows * ld * 4};
  cuuint32_t box[3] = {32, (cuuint32_t)BM, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (3D output) failed with CUresult %d", (int)r);
    return DSS_ERR_CUDA;
  }
  return DSS_OK;
}

// 3D fp16 output [images, rows, cols] written in 128-row x 64-column boxes (128 B swizzle); rows past `rows` of an image
// are clipped by the TMA unit, so a partial last tile never spills into the next image.
int make_tmap_out3d_f16(CUtensorMap* tm, const void* ptr, int images, int rows, int cols) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return DSS_ERR_CUDA;
  DSS_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && cols % 64 == 0, "fp16 tile output must be 16-byte aligned, cols %% 64 == 0");
  cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)images};
  cuuint64_t gstride[2] = {(cuuint64_t)cols * 2, (cuuint64_t)rows * cols * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)BM, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (3D fp16 output) failed with CUresult %d", (int)r);
    return DSS_ERR_CUDA;
  }
  return DSS_OK;
}

template <int EPI, int BN, int ST = default_stages(BN, epi_uses_tma_store(EPI)), int CG = 1>
static int launch_tc_bn(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmC, int M, int N, int K,
                        const EpiParams& p, cudaStream_t st, int kclass, int batch) {
  using Cfg = TileCfg<BN, epi_uses_tma_store(EPI), ST, CG>;
  DSS_CHECK_CUDA(allow_dynamic_smem(gemm_f16_tcgen05_kernel<EPI, BN, ST, CG>, Cfg::SMEM_BYTES));
  const int pairs_m = cdiv(cdiv(M, BM), 2), tiles_n = cdiv(N, BN);
  int per_img = pairs_m * tiles_n;
  if (p.tri) {   // symmetric output: row pair p visits the n-tiles j >= 2p only (see decode_tile)
    per_img = 0;
    for (int q = 0; q < pairs_m; ++q) per_img += tiles_n - 2 * q > 0 ? tiles_n - 2 * q : 0;
  }
  const int total = per_img * batch;   // work items of a CTA pair
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  const int clusters = total < sms / 2 ? total : sms / 2;
  if (epi_uses_tma_store(EPI) && tmC == nullptr) {
    set_error("gemm: this epilogue needs an output tensor map");
    return DSS_ERR_BAD_ARG;
  }
  LaunchScope scope(st, kclass);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * clusters);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DSS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_f16_tcgen05_kernel<EPI, BN, ST, CG>, tmA, tmB, tmC ? *tmC : tmA, M, N, K,
                                    pairs_m, tiles_n, total, p));
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}

// bn = tile width the B tensor map was built for (its TMA box has bn rows)
template <int EPI>
static int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmC, int M, int N, int K,
                     const EpiParams& p, cudaStream_t st, int kclass, int bn, int batch = 1) {
  // CTA-pair MMA (tcgen05.mma.cta_group::2: each CTA holds only its half of the weight tile), measured on the
  // 296-image step against the multicast form: fc2 (K = 1536) 1028 vs 931 TFLOP/s, but qkv / fc1 / proj (K = 384)
  // 844 / 720 / 411 vs 1019 / 760 / 439 -- the pair's shared accumulator-drain handshake costs more than the halved
  // operand traffic saves when a tile has only six K slabs. Hence: the long-K residual GEMM only.
  if constexpr (EPI == DSS_EPI_BIAS_RESID_F32) {
    if (K >= 1024) {
      constexpr int D = 0;   // stage count is derived from the shared-memory budget for CG = 2
      switch (bn) {
        case 128: return launch_tc_bn<EPI, 128, D, 2>(tmA, tmB, tmC, M, N, K, p, st, kclass, batch);
        case 192: return launch_tc_bn<EPI, 192, D, 2>(tmA, tmB, tmC, M, N, K, p, st, kclass, batch);
        case 256: return launch_tc_bn<EPI, 256, D, 2>(tmA, tmB, tmC, M, N, K, p, st, kclass, batch);
      }
    }
  }
  switch (bn) {
    case 128: return launch_tc_bn<EPI, 128>(tmA, tmB, tmC, M, N, K, p, st, kclass, batch);
    case 192:
      if constexpr (epi_uses_tma_store(EPI)) return launch_tc_bn<EPI, 192>(tmA, tmB, tmC, M, N, K, p, st, kclass, batch);
      break;
    case 256:
      if constexpr (epi_uses_tma_store(EPI)) return launch_tc_bn<EPI, 256>(tmA, tmB, tmC, M, N, K, p, st, kclass, batch);
      break;
  }
  set_error("gemm: unsupported tile width %d", bn);
  return DSS_ERR_BAD_ARG;
}

static int check_gemm_args(int M, int N, int K, int epi, const float* bias, const void* out, const float* aux,
                           int rin, int rout) {
  DSS_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: empty problem M=%d N=%d K=%d", M, N, K);
  DSS_REQUIRE(N % 32 == 0 && K % 8 == 0, "gemm: need N %% 32 == 0 and K %% 8 == 0 (N=%d K=%d)", N, K);
  DSS_REQUIRE(bias && out, "gemm: null bias/out");
  if (epi == DSS_EPI_PATCH_F32 || epi == DSS_EPI_DROPCLS_F32) {
    DSS_REQUIRE(rin > 0 && rout > 0 && M % rin == 0, "gemm: bad row remap rin=%d rout=%d M=%d", rin, rout, M);
    if (epi == DSS_EPI_PATCH_F32) DSS_REQUIRE(aux != nullptr, "gemm: patch epilogue needs aux (pos embed)");
  }
  return DSS_OK;
}

// Launch with pre-built tensor maps (used by the ViT forward, which caches them).
int gemm_f16_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmC, const float* bias, void* out,
                int M, int N, int K, int epi, const float* aux, int rin, int rout, cudaStream_t st, int kclass, int bn) {
  int rc = check_gemm_args(M, N, K, epi, bias, out, aux, rin, rout);
  if (rc) return rc;
  EpiParams p{out, bias, aux, N, rin, rout, 0, nullptr, nullptr, nullptr, 0.f, 0, 0, 0, nullptr, 0};
  switch (epi) {
    case DSS_EPI_BIAS_F16: return launch_tc<DSS_EPI_BIAS_F16>(tmA, tmB, tmC, M, N, K, p, st, kclass, bn);
    case DSS_EPI_BIAS_GELU_F16: return launch_tc<DSS_EPI_BIAS_GELU_F16>(tmA, tmB, tmC, M, N, K, p, st, kclass, bn);
    case DSS_EPI_BIAS_RESID_F32: return launch_tc<DSS_EPI_BIAS_RESID_F32>(tmA, tmB, tmC, M, N, K, p, st, kclass, bn);
    case DSS_EPI_BIAS_F32: return launch_tc<DSS_EPI_BIAS_F32>(tmA, tmB, tmC, M, N, K, p, st, kclass, bn);
    case DSS_EPI_PATCH_F32: return launch_tc<DSS_EPI_PATCH_F32>(tmA, tmB, tmC, M, N, K, p, st, kclass, bn);
    case DSS_EPI_DROPCLS_F32: return launch_tc<DSS_EPI_DROPCLS_F32>(tmA, tmB, tmC, M, N, K, p, st, kclass, bn);
  }
  set_error("gemm: unknown epilogue %d", epi);
  return DSS_ERR_BAD_ARG;
}

// Batched Gram product for the affinity build: per image z, W[z] = epilogue(S[z] S'[z]^T) with S = split-fp16 rows
// [images*Nimg, 3d] (see affinity.cu). N output columns cover the padded pitch ldw.
int affinity_gemm_tc(const CUtensorMap& tmS, const CUtensorMap& tmS_half, int images, int Nimg, int d, float* Wout, int ldw,
                     const unsigned int* img_max, const unsigned int* img_absmax, const uint8_t* counts, float lambda,
                     int threshold, float* deg_part, int ld_part, cudaStream_t st) {
  EpiParams p{Wout, nullptr, nullptr, ldw, 0, 0, Nimg, img_max, img_absmax, counts, lambda, threshold, d / BK,
              1, deg_part, ld_part};
  DSS_REQUIRE(d % BK == 0, "affinity: feature dim must be a multiple of %d for the tensor-core path (got %d)", BK, d);
  DSS_REQUIRE(deg_part != nullptr && ld_part >= cdiv(ldw, 128) * 128, "affinity: bad degree partial buffer");
  CUtensorMap tmW;
  int rc = make_tmap_out3d_f32(&tmW, Wout, images, Nimg, ldw);
  if (rc) return rc;
  return launch_tc<EPI_AFFINITY_F32>(tmS, tmS_half, &tmW, Nimg, ldw, 3 * d, p, st, KC_AFFINITY, 128, images);
}

template <int EPI>
static int launch_simt(const void* A, const void* Wt, int M, int N, int K, const EpiParams& p, cudaStream_t st) {
  dim3 block(4, 32);
  dim3 grid(cdiv(N / 32, 4), cdiv(M, 32));
  LaunchScope scope(st, KC_MISC);
  gemm_f16_simt_kernel<EPI><<<grid, block, 0, st>>>(reinterpret_cast<const __half*>(A),
                                                    reinterpret_cast<const __half*>(Wt), M, N, K, p);
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}

}  // namespace dss

using namespace dss;

extern "C" int dss_op_gemm_f16(const void* A, const void* Wt, const float* bias, void* out, int M, int N, int K,
                               int epilogue, const float* aux, int rin, int rout, dss_stream_t stream) {
  int rc = check_gemm_args(M, N, K, epilogue, bias, out, aux, rin, rout);
  if (rc) return rc;
  DSS_REQUIRE(A && Wt, "gemm: null operand");
  CUtensorMap tmA, tmB;
  const int bn = epi_uses_tma_store(epilogue) ? gemm_tile_n(N) : 128;   // row-remapping epilogues: 128-wide only
  if ((rc = make_tmap_f16(&tmA, A, M, K, BM))) return rc;
  if ((rc = make_tmap_f16(&tmB, Wt, N, K, bn / 2))) return rc;   // each CTA of a pair loads (and multicasts) half a tile
  CUtensorMap tmC;
  const bool tma_out = epi_uses_tma_store(epilogue);
  if (tma_out) {
    const int f32 = (epilogue == DSS_EPI_BIAS_RESID_F32 || epilogue == DSS_EPI_BIAS_F32) ? 1 : 0;
    if ((rc = make_tmap_out(&tmC, out, M, N, f32))) return rc;
  }
  return gemm_f16_tc(tmA, tmB, tma_out ? &tmC : nullptr, bias, out, M, N, K, epilogue, aux, rin, rout,
                     static_cast<cudaStream_t>(stream), KC_GEMM_OTHER, bn);
}

extern "C" int dss_op_gemm_f16_simt(const void* A, const void* Wt, const float* bias, void* out, int M, int N, int K,
                                    int epilogue, const float* aux, int rin, int rout, dss_stream_t stream) {
  int rc = check_gemm_args(M, N, K, epilogue, bias, out, aux, rin, rout);
  if (rc) return rc;
  DSS_REQUIRE(A && Wt, "gemm: null operand");
  EpiParams p{out, bias, aux, N, rin, rout, 0, nullptr, nullptr, nullptr, 0.f, 0, 0, 0, nullptr, 0};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (epilogue) {
    case DSS_EPI_BIAS_F16: return launch_simt<DSS_EPI_BIAS_F16>(A, Wt, M, N, K, p, st);
    case DSS_EPI_BIAS_GELU_F16: return launch_simt<DSS_EPI_BIAS_GELU_F16>(A, Wt, M, N, K, p, st);
    case DSS_EPI_BIAS_RESID_F32: return launch_simt<DSS_EPI_BIAS_RESID_F32>(A, Wt, M, N, K, p, st);
    case DSS_EPI_BIAS_F32: return launch_simt<DSS_EPI_BIAS_F32>(A, Wt, M, N, K, p, st);
    case DSS_EPI_PATCH_F32: return launch_simt<DSS_EPI_PATCH_F32>(A, Wt, M, N, K, p, st);
    case DSS_EPI_DROPCLS_F32: return launch_simt<DSS_EPI_DROPCLS_F32>(A, Wt, M, N, K, p, st);
  }
  set_error("gemm: unknown epilogue %d", epilogue);
  return DSS_ERR_BAD_ARG;
}
