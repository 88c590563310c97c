// Multi-head attention (head dim 64) on the 5th-generation tensor cores: O = softmax(Q K^T / 8) V.
//
// Persistent kernel, one CTA per SM. A work item is one (image, head, PAIR of 128-query tiles); the CTA walks its items
// with every ring / barrier phase carried across item boundaries, so the loads and the first score tile of the next
// item overlap the tail of the current one.
//   warp 0      TMA producer: Q tiles (double buffered per query tile) and K_j / V_j tiles straight out of the packed
//               qkv activations [B*T, 3d] (box 64 x 128, 128 B swizzle) through a 3-stage ring shared by both
//               query tiles
//   warps 1, 2  tcgen05.mma issuers of query tile A / B (warp 1 also owns the TMEM allocation); per key tile j:
//                 S_g = Q_g K_j^T   (UMMA 128 x kc x 16, x4, both operands K-major)               -> TMEM S_g
//                 O_g += P_g V_j    (UMMA 128 x 64 x 16, x kc/16, A = P from TMEM, B = V MN-major) -> TMEM O_g
//               kc = 128 except in the last key tile, where it is the number of existing keys rounded up to 16
//               (T = 901: 16 instead of 128).
//   warps 4..7  softmax of query tile A, warps 8..11 of query tile B: ONE thread per query row (tcgen05.ld 32x32b), no
//               cross-thread exchange. The 128 scores of the row are read from TMEM once and S_g is released at once
//               (the next score tile is computed while this one is exponentiated); P = 2^(s c - m c) (MUFU.EX2) goes
//               back to TMEM as packed fp16 pairs (tcgen05.st) and is the A operand of the PV MMA: P never touches
//               shared memory, whose bandwidth the K / V / Q operand reads need.
//               The output accumulates in TMEM across key tiles. The reference maximum m is only raised (and O, l
//               rescaled, by the owning thread through tcgen05.ld/st) when a tile's row maximum exceeds it by more than
//               2^8 -- softmax is shift invariant and fp16 P / fp32 sums have the headroom -- so in the steady state the
//               softmax warps never touch O until the epilogue.
// The two softmax groups run out of phase (B's first tile is held back until A is half way through its first tile), so one
// group's MUFU-bound exp phase overlaps the other's TMEM loads / maxima / fences. The kernel is bound by the MUFU pipe
// (128 x 128 exp2 per tile at 16 per clock per SM), not by the tensor pipe.
#include <math.h>

#include "common.cuh"

namespace dss {

int make_tmap_f16(CUtensorMap* tm, const void* ptr, int rows, int cols, int box_rows);
int make_tmap_out3d_f16(CUtensorMap* tm, const void* ptr, int images, int rows, int cols);

// one MUFU.EX2 (2 ulp), flushes denormal results to zero; exp2f would add range checks and fix-ups per element
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// warp group 0: TMA warp, two MMA warps, one idle warp; warp groups 1 / 2: softmax of query tile A / B.
// Register budget (setmaxnreg, per warp group): 168 at launch -> 56 for group 0, 224 for the softmax groups
// (4 x 32 x (56 + 224 + 224) = 64512 <= 65536).
// exp2 of two values on the FMA pipe (Cody-Waite split + degree-4 minimax polynomial on [-0.5, 0.5], max relative error
// 2.7e-6 -- far below the fp16 rounding of P): a share of the exponentials is taken off the MUFU unit, which at 16 per
// clock per SM is the busiest unit of this kernel. Inputs are <= ~8; anything below -125 (masked keys) clamps to 2^-125,
// which packs to an fp16 zero.
__device__ __forceinline__ void ex2_poly_x2(float x0, float x1, float& p0, float& p1) {
  const uint64_t x = pack_f32x2(fmaxf(x0, -125.0f), fmaxf(x1, -125.0f));
  const uint64_t xf = add_f32x2(x, pack_f32x2(12582912.0f, 12582912.0f));          // integer part in the low mantissa bits
  const uint64_t n = add_f32x2(xf, pack_f32x2(-12582912.0f, -12582912.0f));
  const uint64_t f = fma_f32x2(n, pack_f32x2(-1.0f, -1.0f), x);                    // x - round(x) in [-0.5, 0.5]
  uint64_t p = fma_f32x2(pack_f32x2(0.009570100344717503f, 0.009570100344717503f), f,
                         pack_f32x2(0.05591786280274391f, 0.05591786280274391f));
  p = fma_f32x2(p, f, pack_f32x2(0.240247443318367f, 0.240247443318367f));
  p = fma_f32x2(p, f, pack_f32x2(0.6931217908859253f, 0.6931217908859253f));
  p = fma_f32x2(p, f, pack_f32x2(0.9999992847442627f, 0.9999992847442627f));
  float pa, pb, xa, xb;
  unpack_f32x2(p, pa, pb);
  unpack_f32x2(xf, xa, xb);
  p0 = __int_as_float(__float_as_int(pa) + (__float_as_int(xa) << 23));             // p * 2^n through the exponent field
  p1 = __int_as_float(__float_as_int(pb) + (__float_as_int(xb) << 23));
}
constexpr int FA_POLY_OF_4 = 1;   // of every 4 consecutive key pairs, this many go through ex2_poly_x2

constexpr int FA_BM = 128, FA_BN = 128, FA_D = 64, FA_THREADS = 384;
constexpr int FA_TILE = FA_BM * FA_D * 2;             // 16 KB: one [128 x 64] fp16 tile
constexpr int FA_KV_STAGES = 3;
// Q[g][2] | K ring | V ring | output staging[g] = 12 tiles = 192 KB (P never touches shared memory)
constexpr int FA_SMEM = FA_TILE * (4 + 2 * FA_KV_STAGES + 2);
constexpr int FA_TMEM_COLS = 512;
constexpr int FA_S_COL = 0, FA_O_COL = 256, FA_P_COL = 384;   // S_A, S_B at 0 / 128; O_A, O_B at 256 / 320; P_A, P_B at 384 / 448
constexpr float FA_RESCALE_LOG2 = 8.0f;       // raise the reference maximum only when exceeded by more than 2^8
constexpr int FA_NBARS = 8 + 2 * FA_KV_STAGES + 10;

__global__ void __launch_bounds__(FA_THREADS, 1)
attention_tcgen05_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmO, int T, int heads,
                         int nq2, int total_items) {
  extern __shared__ __align__(1024) uint8_t fa_smem[];
  __shared__ __align__(8) uint64_t bars[FA_NBARS];
  __shared__ uint32_t tmem_ptr_s;

  const uint32_t base = smem_u32(fa_smem);
  if ((base & 1023u) != 0) __trap();  // the 128 B swizzle pattern is a function of address bits [7,10)
  const uint32_t sQ = base, sK = base + 4 * FA_TILE, sV = sK + FA_KV_STAGES * FA_TILE, sO = sV + FA_KV_STAGES * FA_TILE;
  const uint32_t bar0 = smem_u32(bars);
  auto q_full = [&](int g, int i) { return bar0 + 8u * (g * 2 + i); };
  auto q_empty = [&](int g, int i) { return bar0 + 8u * (4 + g * 2 + i); };
  auto kv_full = [&](int s) { return bar0 + 8u * (8 + s); };
  auto kv_empty = [&](int s) { return bar0 + 8u * (8 + FA_KV_STAGES + s); };
  auto s_full = [&](int g) { return bar0 + 8u * (8 + 2 * FA_KV_STAGES + g); };
  auto p_full = [&](int g) { return bar0 + 8u * (10 + 2 * FA_KV_STAGES + g); };
  auto o_full = [&](int g) { return bar0 + 8u * (12 + 2 * FA_KV_STAGES + g); };
  auto s_free = [&](int g) { return bar0 + 8u * (16 + 2 * FA_KV_STAGES + g); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = heads * FA_D;
  const int nt = (T + FA_BN - 1) / FA_BN;
  const int kc_last = (T - (nt - 1) * FA_BN + 15) & ~15;   // key columns of the last tile that are worth computing

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 4; ++i) {
      mbar_init(q_full(i >> 1, i & 1), 1);
      mbar_init(q_empty(i >> 1, i & 1), 1);
    }
    for (int s = 0; s < FA_KV_STAGES; ++s) {
      mbar_init(kv_full(s), 1);
      mbar_init(kv_empty(s), 2);   // one commit per query tile's MMA warp
    }
    for (int g = 0; g < 2; ++g) {
      mbar_init(s_full(g), 1);
      mbar_init(p_full(g), 4);   // one arrival per softmax warp: 128 per-thread arrivals on one barrier serialise
      mbar_init(s_free(g), 4);   // (measured: ~1300 cycles until the phase flips)
      mbar_init(o_full(g), 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(&tmem_ptr_s), FA_TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_ptr_s);

  // Producer and MMA warps run their loops with ALL lanes on warp-uniform values and let one elected lane issue: the
  // smem addresses, coordinates and descriptors then live in uniform registers and each UMMA / TMA issue is a couple
  // of instructions instead of a register-to-uniform "waterfall" loop.
  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  if (warp == 0) {
    const uint32_t uQ = __shfl_sync(0xffffffffu, sQ, 0), uK = __shfl_sync(0xffffffffu, sK, 0),
                   uV = __shfl_sync(0xffffffffu, sV, 0);
    int s = 0;
    uint32_t ph = 0;   // K/V ring position, carried across items
    int qi = 0;        // item counter of this CTA
    for (int w = blockIdx.x; w < total_items; w += gridDim.x, ++qi) {
      // item w -> (image * heads + head, pair of query tiles). The pair index is rotated by the (image, head) index:
      // with the plain w % nq2 a CTA (w = blockIdx + k * 148, 148 % 4 == 0) would get the SAME pair index in every item,
      // and the CTAs that only ever see the light last pair (a 5-row tail tile at T = 901) idle at the end of the
      // kernel while the others are still on full pairs (ncu: 8.5 % of the stall samples on EXIT)
      const int bh = w / nq2, qp = (w % nq2 + bh) % nq2;
      const int h = bh % heads, row0 = (bh / heads) * T;   // first row of this image in the [B*T, 3d] matrix
      const int qb = qi & 1;
      const uint32_t qph = (qi >> 1) & 1;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        mbar_wait(q_empty(g, qb), qph ^ 1u);
        if (elect_one()) {
          mbar_arrive_expect_tx(q_full(g, qb), FA_TILE);
          tma_load_2d(uQ + (g * 2 + qb) * FA_TILE, &tmQKV, q_full(g, qb), h * FA_D, row0 + (2 * qp + g) * FA_BM);
        }
        __syncwarp();
      }
      for (int j = 0; j < nt; ++j) {
        mbar_wait(kv_empty(s), ph ^ 1u);
        if (elect_one()) {
          mbar_arrive_expect_tx(kv_full(s), 2 * FA_TILE);
          tma_load_2d(uK + s * FA_TILE, &tmQKV, kv_full(s), d + h * FA_D, row0 + j * FA_BN);
          tma_load_2d(uV + s * FA_TILE, &tmQKV, kv_full(s), 2 * d + h * FA_D, row0 + j * FA_BN);
        }
        __syncwarp();
        if (++s == FA_KV_STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // one MMA-issuing warp per query tile (a single warp serving both tiles was the bottleneck of the kernel: ~1000
    // cycles per batch of UMMAs, four batches per step). Per tile the events strictly alternate in time
    // (S_g released early in key tile n, P_g published at its end), so plain blocking waits in program order suffice.
    const int g = warp - 1;
    constexpr uint32_t idesc_qk0 = umma_idesc_f16(FA_BM, 0);                    // A, B K-major; N filled in per tile
    constexpr uint32_t idesc_pv = umma_idesc_f16(FA_BM, FA_D) | (1u << 16);     // B (= V) MN-major
    const uint32_t uQ = __shfl_sync(0xffffffffu, sQ, 0) + g * 2 * FA_TILE, uK = __shfl_sync(0xffffffffu, sK, 0),
                   uV = __shfl_sync(0xffffffffu, sV, 0),
                   utmem = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t s_acc = utmem + FA_S_COL + g * FA_BN, o_acc = utmem + FA_O_COL + g * FA_D;
    const uint32_t p_tm = utmem + FA_P_COL + g * (FA_BN / 2);   // P_g: 128 rows x 128 fp16 = 64 columns
    const int my_items = (total_items - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) /
                         static_cast<int>(gridDim.x);
    const int m_total = my_items * nt;   // key-tile steps of this CTA, over all of its items
    int sj = 0, sq = 0, ss = 0;          // cursor of the next score tile: key tile, item, ring stage
    uint32_t sph = 0;
    auto issue_s = [&]() {   // S_g = Q_g K_j^T
      if (sj == 0) mbar_wait(q_full(g, sq & 1), (sq >> 1) & 1);
      mbar_wait(kv_full(ss), sph);
      tc_fence_after();
      const uint64_t qdesc = umma_desc_sw128(uQ + (sq & 1) * FA_TILE);
      const uint64_t kdesc = umma_desc_sw128(uK + ss * FA_TILE);
      const int kc = sj == nt - 1 ? kc_last : FA_BN;
      const uint32_t idesc = idesc_qk0 | (static_cast<uint32_t>(kc >> 3) << 17);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < FA_D / 16; ++k)   // +32 B per 16-wide K step = +2 in the descriptor's address field
          umma_f16_ss(s_acc, qdesc + 2u * k, kdesc + 2u * k, idesc, k != 0 ? 1u : 0u);
        umma_commit(s_full(g));
        if (sj == nt - 1) umma_commit(q_empty(g, sq & 1));   // last score tile of the item: Q_g may be replaced
      }
      __syncwarp();
      if (++sj == nt) { sj = 0; ++sq; }
      if (++ss == FA_KV_STAGES) { ss = 0; sph ^= 1u; }
    };
    if (m_total > 0) issue_s();
    int pj = 0, ps = 0;
    for (int n = 0; n < m_total; ++n) {
      if (n + 1 < m_total) {   // S_g(n+1) as soon as the softmax warps hold S_g(n) in registers
        mbar_wait(s_free(g), n & 1);
        issue_s();
      }
      // O_g (+)= P_g V_j once the softmax warps have published P_g(n) (and rescaled O_g if they had to)
      mbar_wait(p_full(g), n & 1);
      tc_fence_after();
      const int ksteps = (pj == nt - 1 ? kc_last : FA_BN) >> 4;
      const uint64_t vdesc = umma_desc_sw128(uV + ps * FA_TILE);   // +16 key rows = +2048 B = +128
      const bool first = pj == 0;   // first key tile of the item: overwrite
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < FA_BN / 16; ++k)
          if (k < ksteps)
            umma_f16_ts(o_acc, p_tm + 8u * k, vdesc + 128u * k, idesc_pv, (k != 0 || !first) ? 1u : 0u);
        umma_commit(o_full(g));
        umma_commit(kv_empty(ps));   // this query tile is done with K_j / V_j (the ring slot needs both tiles' commits)
      }
      __syncwarp();
      if (++pj == nt) pj = 0;
      if (++ps == FA_KV_STAGES) ps = 0;
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    const int g = (warp - 4) >> 2;        // query tile of the pair
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;          // query row inside the tile
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t s_col = lane_addr + FA_S_COL + g * FA_BN;
    const uint32_t o_col = lane_addr + FA_O_COL + g * FA_D;
    const uint32_t p_col = lane_addr + FA_P_COL + g * (FA_BN / 2);   // this row of P_g (fp16 pairs, 64 columns)
    const float sc = 1.4426950408889634f * 0.125f;  // log2(e) / sqrt(64)
    uint32_t m = 0;   // key-tile step counter of this CTA (all barrier phases derive from it)
    for (int w = blockIdx.x; w < total_items; w += gridDim.x) {
      // item w -> (image * heads + head, pair of query tiles). The pair index is rotated by the (image, head) index:
      // with the plain w % nq2 a CTA (w = blockIdx + k * 148, 148 % 4 == 0) would get the SAME pair index in every item,
      // and the CTAs that only ever see the light last pair (a 5-row tail tile at T = 901) idle at the end of the
      // kernel while the others are still on full pairs (ncu: 8.5 % of the stall samples on EXIT)
      const int bh = w / nq2, qp = (w % nq2 + bh) % nq2;
      const int h = bh % heads;
      const int q0 = (2 * qp + g) * FA_BM;
      const bool dead = q0 >= T;   // odd number of query tiles: nothing to do for B in the last pair
      // a warp whose 32 query rows all lie beyond T (T = 901: three of the four warps of the 8th tile, which has 5 live
      // rows) only keeps the barrier protocol going: its exponentials would occupy the MUFU unit -- the busiest unit of
      // the kernel -- for rows the output tensor map clips anyway
      const bool wdead = dead || q0 + q * 32 >= T;
      float m_ref = -INFINITY, l_run = 0.f;   // reference maximum of the exponent, row sum relative to it
      for (int j = 0; j < nt; ++j, ++m) {
        // tile B starts every item half a key tile behind tile A (A signals from the middle of its first tile): left
        // alone, the two groups drift into lock step within ~10 items and both sit in their MUFU phase together
        if (j == 0 && g == 1) { __syncwarp(); asm volatile("bar.sync 3, 256;" ::: "memory"); }
        mbar_wait(s_full(g), m & 1);
        tc_fence_after();
        if (!wdead) {
          // one key tile, in four chunks of 32 key columns; only the last tile of a row of tiles can be short
          // (kc < 128 columns computed, nvalid <= kc of them real keys)
          const bool tail = j == nt - 1 && (T & (FA_BN - 1)) != 0;
          const int kc = tail ? kc_last : FA_BN;
          const int nvalid = tail ? T - j * FA_BN : FA_BN;
          uint32_t v[128];
          float mxc[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};   // four independent maximum chains
          uint64_t rs2[2] = {0ull, 0ull};                                 // packed partial row sums, two chains
          // chunk c of the tile: (tail mask) -> running maximum of the raw scores -> P = 2^(s*c - m_ref*c) -> row sum
          // -> packed fp16 pairs into TMEM (the A operand of the P V product). The maximum is tracked alongside the
          // exponentials (FMNMX3 on the ALU pipe) instead of in a pass of its own.
          auto chunk = [&](const int c, const float msc, const bool track_max) {
            if (tail) {   // keys beyond T: score -inf -> probability exactly 0
#pragma unroll
              for (int i = c * 32; i < c * 32 + 32; ++i)
                if (i >= nvalid) v[i] = 0xff800000u;
            }
            if (track_max) {
#pragma unroll
              for (int i = c * 32; i < c * 32 + 32; ++i)
                mxc[i & 3] = fmaxf(mxc[i & 3], __uint_as_float(v[i]));
            }
            const uint64_t sc2 = pack_f32x2(sc, sc), nmsc2 = pack_f32x2(-msc, -msc);
            uint32_t pk[16];
#pragma unroll
            for (int e = 0; e < 32; e += 2) {
              const int i = c * 32 + e;
              float x0, x1;
              unpack_f32x2(fma_f32x2(pack_f32x2(__uint_as_float(v[i]), __uint_as_float(v[i + 1])), sc2, nmsc2), x0, x1);
              float p0, p1;
              if (((e >> 1) & 3) < FA_POLY_OF_4) {
                ex2_poly_x2(x0, x1, p0, p1);
              } else {
                p0 = ex2_approx(x0);
                p1 = ex2_approx(x1);
              }
              rs2[(e >> 1) & 1] = add_f32x2(rs2[(e >> 1) & 1], pack_f32x2(p0, p1));
              pk[e >> 1] = pack_half2(p0, p1);
            }
            tmem_st_32x16(p_col + c * 16, pk);
          };
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (c * 32 < kc) tmem_ld_32x32(s_col + c * 32, *reinterpret_cast<uint32_t (*)[32]>(&v[c * 32]));
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(s_free(g));   // S_g is in registers: the next score tile may overwrite it
          if (j == 0) {
            // ---- first key tile of an item: there is no reference yet, so the row maximum comes first
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (c * 32 < kc) {
#pragma unroll
                for (int i = c * 32; i < c * 32 + 32; ++i) {
                  if (tail && i >= nvalid) v[i] = 0xff800000u;
                  mxc[i & 3] = fmaxf(mxc[i & 3], __uint_as_float(v[i]));
                }
              }
            }
            m_ref = fmaxf(fmaxf(mxc[0], mxc[1]), fmaxf(mxc[2], mxc[3]));
            const float msc = m_ref * sc;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (c * 32 < kc) {
                chunk(c, msc, false);
                // release tile B's first key tile when tile A is half way through its first exponentials: the two
                // groups then stay about half a period apart (one in its MUFU phase, the other loading / reducing)
                if (c == 1 && g == 0) { __syncwarp(); asm volatile("bar.arrive 3, 256;" ::: "memory"); }
              }
            }
            if (kc <= 32 && g == 0) { __syncwarp(); asm volatile("bar.arrive 3, 256;" ::: "memory"); }   // (short first tile)
          } else {
            // ---- later key tiles: exponentials are taken relative to the reference maximum of the EARLIER tiles right
            // away (softmax is shift invariant; fp16 P and the fp32 sums have 2^8 of headroom) with the row maximum
            // tracked alongside (FMNMX3, ALU pipe); only if this tile turns out to exceed the reference by more than
            // 2^8 is the reference raised and the tile redone (rare).
            mbar_wait(o_full(g), (m - 1) & 1);   // P_g is single buffered: P_g V_{j-1} must be complete
            tc_fence_after();
            float msc = m_ref * sc;
#pragma unroll
            for (int c = 0; c < 4; ++c)
              if (c * 32 < kc) chunk(c, msc, true);
            const float mx = fmaxf(fmaxf(mxc[0], mxc[1]), fmaxf(mxc[2], mxc[3]));
            const bool raise = (mx - m_ref) * sc > FA_RESCALE_LOG2;
            if (__any_sync(0xffffffffu, raise)) {   // rare: rescale this warp's rows of O_g in TMEM, redo the tile
              const float f = raise ? ex2_approx((m_ref - mx) * sc) : 1.0f;
              tmem_st_wait();
              uint32_t t[32];
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                tmem_ld_32x32(o_col + c * 32, t);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i) t[i] = __float_as_uint(__uint_as_float(t[i]) * f);
                tmem_st_32x32(o_col + c * 32, t);
              }
              tmem_st_wait();
              l_run *= f;
              if (raise) m_ref = mx;
              msc = m_ref * sc;
              rs2[0] = rs2[1] = 0ull;
#pragma unroll
              for (int c = 0; c < 4; ++c)
                if (c * 32 < kc) chunk(c, msc, false);
            }
          }
          float rs, rs_hi;
          unpack_f32x2(add_f32x2(rs2[0], rs2[1]), rs, rs_hi);
          rs += rs_hi;
          l_run += rs;
          tmem_st_wait();
          tc_fence_before();          // order this thread's TMEM accesses before the MMA that accumulates into O_g
          __syncwarp();
          if (lane == 0) mbar_arrive(p_full(g));
        } else {
          // nothing to compute, but keep the protocol: P_g(m) may only be announced once P_g V(m-1) has been issued
          // (the MMA warp probes p_full by parity and must never be lapped by two phases)
          if (j == 0 && g == 0) { __syncwarp(); asm volatile("bar.arrive 3, 256;" ::: "memory"); }   // tile B's start signal (see above)
          if (m > 0) mbar_wait(o_full(g), (m - 1) & 1);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(s_free(g));
            mbar_arrive(p_full(g));
          }
        }
      }
      if (!wdead) {
        mbar_wait(o_full(g), (m - 1) & 1);   // last P V product of this item
        tc_fence_after();
        uint32_t t[FA_D];
        tmem_ld_32x32(o_col, *reinterpret_cast<uint32_t (*)[32]>(&t[0]));
        tmem_ld_32x32(o_col + 32, *reinterpret_cast<uint32_t (*)[32]>(&t[32]));
        tmem_ld_wait();
        tc_fence_before();
        float inv;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(l_run));
        // normalised [128 x 64] fp16 tile -> swizzled staging tile -> one TMA store (rows >= T are clipped by the
        // 3D tensor map). The elected thread first makes sure the previous item's store has finished reading.
        if (q == 0 && lane == 0) tma_store_wait_read<0>();
        __syncwarp();   // named barriers are warp-aligned: reconverge after lane-conditional code
        asm volatile("bar.sync %0, 128;" ::"r"(4 + g) : "memory");
        const uint32_t srow = sO + g * FA_TILE + r * 128;
#pragma unroll
        for (int i = 0; i < FA_D; i += 8) {
          const uint32_t w0 = pack_half2(__uint_as_float(t[i + 0]) * inv, __uint_as_float(t[i + 1]) * inv);
          const uint32_t w1 = pack_half2(__uint_as_float(t[i + 2]) * inv, __uint_as_float(t[i + 3]) * inv);
          const uint32_t w2 = pack_half2(__uint_as_float(t[i + 4]) * inv, __uint_as_float(t[i + 5]) * inv);
          const uint32_t w3 = pack_half2(__uint_as_float(t[i + 6]) * inv, __uint_as_float(t[i + 7]) * inv);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + ((((i >> 3) ^ (r & 7))) << 4)), "r"(w0),
                       "r"(w1), "r"(w2), "r"(w3)
                       : "memory");
        }
        fence_proxy_async_smem();
        __syncwarp();   // named barriers are warp-aligned: reconverge after lane-conditional code
        asm volatile("bar.sync %0, 128;" ::"r"(4 + g) : "memory");
        if (q == 0 && lane == 0) {
          tma_store_3d(&tmO, sO + g * FA_TILE, h * FA_D, q0, bh / heads);
          tma_store_commit();
        }
      } else if (!dead) {
        // rows beyond T inside a live tile (never lane quarter 0): only the two staging-tile barriers of the group
        __syncwarp();   // named barriers are warp-aligned: reconverge after lane-conditional code
        asm volatile("bar.sync %0, 128;" ::"r"(4 + g) : "memory");
        __syncwarp();   // named barriers are warp-aligned: reconverge after lane-conditional code
        asm volatile("bar.sync %0, 128;" ::"r"(4 + g) : "memory");
      }
    }
    if (q == 0 && lane == 0) tma_store_wait_all<0>();   // the staging tile must outlive the last store
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, FA_TMEM_COLS);
}

int launch_attention_tc(const void* qkv, void* out, int B, int T, int heads, cudaStream_t st) {
  DSS_REQUIRE(B > 0 && T > 0 && heads > 0, "attention: empty problem");
  DSS_CHECK_CUDA(allow_dynamic_smem(attention_tcgen05_kernel, FA_SMEM));
  CUtensorMap tm, tmO;
  int rc = make_tmap_f16(&tm, qkv, B * T, 3 * heads * FA_D, FA_BM);
  if (rc) return rc;
  if ((rc = make_tmap_out3d_f16(&tmO, out, B, T, heads * FA_D))) return rc;
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  const int nq2 = cdiv(cdiv(T, FA_BM), 2);   // pairs of 128-query tiles per (image, head)
  const int total = B * heads * nq2;
  const int grid = total < sms ? total : sms;   // persistent: one CTA per SM
  LaunchScope scope(st, KC_ATTENTION);
  attention_tcgen05_kernel<<<grid, FA_THREADS, FA_SMEM, st>>>(tm, tmO, T, heads, nq2, total);
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}

}  // namespace dss

extern "C" int dss_op_attention_tc_f16(const void* qkv, void* out, int B, int T, int heads, dss_stream_t stream) {
  return dss::launch_attention_tc(qkv, out, B, T, heads, static_cast<cudaStream_t>(stream));
}
