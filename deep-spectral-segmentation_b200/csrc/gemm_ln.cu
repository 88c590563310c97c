// LayerNorm fused into an A-stationary tcgen05 GEMM for the K = 384 layers of ViT-S (qkv and fc1):
//     out[M, N] (f16) = epilogue( LayerNorm(x[M, 384]; gamma, beta, eps) @ Wt[N, 384]^T + bias )
// The stand-alone LayerNorm kernel (7.5 % of the step in round 1: 6 bytes of HBM traffic per element and 23 launches)
// disappears: the CTA's own warps read the fp32 residual stream, normalise it and write the fp16 A operand straight
// into shared memory in the layout tcgen05.mma reads (K-major rows of 128 bytes, 128 B swizzle -- what a TMA box
// {64 x f16, 128 rows} would have written). The 128 x 384 panel (96 KB) then stays put while the weight tiles of ALL
// n-tiles stream past it through a TMA ring, so per 16-deep UMMA step the ring refill moves BN x 32 bytes instead of
// (128 + BN) x 32: the shared-memory bandwidth bound of the plain kernel (DESIGN.md section 3) is relaxed as well.
//
// One CTA per SM, CTAs in clusters of two that walk the same n-tiles for two vertically adjacent 128-row blocks; each
// CTA fetches half of every weight tile and multicasts it into both (as gemm.cu does).
//   warp 0        TMA producer of the weight ring
//   warp 1        TMEM allocation + tcgen05.mma issue (two accumulators: tile i+1's MMAs overlap tile i's epilogue)
//   warps 4..19   epilogue (as gemm.cu: TMEM -> +bias (-> GELU) -> fp16 -> swizzled staging box -> TMA store)
//   warps 20..27  LayerNorm producers. Row statistics of the NEXT 128-row block are computed while the current block's
//                 MMAs run (x is read once from HBM; the second read below hits the L2); then, slab by slab (64
//                 columns), as soon as the last n-tile's MMAs have released slab k of the panel ("a_free[k]"), the
//                 rows are re-read, normalised and written: the panel turnover overlaps the tail of the previous block.
#include <math.h>

#include "common.cuh"

namespace dss {

int make_tmap_f16(CUtensorMap* tm, const void* ptr, int rows, int cols, int box_rows);
int make_tmap_out(CUtensorMap* tm, const void* ptr, int rows, int cols, int is_f32);

constexpr int LG_BM = 128, LG_K = 384, LG_SLABS = LG_K / 64, LG_SLAB_BYTES = LG_BM * 128;
constexpr int LG_EPI_WARPS = 16, LG_LN_WARPS = 8;
constexpr int LG_THREADS = (4 + LG_EPI_WARPS + LG_LN_WARPS) * 32;
constexpr int LG_BOX_BYTES = LG_BM * 128;

// (Measured and dropped: storing the fp16 rows straight from registers with 256-bit st.global and spending the 32 KB of
// staging on a fifth weight stage -- qkv 3.67 -> 4.68 ms, fc1 5.37 -> 5.50 ms per 296 images.)
template <int BN> struct LnCfg {
  static constexpr int A_BYTES = LG_SLABS * LG_SLAB_BYTES;          // 96 KB
  static constexpr int B_STAGE = BN * 128;                          // BN rows x 64 f16
  static constexpr int STAGES = BN == 128 ? 6 : 4;                  // 96 KB of weight tiles in flight either way
  static constexpr int NACC = 512 / BN;                             // TMEM accumulator stages: 2 x 192 or 4 x 128 columns
  static constexpr int STAGING = 2 * LG_BOX_BYTES;                  // one 128 x 128 B output box per epilogue group
  static constexpr int VEC_BYTES = 2 * 2 * LG_BM * 4;               // mean[2][128], rstd[2][128]
  static constexpr int NBARS = 2 * STAGES + 2 * NACC + 2 * LG_SLABS;
  static constexpr int SMEM = A_BYTES + STAGES * B_STAGE + STAGING + VEC_BYTES + NBARS * 8 + 16;
  static constexpr int TMEM_COLS = 512;
  static_assert(SMEM <= 232448, "shared memory budget");
  static_assert((B_STAGE / 2) % 1024 == 0, "half tiles must keep the 1024 B swizzle-atom alignment");
};

struct LnParams {
  const float* x;        // [M, 384] fp32 residual stream (read only)
  const float* gamma;    // [384]
  const float* beta;     // [384]
  const float* bias;     // [N]
  float eps;
  int M, N;
};

// Work items of one cluster: full rounds over the row blocks with every n-tile, then ONE tail item in which the
// remaining row blocks (fewer than clusters) are split by n-tile ranges over all clusters: with whole blocks only, 296
// images (2084 row blocks) gave 6 of 74 clusters a 15th block while 68 idled for a block's worth of time (6.5 % of
// the kernel).
struct LnItem { int c, nt0, nt1; };
__device__ __forceinline__ bool ln_item(int i, int cid, int ncl, int units, int tiles_n, LnItem& it) {
  const int rounds = units / ncl, rem = units - rounds * ncl;
  if (i < rounds) { it.c = cid + i * ncl; it.nt0 = 0; it.nt1 = tiles_n; return true; }
  if (i > rounds || rem == 0) return false;
  int seg = ncl / rem;                       // clusters available per remaining block
  if (seg > tiles_n) seg = tiles_n;
  if (seg < 1) seg = 1;
  const int blk = cid / seg, part = cid - blk * seg;
  if (blk >= rem) return false;
  it.c = rounds * ncl + blk;
  it.nt0 = (tiles_n * part) / seg;
  it.nt1 = (tiles_n * (part + 1)) / seg;
  return it.nt1 > it.nt0;
}

// CL = CTAs per cluster: 2 = the pair shares every weight tile by TMA multicast (each CTA loads half), 1 = every CTA
// loads its own weight tiles (no coupling between CTAs). The library launches CL = 2 (DESIGN.md section 9).
template <bool GELU, int BN, int CL>
__global__ void __launch_bounds__(LG_THREADS, 1)
gemm_ln_f16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC, int pairs,
                           LnParams p) {
  using Cfg = LnCfg<BN>;
  constexpr int STAGES = Cfg::STAGES, B_STAGE = Cfg::B_STAGE, NACC = Cfg::NACC;
  constexpr int NT_BOX = BN / 64;   // 64-column output boxes per tile
  extern __shared__ __align__(1024) uint8_t lg_smem_raw[];
  const uint32_t base = smem_u32(lg_smem_raw);
  if ((base & 1023u) != 0) __trap();   // the 128 B swizzle pattern is a function of address bits [7,10)
  uint8_t* gbase = lg_smem_raw;
  const uint32_t sA = base, sB = base + Cfg::A_BYTES, sStage = sB + STAGES * B_STAGE;
  float* s_mean = reinterpret_cast<float*>(gbase + Cfg::A_BYTES + STAGES * B_STAGE + Cfg::STAGING);   // [2][128]
  float* s_rstd = s_mean + 2 * LG_BM;                                                                  // [2][128]
  const uint32_t bar_base = sStage + Cfg::STAGING + Cfg::VEC_BYTES;
  auto b_full = [&](int s) { return bar_base + 8u * s; };
  auto b_empty = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull = [&](int i) { return bar_base + 8u * (2 * STAGES + i); };
  auto tempty = [&](int i) { return bar_base + 8u * (2 * STAGES + NACC + i); };
  auto a_full = [&](int k) { return bar_base + 8u * (2 * STAGES + 2 * NACC + k); };
  auto a_free = [&](int k) { return bar_base + 8u * (2 * STAGES + 2 * NACC + LG_SLABS + k); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * Cfg::NBARS;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(
      gbase + Cfg::A_BYTES + STAGES * B_STAGE + Cfg::STAGING + Cfg::VEC_BYTES + 8 * Cfg::NBARS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = CL == 2 ? (int)cluster_ctarank() : 0;
  const int cid = blockIdx.x / CL, ncl = gridDim.x / CL;
  const int tiles_n = p.N / BN;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(b_full(s), 1);
      mbar_init(b_empty(s), CL);  // released by the MMA warps of both CTAs (each multicasts into the other's ring)
    }
    for (int i = 0; i < NACC; ++i) {
      mbar_init(tfull(i), 1);
      mbar_init(tempty(i), LG_EPI_WARPS);
    }
    for (int k = 0; k < LG_SLABS; ++k) {
      mbar_init(a_full(k), LG_LN_WARPS);
      mbar_init(a_free(k), 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_addr, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0) {
      // ---- weight ring producer: (block pair, n-tile, k-slab) in lock step with the peer CTA
      const uint32_t uB = __shfl_sync(0xffffffffu, sB, 0);
      int s = 0;
      uint32_t ph = 0;
      LnItem it;
      for (int i = 0; ln_item(i, cid, ncl, pairs, tiles_n, it); ++i) {
        for (int nt = it.nt0; nt < it.nt1; ++nt) {
          for (int k = 0; k < LG_SLABS; ++k) {
            mbar_wait(b_empty(s), ph ^ 1u);
            if (elect_one()) {
              mbar_arrive_expect_tx(b_full(s), B_STAGE);
              if constexpr (CL == 2) {
                tma_load_2d_mc(uB + s * B_STAGE + rank * (B_STAGE / 2), &tmB, b_full(s), k * 64, nt * BN + rank * (BN / 2),
                               (uint16_t)0x3);
              } else {
                tma_load_2d(uB + s * B_STAGE, &tmB, b_full(s), k * 64, nt * BN);
                tma_load_2d(uB + s * B_STAGE + B_STAGE / 2, &tmB, b_full(s), k * 64, nt * BN + BN / 2);
              }
            }
            __syncwarp();
            if (++s == STAGES) { s = 0; ph ^= 1u; }
          }
        }
      }
    } else if (warp == 1) {
      // ---- MMA issuer
      constexpr uint32_t idesc = umma_idesc_f16(LG_BM, BN);
      const uint32_t uA = __shfl_sync(0xffffffffu, sA, 0), uB = __shfl_sync(0xffffffffu, sB, 0);
      const uint32_t utmem = __shfl_sync(0xffffffffu, tmem_base, 0);
      int s = 0, lt = 0, li = 0;
      uint32_t ph = 0;
      LnItem it;
      for (; ln_item(li, cid, ncl, pairs, tiles_n, it); ++li) {
        for (int nt = it.nt0; nt < it.nt1; ++nt, ++lt) {
          const int buf = lt % NACC;
          mbar_wait(tempty(buf), ((lt / NACC) & 1) ^ 1u);
          tc_fence_after();
          const uint32_t acc = utmem + buf * BN;
          for (int k = 0; k < LG_SLABS; ++k) {
            if (nt == it.nt0) mbar_wait(a_full(k), li & 1);   // slab k of this block's normalised panel is in place
            mbar_wait(b_full(s), ph);
            tc_fence_after();
            const uint64_t adesc = umma_desc_sw128(uA + k * LG_SLAB_BYTES);
            const uint64_t bdesc = umma_desc_sw128(uB + s * B_STAGE);
            if (elect_one()) {
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)
                umma_f16_ss(acc, adesc + 2u * kk, bdesc + 2u * kk, idesc, (k | kk) != 0 ? 1u : 0u);
              if constexpr (CL == 2) umma_commit_mc(b_empty(s), (uint16_t)0x3);
              else umma_commit(b_empty(s));
              if (nt == it.nt1 - 1) umma_commit(a_free(k));   // last reader of slab k: the next block may overwrite it
            }
            __syncwarp();
            if (++s == STAGES) { s = 0; ph ^= 1u; }
          }
          if (elect_one()) umma_commit(tfull(buf));
          __syncwarp();
        }
      }
    }
  } else if (warp < 4 + LG_EPI_WARPS) {
    {
      // ---- epilogue: two independent groups of 8 warps, each owning every other 64-column output box (own staging
      // buffer, own named barrier): while one group sits in a barrier or waits for its TMA store the other computes.
      // Inside a thread the box is a stream of four 8-column chunks, software pipelined: the tcgen05.ld and the bias
      // loads of chunk j + 1 are issued before the arithmetic of chunk j, and those of the NEXT box's first chunk before
      // this box's staging barriers (ncu: with load -> wait -> compute per box, 30 % of the epilogue's time was the
      // exposed latency of those loads, and the epilogue, not the tensor core, set the pace).
      static_assert(NT_BOX >= 2, "every tile needs a box for each of the two epilogue groups");
      const int ew = warp - 4;
      const int q = warp & 3, h = (ew >> 2) & 1, grp = ew >> 3;   // TMEM lane quadrant, 32-column half of the box, group
      const int row = q * 32 + lane;
      constexpr int W = 8, NCH = 32 / W;                          // columns per chunk, chunks per thread and box
      const bool issuer = ((ew & 7) == 0) && (lane == 0);
      const uint32_t sbuf = sStage + grp * LG_BOX_BYTES;
      const uint32_t srow = sbuf + row * 128;
      const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);

      // this group's boxes in order: (item i, n-tile nt, box b); lt counts tiles. Box number lt NT_BOX + b over ALL boxes
      // decides the owner: its parity is the group.
      LnItem it;
      int i = 0, nt = 0, b = -1, lt = -1;
      bool valid = ln_item(0, cid, ncl, pairs, tiles_n, it);
      if (valid) nt = it.nt0 - 1, b = NT_BOX - 1;
      auto advance = [&]() {   // -> the next box that belongs to this group (valid = false at the end)
        while (valid) {
          if (++b == NT_BOX) {
            b = 0;
            ++lt;
            if (++nt == it.nt1) {
              valid = ln_item(++i, cid, ncl, pairs, tiles_n, it);
              if (!valid) return;
              nt = it.nt0;
            }
          }
          if (((lt * NT_BOX + b) & 1) == grp) return;
        }
      };
      uint32_t ra[W], rb[W];
      float ba[W], bb[W];
      auto issue = [&](int j, uint32_t (&r)[W], float (&bs)[W]) {   // loads of chunk j of the current box
        tmem_ld_32x8(tlane + (lt % NACC) * BN + b * 64 + h * 32 + j * W, r);
        const float4* bp = reinterpret_cast<const float4*>(p.bias + nt * BN + b * 64 + h * 32 + j * W);
        const float4 b0 = __ldg(bp), b1 = __ldg(bp + 1);
        bs[0] = b0.x; bs[1] = b0.y; bs[2] = b0.z; bs[3] = b0.w; bs[4] = b1.x; bs[5] = b1.y; bs[6] = b1.z; bs[7] = b1.w;
      };
      auto wait_tile = [&]() {   // first box of this group in the tile: wait until the tile's accumulator is complete
        if (b == ((grp ^ (lt * NT_BOX)) & 1)) {
          mbar_wait(tfull(lt % NACC), (lt / NACC) & 1);
          tc_fence_after();
        }
      };
      advance();
      if (valid) { wait_tile(); issue(0, ra, ba); }
      while (valid) {
        const int m0 = (CL * it.c + rank) * LG_BM, nc = nt * BN + b * 64, buf = lt % NACC;
        // is this the group's last box of the tile? (boxes b' > b of this tile with this group's parity)
        bool last_own = true;
#pragma unroll
        for (int b2 = 1; b2 < NT_BOX; ++b2)
          if (b + b2 < NT_BOX && ((b2 & 1) == 0)) last_own = false;
        uint32_t pk[16];   // 32 columns of this row as 16 packed half2
#pragma unroll
        for (int j = 0; j < NCH; ++j) {
          tmem_ld_wait();   // chunk j has landed (the only tcgen05.ld in flight)
          if (j + 1 < NCH) {
            if (j & 1) issue(j + 1, ra, ba); else issue(j + 1, rb, bb);
          } else if (last_own) {   // the accumulator is in registers: the MMA warp may reuse this TMEM buffer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty(buf));
          }
#pragma unroll
          for (int e = 0; e < W; e += 2) {
            const uint32_t a0 = (j & 1) ? rb[e] : ra[e], a1 = (j & 1) ? rb[e + 1] : ra[e + 1];
            const float c0 = (j & 1) ? bb[e] : ba[e], c1 = (j & 1) ? bb[e + 1] : ba[e + 1];
            float x0, x1;
            unpack_f32x2(add_f32x2(pack_f32x2(__uint_as_float(a0), __uint_as_float(a1)), pack_f32x2(c0, c1)), x0, x1);
            if constexpr (GELU) gelu_erf_x2(x0, x1, x0, x1);
            pk[j * (W / 2) + (e >> 1)] = pack_half2(x0, x1);
          }
        }
        // next box of this group: start its first chunk now, so that the loads overlap the staging of this box
        const int st_m0 = m0, st_nc = nc;
        advance();
        if (valid) { wait_tile(); issue(0, ra, ba); }
        if (issuer) tma_store_wait_read<0>();   // this group's previous store has finished reading the buffer
        if (grp == 0) { __syncwarp(); asm volatile("bar.sync 1, 256;" ::: "memory"); }
        else { __syncwarp(); asm volatile("bar.sync 2, 256;" ::: "memory"); }
#pragma unroll
        for (int i4 = 0; i4 < 4; ++i4) {
          const int j16 = h * 4 + i4;   // 16-byte chunk of the 128-byte row, XOR-swizzled with the row (SW128)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + ((j16 ^ (row & 7)) << 4)), "r"(pk[i4 * 4 + 0]),
                       "r"(pk[i4 * 4 + 1]), "r"(pk[i4 * 4 + 2]), "r"(pk[i4 * 4 + 3])
                       : "memory");
        }
        fence_proxy_async_smem();
        if (grp == 0) { __syncwarp(); asm volatile("bar.sync 1, 256;" ::: "memory"); }
        else { __syncwarp(); asm volatile("bar.sync 2, 256;" ::: "memory"); }
        if (issuer) {
          if (st_m0 < p.M) tma_store_2d(&tmC, sbuf, st_nc, st_m0);   // rows >= M are clipped by the tensor map
          tma_store_commit();
        }
      }
      if (issuer) tma_store_wait_all<0>();
    }
  } else {
    // ---- LayerNorm producers: warp w owns rows [16 w, 16 w + 16) of the block. They get the registers the service
    // warps gave up: 4 rows x 3 float4 per lane in flight in the statistics pass (the first, HBM, read of x) -- with 2
    // rows in flight the 8 producer warps could not pull a 196 KB block in less time than its MMAs take
    asm volatile("setmaxnreg.inc.sync.aligned.u32 88;");
    const int w = warp - 4 - LG_EPI_WARPS;
    auto stats = [&](int m0, int par) {
      // two-pass mean / variance like torch (and like the stand-alone kernel it replaces), 4 rows at a time
#pragma unroll 1
      for (int rr = 0; rr < 16; rr += 4) {
        float4 v[4][3];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m0 + w * 16 + rr + i;
          const float4* xr = reinterpret_cast<const float4*>(p.x + (long long)(m < p.M ? m : 0) * LG_K);
#pragma unroll
          for (int j = 0; j < 3; ++j) v[i][j] = m < p.M ? xr[lane + 32 * j] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float s = 0.f;
#pragma unroll
          for (int j = 0; j < 3; ++j) s += (v[i][j].x + v[i][j].y) + (v[i][j].z + v[i][j].w);
          const float mean = warp_sum(s) * (1.0f / LG_K);
          float qv = 0.f;
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            const float a = v[i][j].x - mean, b = v[i][j].y - mean, c = v[i][j].z - mean, e = v[i][j].w - mean;
            qv += (a * a + b * b) + (c * c + e * e);
          }
          const float rstd = rsqrtf(warp_sum(qv) * (1.0f / LG_K) + p.eps);
          if (lane == 0) {
            s_mean[par * LG_BM + w * 16 + rr + i] = mean;
            s_rstd[par * LG_BM + w * 16 + rr + i] = rstd;
          }
        }
      }
      __syncwarp();
    };
    auto write_panel = [&](int m0, int par, int li) {
      // slab k = columns [64 k, 64 k + 64): per instruction the warp covers two rows x 256 contiguous bytes. The loads
      // of slab k + 1 (second read of x: L2) are issued before slab k is normalised, so the L2 latency of the six
      // slabs overlaps the arithmetic instead of adding up (the producers' latency chain per block was longer than
      // the six n-tiles of the qkv layer take on the tensor cores)
      const int c4 = lane & 15, rsel = lane >> 4;
      auto load_slab = [&](int k, float4 (&xv)[8]) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int m = m0 + w * 16 + 2 * i + rsel;
          xv[i] = m < p.M ? __ldg(reinterpret_cast<const float4*>(p.x + (long long)m * LG_K + k * 64) + c4)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      auto put_slab = [&](int k, const float4 (&xv)[8]) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(p.gamma + k * 64 + c4 * 4));   // 3 KB, L1 resident
        const float4 bt = __ldg(reinterpret_cast<const float4*>(p.beta + k * 64 + c4 * 4));
        // normalise BEFORE waiting for the slab: what remains on the critical path between "the previous block's MMAs
        // have read slab k" and "slab k of this block is in place" is 8 shared-memory stores, the proxy fence and the
        // arrive (the MMA warp spent 29 % of its time waiting here when the arithmetic came after the wait)
        uint32_t lo[8], hi[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = w * 16 + 2 * i + rsel;
          const float mean = s_mean[par * LG_BM + r], rstd = s_rstd[par * LG_BM + r];
          lo[i] = pack_half2((xv[i].x - mean) * rstd * g.x + bt.x, (xv[i].y - mean) * rstd * g.y + bt.y);
          hi[i] = pack_half2((xv[i].z - mean) * rstd * g.z + bt.z, (xv[i].w - mean) * rstd * g.w + bt.w);
        }
        if (li > 0) mbar_wait(a_free(k), (li - 1) & 1);   // the previous block's MMAs have read slab k
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = w * 16 + 2 * i + rsel;
          // 8 bytes at column 4 c4 of row r: 16-byte chunk c4 / 2 (XOR-swizzled with the row), half c4 & 1
          const uint32_t addr = sA + k * LG_SLAB_BYTES + r * 128 + ((((c4 >> 1) ^ (r & 7))) << 4) + ((c4 & 1) << 3);
          asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(lo[i]), "r"(hi[i]) : "memory");
        }
        fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full(k));
      };
      float4 xa[8], xb[8];
      load_slab(0, xa);
#pragma unroll
      for (int k = 0; k < LG_SLABS; k += 2) {
        load_slab(k + 1, xb);
        put_slab(k, xa);
        if (k + 2 < LG_SLABS) load_slab(k + 2, xa);
        put_slab(k + 1, xb);
      }
    };
    LnItem it, nx;
    bool have = ln_item(0, cid, ncl, pairs, tiles_n, it);
    if (have) stats((CL * it.c + rank) * LG_BM, 0);
    for (int li = 0; have; ++li) {
      write_panel((CL * it.c + rank) * LG_BM, li & 1, li);
      have = ln_item(li + 1, cid, ncl, pairs, tiles_n, nx);
      if (have) stats((CL * nx.c + rank) * LG_BM, (li + 1) & 1);   // next block: overlaps this block's MMAs
      it = nx;
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

template <bool GELU, int BN>
static int launch_ln(const CUtensorMap& tmB, const CUtensorMap& tmC, const LnParams& p, cudaStream_t st, int kclass) {
  using Cfg = LnCfg<BN>;
  constexpr int CL = 2;
  DSS_CHECK_CUDA(allow_dynamic_smem(gemm_ln_f16_tcgen05_kernel<GELU, BN, CL>, Cfg::SMEM));
  const int units = cdiv(cdiv(p.M, LG_BM), CL);   // row blocks (CL = 1) or pairs of row blocks (CL = 2)
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  const int clusters = units < sms / CL ? units : sms / CL;
  LaunchScope scope(st, kclass);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CL * clusters);
  cfg.blockDim = dim3(LG_THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DSS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_ln_f16_tcgen05_kernel<GELU, BN, CL>, tmB, tmC, units, p));
  DSS_CHECK_CUDA(cudaGetLastError());
  return DSS_OK;
}

// tile width of the fused kernel for an N-column layer (0: not supported)
int gemm_ln_tile_n(int N) {
  return N % 192 == 0 ? 192 : (N % 128 == 0 ? 128 : 0);
}

// tmB: weights [N, 384] f16 with box rows gemm_ln_tile_n(N) / 2; tmC: output [M, N] f16 (make_tmap_out)
int gemm_ln_f16_tc(const CUtensorMap& tmB, const CUtensorMap& tmC, const float* x, const float* gamma, const float* beta,
                   const float* bias, int M, int N, float eps, bool gelu, cudaStream_t st, int kclass) {
  DSS_REQUIRE(x && gamma && beta && bias, "gemm_ln: null pointer");
  DSS_REQUIRE(M > 0 && N > 0, "gemm_ln: empty problem");
  const int bn = gemm_ln_tile_n(N);
  DSS_REQUIRE(bn != 0, "gemm_ln: N = %d is not a multiple of 128", N);
  LnParams p{x, gamma, beta, bias, eps, M, N};
  if (bn == 192) return gelu ? launch_ln<true, 192>(tmB, tmC, p, st, kclass) : launch_ln<false, 192>(tmB, tmC, p, st, kclass);
  return gelu ? launch_ln<true, 128>(tmB, tmC, p, st, kclass) : launch_ln<false, 128>(tmB, tmC, p, st, kclass);
}

}  // namespace dss

using namespace dss;

extern "C" int dss_op_gemm_ln_f16(const float* x, const float* gamma, const float* beta, const void* Wt, const float* bias,
                                  void* out, int M, int N, int K, float eps, int gelu, dss_stream_t stream) {
  DSS_REQUIRE(K == LG_K, "gemm_ln: the fused LayerNorm GEMM is built for K = %d (ViT-S), got %d", LG_K, K);
  DSS_REQUIRE(Wt && out, "gemm_ln: null pointer");
  const int bn = gemm_ln_tile_n(N);
  DSS_REQUIRE(bn != 0, "gemm_ln: N = %d is not a multiple of 128", N);
  CUtensorMap tmB, tmC;
  int rc;
  if ((rc = make_tmap_f16(&tmB, Wt, N, K, bn / 2))) return rc;
  if ((rc = make_tmap_out(&tmC, out, M, N, 0))) return rc;
  return gemm_ln_f16_tc(tmB, tmC, x, gamma, beta, bias, M, N, eps, gelu != 0, static_cast<cudaStream_t>(stream), KC_GEMM_OTHER);
}
