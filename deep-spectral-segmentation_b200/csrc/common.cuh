// Shared device/host helpers for libdss_b200 (sm_100a only).
// PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA + TMEM), cp.async, ldmatrix, mma.sync.
#pragma once
#include <cuda.h>  // CUtensorMap (types only; the driver entry point is resolved at run time, no -lcuda)
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dss_b200.h"

#if defined(__CUDA_ARCH__) && !defined(__CUDA_ARCH_FEAT_SM100_ALL)
#error "libdss_b200 is written for sm_100a only: compile with -gencode arch=compute_100a,code=sm_100a"
#endif

namespace dss {

// ---------------------------------------------------------------- host side error plumbing
void set_error(const char* fmt, ...);
const char* last_error();

#define DSS_CHECK_CUDA(expr)                                                                      \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) {                                                                      \
      ::dss::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));     \
      return DSS_ERR_CUDA;                                                                        \
    }                                                                                             \
  } while (0)

#define DSS_REQUIRE(cond, ...)                                                                    \
  do {                                                                                            \
    if (!(cond)) {                                                                                \
      ::dss::set_error(__VA_ARGS__);                                                              \
      return DSS_ERR_BAD_ARG;                                                                     \
    }                                                                                             \
  } while (0)

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int device_sm_count();

// ---------------------------------------------------------------- launch accounting / per-class device timing
enum KernelClass {
  KC_IM2COL = 0, KC_GEMM_PATCH, KC_CLS_ROW, KC_LAYERNORM, KC_GEMM_QKV, KC_ATTENTION, KC_GEMM_PROJ, KC_GEMM_FC1,
  KC_GEMM_FC2, KC_GEMM_KPROJ, KC_GEMM_OTHER, KC_ROWNORM, KC_AFFINITY, KC_KNN, KC_EIGSH, KC_MISC, KC_COUNT
};
// Counts the launch and, when profiling is enabled, brackets it with CUDA events on the launching stream.
struct LaunchScope {
  cudaStream_t st;
  int slot;
  LaunchScope(cudaStream_t stream, int kernel_class);
  ~LaunchScope();
};

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t.reg .b32 R;\n\t"
      "elect.sync R|P, 0xFFFFFFFF;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Spin on try_wait (HW-suspended probe). A bounded spin turns a protocol bug into a trap instead of a hang.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
#ifndef DSS_NO_MBAR_TIMEOUT
  uint32_t spins = 0;
#endif
  while (true) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P1;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
#ifndef DSS_NO_MBAR_TIMEOUT
    if (++spins > (1u << 24)) __trap();
#endif
  }
}

// Non-blocking probe, made warp-uniform by a vote (for event loops that watch several barriers).
__device__ __forceinline__ bool mbar_test_all(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return __all_sync(0xffffffffu, done != 0);
}

// ---- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
// 2D tiled load global -> shared, completion signalled on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// 2D tiled store shared -> global (bulk async-group completion); rows/columns outside the tensor are clipped
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
// 2D tiled reduction global += shared, performed element-wise at the L2 (residual add without reading it back)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* tm, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
// 3D tiled store (box depth 1): used for per-image matrices [B, rows, cols] so that rows are clipped per image
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N bulk groups still READ their shared-memory source (the buffers may then be reused)
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---- thread-block clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 2D tiled load, multicast: the box lands at the same shared-memory offset in every CTA of `cta_mask`, and each
// destination CTA's mbarrier (same offset) receives the complete_tx for the bytes written into that CTA
__device__ __forceinline__ void tma_load_2d_mc(uint32_t smem_dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1,
                                               uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}

// ---- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (fp16/bf16 operands, fp32 accumulate), one CTA.
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand (128 rows x 16 fp16) is read from TMEM -- lane = row, 8 consecutive
// 32-bit columns holding the 16 K-values of the row as packed pairs (what tcgen05.st 32x32b of half2 words writes)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// same, arriving on the mbarrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(cta_mask)
               : "memory");
}
// ---- CTA-pair ("2-SM") forms: one MMA spans the tensor cores of both CTAs of a cluster pair (M = 256: each CTA owns 128
// rows and its own TMEM accumulator; B is split along N between the two CTAs' shared memories). Issued by ONE thread
// of the even CTA; completion is multicast to a barrier at the same offset in both CTAs.
__device__ __forceinline__ void umma_f16_ss_cg2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_cg2_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(cta_mask)
               : "memory");
}
// TMEM allocation for a CTA pair: executed by the same-numbered warp of BOTH CTAs with the same shared-memory offset
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// TMA load whose completion bytes are credited to the mbarrier at the same offset in the EVEN CTA of the pair
// (bit 24 of a shared::cluster address selects the CTA of the pair)
__device__ __forceinline__ void tma_load_2d_cg2(uint32_t smem_dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
// arrive on the mbarrier at this shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(rank)
      : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives lane (base_lane + i), columns c..c+31
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// narrower variants: 32 lanes x 8 / 16 consecutive columns
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM: lane = this thread's row of its warp's lane quarter, 32 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor for a K-major tile stored as rows of 128 bytes with the 128B swizzle
// (exactly what a TMA box {64 x b16, rows} with CU_TENSOR_MAP_SWIZZLE_128B writes): 8-row groups are 1024 B apart.
//   bits [0,14) start>>4 | [16,30) LBO>>4 (=1, unused for swizzled K-major) | [32,46) SBO>>4 (=64)
//   bits [46,48) version=1 (sm_100) | [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  const uint32_t lo = ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16);
  const uint32_t hi = 64u | (1u << 14) | (2u << 29);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
// Instruction descriptor, kind::f16: [4,6) D fmt (1=f32) | [7,10) A fmt (0=f16,1=bf16) | [10,13) B fmt |
// [15] A major (0=K) | [16] B major (0=K) | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// ---- Ampere-style async copy + legacy tensor-core path (used by the attention kernel)
__device__ __forceinline__ void cp_async_16(uint32_t smem_dst, const void* gsrc, bool valid) {
  const int src_bytes = valid ? 16 : 0;  // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_dst), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                                  uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
// D(16x8,f32) += A(16x16,f16,row) * B(16x8,f16,col)
__device__ __forceinline__ void mma_m16n8k16_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

// ---- packed fp32 pairs (sm_100: FFMA2 / FADD2 process two floats per instruction)
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t mul_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// Exact-erf GELU, branch-free:  gelu(x) = x Phi(x) = relu(x) - |x| q(|x|),  q(a) = 0.5 erfc(a / sqrt 2) = 2^P(u),
// u = min(a / sqrt 2, 5), P = degree-4 minimax fit of log2(erfc(u)) - 1 on [0, 5] weighted by the error it causes in
// gelu (|x| q ln 2 dP). Max |gelu error| 6.4e-6 over the whole fp32 range, relative error <= 1e-3 for x >= -3
// (tests/test_cpu_host.py emulates this arithmetic in float32 against torch's float64 GELU); the value is then rounded
// to fp16 (relative 4.9e-4, smallest normal 6.1e-5).
// Cost per element: 7 FMA-pipe lane operations (bias add, scale, 4 Horner steps, final fma -- issued as packed FFMA2),
// one MUFU.EX2 and three ALU-pipe operations (sign, min, max), spread over three pipes. History: Abramowitz-Stegun
// 7.1.26 (round 1: MUFU.RCP + MUFU.EX2 + ~14 scalar FMA-pipe instructions; ncu XU pipe 38 % vs tensor pipe 27 %) ->
// u P(u^2) erf polynomial of degree 8 on the FMA pipe only (14 lane operations: ncu showed the epilogue warps stalled on
// the FMA pipe, 2 500 cycles per 128 x 64 box against 2 300 cycles of MMA per tile; packed FFMA2 with register operands
// issues at the same lane rate as scalar FFMA) -> this form.
#define DSS_GELU_P0 -1.0004795789718628f
#define DSS_GELU_P1 -1.6226296424865723f
#define DSS_GELU_P2 -0.9360293745994568f
#define DSS_GELU_P3 -0.12467514723539352f
#define DSS_GELU_P4 0.015465063974261284f
#define DSS_GELU_CLAMP 5.0f
__device__ __forceinline__ void gelu_erf_x2(float x0, float x1, float& y0, float& y1) {
  const float na0 = __uint_as_float(__float_as_uint(x0) | 0x80000000u);   // -|x|
  const float na1 = __uint_as_float(__float_as_uint(x1) | 0x80000000u);
  const uint64_t na = pack_f32x2(na0, na1);
  float u0, u1;
  unpack_f32x2(mul_f32x2(na, pack_f32x2(-0.70710678118654752440f, -0.70710678118654752440f)), u0, u1);
  u0 = fminf(u0, DSS_GELU_CLAMP);
  u1 = fminf(u1, DSS_GELU_CLAMP);
  const uint64_t u = pack_f32x2(u0, u1);
  uint64_t p = fma_f32x2(pack_f32x2(DSS_GELU_P4, DSS_GELU_P4), u, pack_f32x2(DSS_GELU_P3, DSS_GELU_P3));
  p = fma_f32x2(p, u, pack_f32x2(DSS_GELU_P2, DSS_GELU_P2));
  p = fma_f32x2(p, u, pack_f32x2(DSS_GELU_P1, DSS_GELU_P1));
  p = fma_f32x2(p, u, pack_f32x2(DSS_GELU_P0, DSS_GELU_P0));
  float p0, p1, q0, q1;
  unpack_f32x2(p, p0, p1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(q0) : "f"(p0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(q1) : "f"(p1));
  unpack_f32x2(fma_f32x2(na, pack_f32x2(q0, q1), pack_f32x2(fmaxf(x0, 0.f), fmaxf(x1, 0.f))), y0, y1);
}
__device__ __forceinline__ float gelu_erf(float x) {
  float y0, y1;
  gelu_erf_x2(x, x, y0, y1);
  return y0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

#endif  // __CUDACC__

// Lets `kernel` be launched with up to `bytes` of dynamic shared memory on the current device. The limit is a property
// of the kernel in that device's context, so it is set once per kernel and device (again only to raise it); thread-safe.
cudaError_t allow_dynamic_smem(const void* kernel, int bytes);
template <class Kernel>
inline cudaError_t allow_dynamic_smem(Kernel* kernel, int bytes) {
  return allow_dynamic_smem(reinterpret_cast<const void*>(kernel), bytes);
}

}  // namespace dss
