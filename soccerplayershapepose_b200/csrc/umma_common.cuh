// tcgen05 / TMA / mbarrier PTX wrappers and descriptors shared by the tensor-core kernels (blend_umma.cu,
// fused_fwd.cu).
#pragma once

#include <cuda.h>

#include "skin_common.cuh"

namespace b200smpl {

constexpr int BM = 128;
constexpr int BK = 64;                 // bf16 elements = 128 bytes = one swizzle row
constexpr int UMMA_K = 16;
constexpr int GEMM_THREADS = 192;

// backward operands: A = dvp chunks [S/128][n/8][128][8] (plain pointers, one 16 KB bulk copy per stage
// straight into the no-swizzle core-matrix layout), B = Wb rows through a 128-byte-swizzle tensor map.
// The lo halves are read only by the bf16x3 split (fp32 modes).
struct GemmOps {
  const __nv_bfloat16* dvp_hi;
  const __nv_bfloat16* dvp_lo;
  CUtensorMap wb_hi, wb_lo;
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// one lane of a converged warp: lets the whole warp run the (warp-uniform) role loops so that descriptors and
// barrier addresses live in uniform registers, with only the async instruction itself predicated
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// the same two copies with an L2 eviction-priority hint (createpolicy): a stream that is read once must not push
// the small operand every cluster re-reads out of L2
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(void* smem_dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_u32(smem_dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// 32 lanes x 32 columns of fp32 accumulators -> 32 registers per thread (thread = TMEM lane)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128-byte swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// start>>4 [0,14) | LBO>>4 [16,30) = 1 (unused for swizzled K-major) | SBO>>4 [32,46) = 1024 B
// between 8-row groups | version [46,48) = 1 | layout [61,64) = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
         (2ull << 61);
}

// K-major, no-swizzle descriptor: core matrix = 8 rows x 16 bytes, contiguous (128 B); LBO = byte distance
// between core matrices adjacent along K, SBO = between core matrices adjacent along M/N
__device__ __forceinline__ uint64_t make_nosw_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
         (1ull << 46);
}

// cute::UMMA::InstrDescriptor: c_format F32 [4,6)=1, a/b format BF16 [7,10)=[10,13)=1, K-major both,
// n_dim = N>>3 at [17,23), m_dim = M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] . B[smem]^T, bf16 x bf16 -> fp32, issued by the leader CTA for the pair
__device__ __forceinline__ void umma_bf16_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void remote_arrive(uint64_t* local_bar, uint32_t cta) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local_bar)), "r"(cta));
  // relaxed: the payload was written by the TMA (async proxy) and is consumed by the tensor core (async proxy);
  // a cluster-scope release here costs a full membar per stage and serialises the pipeline
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

// work list of the body-stationary forward kernels: cluster c = body-tile pair bp[c], model-row tiles [w0[c], w1[c])
constexpr int BS_MAX_WORK = 160;
struct BsWork {
  uint16_t bp[BS_MAX_WORK], w0[BS_MAX_WORK], w1[BS_MAX_WORK];
};
// host helpers defined in blend_umma.cu
int build_bs_work(int bp_total, int wtp_total, int tpcs, BsWork& work);
// bf16 matrix [rows][pitch] (K contiguous), visible extent k_extent x rows, box 64 x box_rows, 128B swizzle
int make_map(CUtensorMap* map, const void* base, int k_extent, int rows, int pitch_elems, int box_rows);

}  // namespace b200smpl
