// Blend-shape contractions on the 5th-gen tensor cores (tcgen05 + TMEM, operands staged by TMA).
//
//   forward : vp[b][n]    = sum_k feat[b][k]  * Wf[n][k]       (SURVEY.md section 8 rows a4 + a7:
//             shape blend + pose-corrective blend + template, all folded into one K axis)
//   backward: dfeat[b][f] = sum_n dvp[b][n]  * Wb[f][n]        (data gradient, split-K over n)
//
// In both the M axis (= TMEM lane = epilogue thread) is the BODY, so the skinning kernels on either
// side (lane = body) exchange data with the GEMMs in layouts where a warp moves 512 contiguous bytes
// per instruction (skin_common.cuh).  bf16 K-major operands; fp32 accuracy comes from the bf16x3
// error-compensated split laid out along K (see FeatLayout in common.cuh), so the tensor pipe only
// ever sees kind::f16 MMAs with fp32 accumulation in TMEM.
//
// Both GEMMs run on CTA pairs (tcgen05 cta_group::2, cluster of 2): M = 256 bodies, 128 per CTA, and each
// CTA holds half of the model operand, which halves the per-SM shared-memory operand traffic that bounds a
// single-CTA tensor-core GEMM of this shape.  CTA = 6 warps: warp 0 TMA producer, warp 1 MMA issuer (+ TMEM
// alloc; only the leader of the pair issues), warps 2-5 epilogue (tcgen05.ld -> registers -> 16-byte global
// stores).  Operand stages are bf16 tiles of 64 K elements in the 128-byte swizzle.
#include <cuda.h>
#include <algorithm>

#include "umma_common.cuh"

namespace b200smpl {

// ---------------------------------------------------------------------------------------------
// Backward (data-gradient) GEMM on a CTA PAIR (cluster of 2 along the body tiles).  grid: (body tiles rounded up
// to even, 1, k splits)
//   D[split][body][f] = sum_{n in split} dvp[body][n] * Wb[f][n],   D row-major, ld = ldd
// Each CTA streams its own dvp tile and accumulates into its own TMEM; the B operand (Wb slab, BN x 64) is split --
// each CTA loads and holds BN/2 rows, the pair's tensor cores read both halves.  Only the leader (rank 0) issues
// MMAs; it waits for its own stage and, through a relayed remote arrive, for the peer's; its commits are multicast
// to the barriers of both CTAs.
// An odd number of body tiles leaves rank 1 of the last cluster without a tile: that padding CTA streams the last
// real tile's dvp again (so the pair MMA reads defined operands) and stores nothing.
// ---------------------------------------------------------------------------------------------
// One stage = one 64-row K slab with everything the split needs, each loaded ONCE: dvp_hi (and dvp_lo) tiles of
// this CTA's 128 bodies, this CTA's half of the Wb_hi (and Wb_lo) slab; the three products hi.hi, lo.hi, hi.lo
// are issued back to back on the resident tiles (fp32 mode: 60 KB per stage, 3 stages; bf16 mode: 30 KB, 6).
// A stage = 8 chunks x (128 bodies x 16 B): chunk c at +2048 B  ->  LBO = 2048, SBO = 128.
template <int BN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
umma_gemm2_kernel(const __grid_constant__ GemmOps ops, int split3, int ntiles, int nc8, int slab_begin, int slab_end,
                  int slabs_per_split, float* __restrict__ D, int ldd, long long split_stride) {
  constexpr int BNH = BN / 2;
  constexpr int A_BYTES = BM * BK * 2, B_BYTES = BNH * BK * 2;
  static_assert(B_BYTES % 1024 == 0, "the 128-byte swizzle needs every stage offset 1024-byte aligned");
  constexpr int MAX_STAGES = 6;
  constexpr uint32_t TMEM_COLS = 256;
  const int stage_bytes = (split3 ? 2 : 1) * (A_BYTES + B_BYTES);
  const int nstages = split3 ? 3 : 6;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + MAX_STAGES * (A_BYTES + B_BYTES));
  uint64_t* peer_full_bar = full_bar + MAX_STAGES;
  uint64_t* empty_bar = peer_full_bar + MAX_STAGES;
  uint64_t* tmem_full_bar = empty_bar + MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool padding = (int)blockIdx.x >= ntiles;     // CTA-uniform
  const int m0 = blockIdx.x * BM;
  const int s_begin = slab_begin + blockIdx.z * slabs_per_split;
  const int s_end = min(slab_end, s_begin + slabs_per_split);
  const int total_iters = max(0, s_end - s_begin);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&ops.wb_hi);
    if (split3) prefetch_tmap(&ops.wb_lo);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < MAX_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&peer_full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // launched with the PDL attribute behind the kernels that write dvp: everything above overlapped their tail
  pdl_wait();
  if (threadIdx.x == 0) pdl_trigger();
  // stage layout: [A_hi | B_hi | A_lo | B_lo]
  const int off_bhi = A_BYTES, off_alo = A_BYTES + B_BYTES, off_blo = 2 * A_BYTES + B_BYTES;

  if (warp == 0) {
    // ===== producer (both CTAs): own dvp tiles + own halves of the Wb slabs =====
    // dvp is read once, the model slabs by every body pair: keep the latter in L2
    const uint64_t pol_stream = l2_policy_evict_first(), pol_keep = l2_policy_evict_last();
    const int tile = padding ? ntiles - 1 : (int)blockIdx.x;
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < total_iters; ++it) {
      const int slab = s_begin + it;
      mbar_wait(&empty_bar[stage], phase ^ 1);
      unsigned char* sa = smem + stage * stage_bytes;
      if (elect_one()) {
        mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)stage_bytes);
        const size_t aoff = (((size_t)tile * nc8 + (size_t)slab * 8) * 128) * 8;
        bulk_g2s_hint(sa, ops.dvp_hi + aoff, A_BYTES, &full_bar[stage], pol_stream);
        tma_load_2d_hint(sa + off_bhi, &ops.wb_hi, &full_bar[stage], slab * BK, (int)rank * BNH, pol_keep);
        if (split3) {
          bulk_g2s_hint(sa + off_alo, ops.dvp_lo + aoff, A_BYTES, &full_bar[stage], pol_stream);
          tma_load_2d_hint(sa + off_blo, &ops.wb_lo, &full_bar[stage], slab * BK, (int)rank * BNH, pol_keep);
        }
      }
      __syncwarp();
      if (++stage == nstages) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    if (rank == 0) {
      // ===== leader: MMA issuer for the pair =====
      constexpr uint32_t idesc = make_idesc(2 * BM, BN);
      for (int it = 0; it < total_iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        mbar_wait(&peer_full_bar[stage], phase);                   // relaxed remote arrive of the peer's relay
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + stage * stage_bytes);
        const uint64_t da_hi = make_nosw_desc(sa, 2048, 128), db_hi = make_sw128_desc(sa + off_bhi);
        const uint64_t da_lo = make_nosw_desc(sa + off_alo, 2048, 128), db_lo = make_sw128_desc(sa + off_blo);
        if (elect_one()) {
          // A: two 16-byte chunks per UMMA_K -> +4096 B; B: +32 bytes inside the swizzle row (16-byte units)
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k)
            umma_bf16_2cta(tmem_base, da_hi + (uint64_t)(k * (4096 >> 4)), db_hi + 2 * k, idesc, (it | k) != 0);
          if (split3) {
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k)
              umma_bf16_2cta(tmem_base, da_lo + (uint64_t)(k * (4096 >> 4)), db_hi + 2 * k, idesc, 1u);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k)
              umma_bf16_2cta(tmem_base, da_hi + (uint64_t)(k * (4096 >> 4)), db_lo + 2 * k, idesc, 1u);
          }
          umma_commit_2cta(&empty_bar[stage]);
          if (it == total_iters - 1) umma_commit_2cta(tmem_full_bar);
        }
        __syncwarp();
        if (++stage == nstages) { stage = 0; phase ^= 1; }
      }
    } else {
      // ===== peer: tell the leader when this CTA's stage has landed =====
      for (int it = 0; it < total_iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        if (elect_one()) remote_arrive(&peer_full_bar[stage], 0);
        __syncwarp();
        if (++stage == nstages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (!padding) {
    // ===== epilogue: warps 2..5 own TMEM lane quadrants (warp % 4) of this CTA's 128 bodies =====
    // (the padding CTA skips it: the leader's epilogue waits for the pair's last MMA before the cluster barrier
    // that precedes the TMEM dealloc)
    const int q = warp & 3;
    const int row = m0 + q * 32 + lane;
    float* drow = D + (long long)blockIdx.z * split_stride + (long long)row * ldd;
    if (total_iters > 0) {
      mbar_wait(tmem_full_bar, 0);
      tc_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
        float* o = drow + c0;
#pragma unroll
        for (int i = 0; i < 32; i += 4)
          if (c0 + i < BN)                         // BN is a multiple of 16, not of 32: the last block may be half
            *reinterpret_cast<uint4*>(o + i) = make_uint4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
    } else {
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 4) *reinterpret_cast<uint4*>(drow + c0) = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// Forward blend GEMMs.  K schedule per body tile (FeatLayout): slab 0 (constants + shape) against model slab 0; each
// pf_hi slab j against P_hi slab j and (fp32 mode) P_lo slab j; each pf_lo slab j against P_hi slab j.  M = bodies
// (A operand = features), N = model rows: the epilogue thread owns one body and writes float4s of the group-blocked
// vpB.  (The single-CTA kernel these grew out of -- one resident 128-row model slice per CTA, bound by the shared-memory
// operand reads of an N = 128 SS-mode MMA at 175 us -- is in the history: commit ee3a35b and before.)
// ---------------------------------------------------------------------------------------------
constexpr int WS_STAGES = 5;
constexpr int WS_MAX_SLABS = 9;        // resident slabs: constants+shape, 4 x hi, 4 x lo
constexpr int WS_BN = 128;

// ---------------------------------------------------------------------------------------------
// Forward blend GEMM on a CTA PAIR (cta_group::2), BODY-stationary: the pair owns one pair of body tiles (each CTA
// keeps the feature slabs of ITS 128 bodies resident: 9 x 16 KB, loaded once) and walks a contiguous range of
// model-row tile pairs, streaming ITS 128 rows of each model slab through the stage ring.  The pair's tensor cores
// read both CTAs' rows (N = 256) and each CTA accumulates 128 bodies x 256 rows in its own TMEM (2 x 256 columns):
// per SM and K step that is 8 KB of operand reads for 128 x 256 x 16 MACs instead of 8 KB for 128 x 128 x 16, half
// the shared-memory operand bandwidth that bounds a single-CTA kernel.  Only the leader issues MMAs; the peer relays
// its "stage landed" / "accumulator drained" events to the leader's barriers with remote arrives.  With 16 body-tile
// pairs x 4 row chunks the whole GEMM is ONE wave of 64 clusters with ~22 tiles each, so the prologue (resident
// load, pipeline fill) and the drain (last tile's MMAs + epilogue) are paid once per cluster instead of once per
// 4 tiles (measured with clock64 counters in the MMA warp: 8-9 k of 35 k cycles waiting for the resident slice,
// another 12 k refilling the ring, ~10 k draining).
// ---------------------------------------------------------------------------------------------
// work list of the body-stationary kernel: cluster c = body-tile pair bp[c], model-row tile pairs [w0[c], w1[c])

template <int DUMMY>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
blend_fwd_bs2_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_f, int pslabs,
                     int ksteps_cs, int ksteps_p, int use_lo, int row0, int mtiles, int ntiles_n,
                     const __grid_constant__ BsWork work, float4* __restrict__ vpB, int nc4) {
  constexpr int SLAB = BM * BK * 2;
  constexpr int KS = BK / UMMA_K;
  constexpr uint32_t TMEM_COLS = 512;
  const int nslab_f = 1 + 2 * pslabs;                                  // resident: constants+shape, P_hi, P_lo features
  const int nslab_w = 1 + (use_lo ? 2 : 1) * pslabs;                   // streamed per row-tile pair
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  unsigned char* f_s = smem;                                          // [nslab_f][16 KB] this CTA's 128 bodies
  unsigned char* w_s = smem + WS_MAX_SLABS * SLAB;                    // [WS_STAGES][16 KB] this CTA's 128 model rows
  uint64_t* bars = reinterpret_cast<uint64_t*>(w_s + WS_STAGES * SLAB);
  uint64_t* f_full = bars;
  uint64_t* peer_f_full = bars + 1;
  uint64_t* full_bar = bars + 2;
  uint64_t* peer_full_bar = full_bar + WS_STAGES;
  uint64_t* empty_bar = peer_full_bar + WS_STAGES;
  uint64_t* tfull_bar = empty_bar + WS_STAGES;      // [2]
  uint64_t* tempty_bar = tfull_bar + 2;             // [2] (leader's are the ones waited on: 8 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int piece = (int)(blockIdx.x >> 1);
  const int btile = (int)work.bp[piece] * 2 + (int)rank;              // this CTA's body tile
  const int wtp_begin = work.w0[piece], wtp_end = work.w1[piece];

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_w);
    prefetch_tmap(&map_f);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(f_full, 1);
    mbar_init(peer_f_full, 1);
    for (int i = 0; i < WS_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&peer_full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 8);                 // four epilogue warps of each CTA of the pair
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // launched with the PDL attribute behind pose_fwd (which writes the feature rows): everything above overlapped it
  pdl_wait();
  if (threadIdx.x == 0) pdl_trigger();

  if (warp == 0) {
    // ===== TMA producer (both CTAs): own body tile once, then own half of every model-row tile pair =====
    if (elect_one()) {
      mbar_arrive_expect_tx(f_full, (uint32_t)nslab_f * SLAB);
      // rows beyond the slab (odd number of body tiles) are zero-filled by the TMA unit
      for (int s = 0; s < nslab_f; ++s) tma_load_2d(f_s + s * SLAB, &map_f, f_full, s * BK, btile * WS_BN);
    }
    __syncwarp();
    const uint64_t pol_keep = l2_policy_evict_last();       // the model slabs are re-read by every body pair
    int stage = 0;
    uint32_t phase = 0;
    for (int wtp = wtp_begin; wtp < wtp_end; ++wtp)
      for (int s = 0; s < nslab_w; ++s) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&full_bar[stage], SLAB);
          // a row tile beyond the model (odd number of row tiles) is zero-filled by the TMA unit
          tma_load_2d_hint(w_s + stage * SLAB, &map_w, &full_bar[stage], s * BK, row0 + (wtp * 2 + (int)rank) * BM, pol_keep);
        }
        __syncwarp();
        if (++stage == WS_STAGES) { stage = 0; phase ^= 1; }
      }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    if (rank == 0) {
      // ===== leader: MMA issuer of the pair =====
      constexpr uint32_t idesc = make_idesc(2 * BM, 2 * WS_BN);
      mbar_wait(f_full, 0);
      mbar_wait(peer_f_full, 0);
      uint32_t tph0 = 0, tph1 = 0;
      int acc = 0;
      for (int wtp = wtp_begin; wtp < wtp_end; ++wtp, acc ^= 1) {
        const uint32_t tph = acc ? tph1 : tph0;
        mbar_wait(&tempty_bar[acc], tph ^ 1);           // both CTAs' epilogues have drained this accumulator
        if (acc) tph1 ^= 1; else tph0 ^= 1;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 2 * WS_BN);
        for (int s = 0; s < nslab_w; ++s) {
          mbar_wait(&full_bar[stage], phase);
          mbar_wait(&peer_full_bar[stage], phase);
          tc_fence_after();
          const uint64_t db = make_sw128_desc(smem_u32(w_s + stage * SLAB));
          // model slab s meets: s = 0 the constants+shape features; 1..pslabs (W_hi[j]) the hi AND lo pose
          // features; pslabs+1.. (W_lo[j], fp32 mode) the hi pose features
          int ks = ksteps_cs, f0 = 0, f1 = -1;
          if (s > 0) {
            const int j = (s - 1) % pslabs;
            ks = min(KS, ksteps_p - j * KS);
            f0 = 1 + j;
            if (s <= pslabs) f1 = 1 + pslabs + j;
          }
          const uint64_t da0 = make_sw128_desc(smem_u32(f_s + f0 * SLAB));
          const uint64_t da1 = make_sw128_desc(smem_u32(f_s + max(f1, 0) * SLAB));
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < KS; ++k)
              if (k < ks) umma_bf16_2cta(d_tmem, da0 + 2 * k, db + 2 * k, idesc, (s | k) != 0);
            if (f1 >= 0) {
#pragma unroll
              for (int k = 0; k < KS; ++k)
                if (k < ks) umma_bf16_2cta(d_tmem, da1 + 2 * k, db + 2 * k, idesc, 1u);
            }
            umma_commit_2cta(&empty_bar[stage]);
            if (s == nslab_w - 1) umma_commit_2cta(&tfull_bar[acc]);
          }
          __syncwarp();
          if (++stage == WS_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    } else {
      // ===== peer: relay "body tile landed" and every "stage landed" to the leader =====
      mbar_wait(f_full, 0);
      if (elect_one()) remote_arrive(peer_f_full, 0);
      __syncwarp();
      for (int wtp = wtp_begin; wtp < wtp_end; ++wtp)
        for (int s = 0; s < nslab_w; ++s) {
          mbar_wait(&full_bar[stage], phase);
          if (elect_one()) remote_arrive(&peer_full_bar[stage], 0);
          __syncwarp();
          if (++stage == WS_STAGES) { stage = 0; phase ^= 1; }
        }
    }
  } else {
    // ===== epilogue (both CTAs): 128 bodies x 256 model rows of the tile pair per accumulator =====
    const int q = warp & 3;
    uint32_t tph0 = 0, tph1 = 0;
    int acc = 0;
    for (int wtp = wtp_begin; wtp < wtp_end; ++wtp, acc ^= 1) {
      const uint32_t tph = acc ? tph1 : tph0;
      mbar_wait(&tfull_bar[acc], tph);
      if (acc) tph1 ^= 1; else tph0 ^= 1;
      tc_fence_after();
      if (btile < ntiles_n) {
        const bool live_hi = wtp * 2 + 1 < mtiles;
        float4* colbase = vpB + ((size_t)(btile * 4 + q) * nc4 + ((row0 + wtp * 2 * BM) >> 2)) * 32 + lane;
#pragma unroll 1
        for (int c0 = 0; c0 < 2 * WS_BN; c0 += 32) {
          if (c0 >= WS_BN && !live_hi) continue;
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * 2 * WS_BN + c0), v);
          float4* o = colbase + (size_t)(c0 >> 2) * 32;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            o[i * 32] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                    __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&tempty_bar[acc])) : "memory");
        else remote_arrive(&tempty_bar[acc], 0);
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---- host side ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 matrix [rows][pitch] (K contiguous), visible extent k_extent x rows, box 64 x box_rows, 128B swizzle
int make_map(CUtensorMap* map, const void* base, int k_extent, int rows, int pitch_elems, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) return fail(B200SMPL_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)k_extent, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(B200SMPL_ERR_CUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
  return 0;
}

// Work list of the body-stationary forward GEMM (host side; pure arithmetic, also exposed to the CPU tests through
// b200smpl_debug_fwd_gemm_worklist).  CTA pairs are scheduled per TPC (2 SMs).  The (body pair, row-tile pair) list,
// body pair major, is cut into one equal range per TPC; a range that crosses into the next body pair becomes two
// clusters (the resident operand changes), longest pieces first so that the short ones fill the tail of the wave.
// Returns the number of clusters, or -1 when the list does not fit.
int build_bs_work(int bp_total, int wtp_total, int tpcs, BsWork& work) {
  if (bp_total < 1 || wtp_total < 1) return -1;
  const long long total = (long long)bp_total * wtp_total;
  const int nranges = (int)std::min<long long>(total, std::max(tpcs, bp_total));
  struct Piece { int bp, w0, w1; };
  std::vector<Piece> pieces;
  for (int r = 0; r < nranges; ++r) {
    long long lo = total * r / nranges, hi = total * (r + 1) / nranges;
    while (lo < hi) {
      const int bp = (int)(lo / wtp_total);
      const long long end = std::min<long long>(hi, (long long)(bp + 1) * wtp_total);
      pieces.push_back({bp, (int)(lo - (long long)bp * wtp_total), (int)(end - (long long)bp * wtp_total)});
      lo = end;
    }
  }
  // the plain rectangular split (every body pair cut into the same number of row chunks, one wave) is kept when
  // its longest cluster is no longer than the flattened one plus a prologue, and for very wide slabs
  const int rect_chunks = std::max(1, std::min(wtp_total, tpcs / std::max(1, bp_total)));
  const int rect_len = (wtp_total + rect_chunks - 1) / rect_chunks;
  const int flat_len = (int)((total + nranges - 1) / nranges);
  if ((int)pieces.size() > BS_MAX_WORK || rect_len <= flat_len + 1) {
    pieces.clear();
    const int chunks = std::max(1, std::min(rect_chunks, BS_MAX_WORK / bp_total));
    const int wpc = (wtp_total + chunks - 1) / chunks;
    for (int bp = 0; bp < bp_total; ++bp)
      for (int w = 0; w < wtp_total; w += wpc) pieces.push_back({bp, w, std::min(wtp_total, w + wpc)});
    if ((int)pieces.size() > BS_MAX_WORK) return -1;
  }
  std::stable_sort(pieces.begin(), pieces.end(), [](const Piece& a, const Piece& b) { return a.w1 - a.w0 > b.w1 - b.w0; });
  memset(&work, 0, sizeof(work));
  int npieces = 0;
  for (const Piece& pc : pieces) {
    work.bp[npieces] = (uint16_t)pc.bp; work.w0[npieces] = (uint16_t)pc.w0; work.w1[npieces] = (uint16_t)pc.w1;
    ++npieces;
  }
  return npieces;
}

// body-stationary CTA-pair launch: one wave of (body-tile pair) x (row chunk) clusters.  Slabs are at most MAX_SLAB
// bodies wide (make_plan), which the work list always fits.
int launch_blend_fwd_umma(const DevModel& m, int mode, const __nv_bfloat16* feat, int S, int Sw, float* vpT,
                          int row_begin, int row_end, int num_sms, cudaStream_t st) {
  // a joints-only call on a model without picked or regressed joints has no rows to blend
  if (row_begin >= row_end) return 0;
  const int pslabs = m.fl.pseg / BK;
  const int use_lo = (mode == B200SMPL_MODE_BF16) ? 0 : 1;
  if (1 + 2 * pslabs > WS_MAX_SLABS) return fail(B200SMPL_ERR_INVALID, "feature pitch too large for the resident operand");
  CUtensorMap map_w, map_f;
  int rc;
  if ((rc = make_map(&map_w, m.Wf, m.fl.pitch, m.n_pad, m.fl.pitch, BM))) return rc;
  if ((rc = make_map(&map_f, feat, m.fl.pitch, Sw, m.fl.pitch, WS_BN))) return rc;   // rows >= Sw read as zero
  constexpr int smem = (WS_MAX_SLABS + WS_STAGES) * BM * BK * 2 + 1024 + 256;
  auto kern = blend_fwd_bs2_kernel<0>;
  B200_SMEM_ATTR_ONCE(kern, smem);
  const int mtiles = (row_end - row_begin) / BM;
  const int wtp_total = (mtiles + 1) / 2;
  const int ntiles_n = Sw / WS_BN;
  const int bp_total = (ntiles_n + 1) / 2;
  BsWork work;
  const int npieces = build_bs_work(bp_total, wtp_total, std::max(1, num_sms / 2), work);
  if (npieces < 0) return fail(B200SMPL_ERR_INVALID, "slab too wide for the forward GEMM work list");
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * npieces, 1, 1);
  cfg.blockDim = dim3(GEMM_THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  LaunchTimer _timer("blend_fwd_umma", st);
  B200_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, map_w, map_f, pslabs, (m.fl.k_cs + UMMA_K - 1) / UMMA_K,
                                   (NPOSE + UMMA_K - 1) / UMMA_K, use_lo, row_begin, mtiles, ntiles_n, work,
                                   reinterpret_cast<float4*>(vpT), m.n_pad / 4));
  B200_LAUNCH_CHECK("blend_fwd_umma");
  return 0;
}

}  // namespace b200smpl
extern "C" int b200smpl_debug_fwd_gemm_worklist(int body_tiles, int row_tiles, int num_sms, uint16_t* out, int capacity) {
  using namespace b200smpl;
  BsWork work;
  const int n = build_bs_work((body_tiles + 1) / 2, (row_tiles + 1) / 2, std::max(1, num_sms / 2), work);
  if (n < 0 || out == nullptr || n > capacity) return n < 0 ? -1 : n;
  for (int c = 0; c < n; ++c) { out[c * 3] = work.bp[c]; out[c * 3 + 1] = work.w0[c]; out[c * 3 + 2] = work.w1[c]; }
  return n;
}
namespace b200smpl {

// number of split-K partials the backward GEMM writes for slab width S
int blend_bwd_umma_splits(const DevModel& m, int S, int num_sms) {
  const int mtiles = round_up((S + BM - 1) / BM, 2);      // an odd tile count launches one padding CTA
  const int slabs = (m.n_rows + BK - 1) / BK;
  // CTA pairs are scheduled per TPC (2 SMs): never more pairs than TPCs, or a second, nearly empty wave runs
  int want = std::max(1, num_sms / mtiles);
  want = std::max(1, std::min(want, slabs / 8));
  return want;
}

template <int BN>
static int launch_bwd_pair(const GemmOps& ops, int split3, int ntiles, int nc8, int slab_begin, int slab_end,
                           int nsplit, float* dfeat_part, long long split_stride, cudaStream_t st) {
  constexpr int smem = 6 * (BM * BK * 2 + (BN / 2) * BK * 2) + 1024 + 512;
  auto kern = umma_gemm2_kernel<BN>;
  B200_SMEM_ATTR_ONCE(kern, smem);
  const int slabs = slab_end - slab_begin;
  const int sps = (slabs + nsplit - 1) / nsplit;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(round_up(ntiles, 2), 1, nsplit);
  cfg.blockDim = dim3(GEMM_THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  LaunchTimer _timer("blend_bwd_umma", st);
  B200_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ops, split3, ntiles, nc8, slab_begin, slab_end, sps, dfeat_part, BN,
                                   split_stride));
  B200_LAUNCH_CHECK("blend_bwd_umma");
  return 0;
}

// dfeat_part[nsplit][S][nf_pad]; rows [0, Sw) of every split are written.  dvp rows in
// [row_end, round_up(row_end, 64)) must be finite (the api zeroes them): the model operand is zero there.
int launch_blend_bwd_umma(const DevModel& m, int mode, const __nv_bfloat16* dvp_hi, const __nv_bfloat16* dvp_lo,
                          int S, int Sw, float* dfeat_part, int nsplit, int row_begin, int row_end,
                          cudaStream_t st) {
  // nf_pad = round_up(num_betas + NPOSE, 16): 208 for 1 beta, 224 for 2..MAX_BETAS
  const int nf_pad = m.fl.nf_pad;
  if (nf_pad != 208 && nf_pad != 224)
    return fail(B200SMPL_ERR_INVALID, "unsupported num_betas for the tensor-core backward (nf_pad=" + std::to_string(nf_pad) + ")");
  const bool split3 = (mode != B200SMPL_MODE_BF16) && dvp_lo != nullptr;
  GemmOps ops;
  memset(&ops, 0, sizeof(ops));
  ops.dvp_hi = dvp_hi;
  ops.dvp_lo = dvp_lo;
  // every CTA of a pair loads nf_pad/2 rows of the Wb slab.  K extent = row_end: model columns beyond it are never
  // read (TMA zero-fills out-of-bounds)
  int rc;
  if ((rc = make_map(&ops.wb_hi, m.Wb_hi, row_end, nf_pad, m.n_pad, nf_pad / 2))) return rc;
  if (split3 && (rc = make_map(&ops.wb_lo, m.Wb_lo, row_end, nf_pad, m.n_pad, nf_pad / 2))) return rc;
  const int slab_begin = row_begin / BK, slab_end = (row_end + BK - 1) / BK;
  const long long split_stride = (long long)S * nf_pad;
  auto launch = nf_pad == 224 ? launch_bwd_pair<224> : launch_bwd_pair<208>;
  return launch(ops, split3 ? 1 : 0, Sw / BM, m.n_pad / 8, slab_begin, slab_end, nsplit, dfeat_part, split_stride, st);
}

}  // namespace b200smpl
