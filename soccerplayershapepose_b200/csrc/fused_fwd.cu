// Fused forward: blend GEMM (SURVEY.md section 8 rows a4 + a7) with the linear blend skinning (row a9) in its
// epilogue, so that v_posed never makes the HBM round trip between the two.  Used for forward-only calls (no
// products kept for a backward): 188 us against 108 + 136 us of blend GEMM + skinning kernel at B = 4096.  A call
// that keeps the products needs v_posed in HBM; writing it from this kernel as well stored 658 MB without reading
// anything and ran at the speed of the two kernels (242 us), so those calls run the two kernels (see DESIGN.md,
// "fused forward").
//
// The GEMM is the body-stationary CTA-pair kernel of blend_umma.cu (tcgen05 cta_group::2, features resident in
// shared memory, model slabs streamed by TMA) with two changes:
//   * a tile is 96 model rows = one 32-vertex skinning tile (N = 96, each CTA stages 48 rows of every slab), two
//     alternating 96-column TMEM accumulators;
//   * the 24 skinning transforms of every body live in TENSOR MEMORY next to the accumulators: lane = body (the
//     accumulator row of that body), 12 columns per joint, columns [192, 480).  Shared memory cannot hold them
//     (128 bodies x 1152 B = 147 KB next to 147 KB of resident features); TMEM has exactly the room the narrower
//     accumulators leave.  A slot reload is three warp-uniform tcgen05.ld of 4 columns.
// Epilogue warps (two per TMEM lane quadrant; each takes one half -- 16 vertices, 48 columns -- of every tile, so the
// epilogue of tile t overlaps the MMAs of tile t + 1): thread = body reads its accumulator columns 24 at a time,
// skins the 8 vertices with the packed-pair slot arithmetic of lbs.cu and flushes them through a per-warp
// transposing tile as 96-byte row segments of the (B, V, 3) output.
// Virtual (joint) row tiles are only stored, to the group-blocked vpB.
//
// The variants that lost (three epilogue warps per quadrant on setmaxnreg registers, the half tile staged in 48
// registers with the accumulator released at once, 192-byte row segments) are in the history (commit cf06df6) and in
// profiles/r02_experiments.md section 8.
#include <algorithm>

#include "lbs_tiles.cuh"
#include "umma_common.cuh"

namespace b200smpl {

constexpr int FF_BN = 96;                           // model rows per tile = 32 vertices
constexpr int FF_BNH = FF_BN / 2;                   // rows of a slab each CTA of the pair stages
constexpr int FF_NW = 2;                            // epilogue warps per TMEM lane quadrant
constexpr int FF_STAGES = 7;
constexpr int FF_STAGE_BYTES = FF_BNH * BK * 2;     // 6 KB
constexpr int FF_PS = (NPOSE + BK - 1) / BK;        // 64-wide K slabs of one pose segment (4)
constexpr int FF_KSP = (NPOSE + UMMA_K - 1) / UMMA_K;   // K steps of one pose segment (13)
constexpr int FF_MAX_SLABS = 1 + 2 * FF_PS;         // resident feature slabs: constants+shape, 4 x pf_hi, 4 x pf_lo
constexpr int FF_SLAB = BM * BK * 2;                // 16 KB
constexpr int FF_EPI_WARPS = 4 * FF_NW;
constexpr int FF_EPI_WARP0 = 2;                     // warps 0 / 1 = TMA / MMA, warps 2.. epilogue
constexpr int FF_THREADS = (FF_EPI_WARP0 + FF_EPI_WARPS) * 32;
constexpr int FF_HV = 8;                            // vertices per flush of the staging tile
constexpr int FF_TR_COL = 2 * FF_BN;                // first TMEM column of the transforms (12 per joint)
constexpr int FF_WV = TILE_V / 2;                   // vertices of a half tile (one epilogue warp's unit of work)
constexpr int FF_PLAN_WORDS = (FF_WV / 8) * 40;     // plan records of a half tile
constexpr int FF_TILE_WORDS = ItemShape<FF_HV>::TILE_WORDS;
constexpr int FF_NBARS = 1 + 2 * FF_STAGES + 4 + 2 * FF_EPI_WARPS;
constexpr size_t FF_SMEM = (size_t)FF_MAX_SLABS * FF_SLAB + (size_t)FF_STAGES * FF_STAGE_BYTES +
                           (size_t)FF_EPI_WARPS * (FF_TILE_WORDS + 2 * FF_PLAN_WORDS) * 4 + FF_NBARS * 8 + 16 +
                           1024 /*alignment slack*/;
static_assert(FF_SMEM <= 232448, "fused forward: shared memory budget");
static_assert(FF_TR_COL + NJ * AELEMS <= 512, "fused forward: tensor memory budget");
static_assert(NJ % FF_NW == 0, "joints split evenly over the warps of a quadrant");

// TMA load of a CTA pair: the bytes land in THIS CTA's shared memory, the transaction count on the LEADER's
// mbarrier (same offset, CTA rank bit of the shared::cluster address cleared), so the MMA issuer waits on one
// barrier per stage and no warp has to relay the peer's "stage landed"
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}

// ---- tensor memory <-> registers (thread = lane of the warp's quadrant) --------------------------------------
__device__ __forceinline__ void tmem_st_x4(uint32_t taddr, const float4& v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(__float_as_uint(v.x)), "r"(__float_as_uint(v.y)), "r"(__float_as_uint(v.z)),
                 "r"(__float_as_uint(v.w))
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 12 columns (one joint's transform) -> registers, complete on return
__device__ __forceinline__ void tmem_ld_12(uint32_t taddr, uint32_t (&r)[12]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%12];\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%4, %5, %6, %7}, [%13];\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%8, %9, %10, %11}, [%14];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11])
      : "r"(taddr), "r"(taddr + 4), "r"(taddr + 8)
      : "memory");
}
// 24 accumulator columns (8 vertices of this body) -> registers, complete on return
__device__ __forceinline__ void tmem_ld_24(uint32_t taddr, uint32_t (&r)[24]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%24];\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%8, %9, %10, %11, %12, %13, %14, %15}, [%25];\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%16, %17, %18, %19, %20, %21, %22, %23}, [%26];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23])
      : "r"(taddr), "r"(taddr + 8), "r"(taddr + 16)
      : "memory");
}

// slot (re)load from tensor memory: columns of joint `joint` hold (r00 r10 r01 r11) (r02 r12 t0 t1) (r20 r21 r22 t2)
template <bool HI>
__device__ __forceinline__ void load_slot_tm(SlotXY& s, SlotZ2& z, uint32_t tr_base, int joint) {
  uint32_t r[12];
  tmem_ld_12(tr_base + (uint32_t)(joint * AELEMS), r);
  s.c0 = mk2(__uint_as_float(r[0]), __uint_as_float(r[1]));
  s.c1 = mk2(__uint_as_float(r[2]), __uint_as_float(r[3]));
  s.c2 = mk2(__uint_as_float(r[4]), __uint_as_float(r[5]));
  s.t = mk2(__uint_as_float(r[6]), __uint_as_float(r[7]));
  z.r20 = set_half<HI>(z.r20, __uint_as_float(r[8]));
  z.r21 = set_half<HI>(z.r21, __uint_as_float(r[9]));
  z.r22 = set_half<HI>(z.r22, __uint_as_float(r[10]));
  z.t2 = set_half<HI>(z.t2, __uint_as_float(r[11]));
}

// 4 vertices: v_posed in registers (P[12]) -> skinned coordinates into the lane's row of the staging tile
// (the arithmetic of lbs.cu::skin_fwd4)
__device__ __forceinline__ void skin_fwd4_tm(Slots& s, uint32_t tr_base, const uint32_t* meta_s, const float4* wts_s,
                                             uint32_t force, float tx, float ty, float tz, const float (&P)[12],
                                             float* row_out) {
  const uint4 m4 = *reinterpret_cast<const uint4*>(meta_s);
  const uint32_t mts[4] = {m4.x | force, m4.y, m4.z, m4.w};
  float4 ws[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) ws[i] = wts_s[i];
  float o[12];
  const f2 txy = mk2(tx, ty), tz0 = mk2(tz, 0.f);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t mt = mts[i];
    const float4 w = ws[i];
    if (mt & (0xFu << 20)) {
      if (mt & (1u << 20)) load_slot_tm<false>(s.s0, s.zA, tr_base, mt & 31);
      if (mt & (1u << 21)) load_slot_tm<true>(s.s1, s.zA, tr_base, (mt >> 5) & 31);
      if (mt & (1u << 22)) load_slot_tm<false>(s.s2, s.zB, tr_base, (mt >> 10) & 31);
      if (mt & (1u << 23)) load_slot_tm<true>(s.s3, s.zB, tr_base, (mt >> 15) & 31);
    }
    const f2 px = bc2(P[i * 3]), py = bc2(P[i * 3 + 1]), pz = bc2(P[i * 3 + 2]);
    f2 oxy = txy;
#define B200_SKIN_XY(sl, wk) oxy = fma2(bc2(wk), fma2(sl.c0, px, fma2(sl.c1, py, fma2(sl.c2, pz, sl.t))), oxy);
    B200_SKIN_XY(s.s0, w.x)
    B200_SKIN_XY(s.s1, w.y)
    B200_SKIN_XY(s.s2, w.z)
    B200_SKIN_XY(s.s3, w.w)
#undef B200_SKIN_XY
    f2 oz = fma2(mk2(w.x, w.y), fma2(s.zA.r20, px, fma2(s.zA.r21, py, fma2(s.zA.r22, pz, s.zA.t2))), tz0);
    oz = fma2(mk2(w.z, w.w), fma2(s.zB.r20, px, fma2(s.zB.r21, py, fma2(s.zB.r22, pz, s.zB.t2))), oz);
    o[i * 3] = lo2(oxy); o[i * 3 + 1] = hi2(oxy); o[i * 3 + 2] = lo2(oz) + hi2(oz);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
    *reinterpret_cast<float4*>(row_out + i * 4) = make_float4(o[i * 4], o[i * 4 + 1], o[i * 4 + 2], o[i * 4 + 3]);
}

// grid: 2 x (clusters of the work list), cluster = CTA pair.  Row tiles are counted from model row 0.
//   vpB     group-blocked blend output (skin_common.cuh); written for the virtual (joint) row tiles only
//   n_vtiles  vertex tiles (m.ntiles): row tiles below it are skinned into verts, the others only stored
template <bool USE_LO>
__global__ void __launch_bounds__(FF_THREADS, 1)
blend_lbs_fwd_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_f,
                     int ksteps_cs, int n_pad, int ntiles_n,
                     const __grid_constant__ BsWork work, float4* __restrict__ vpB, int nc4,
                     const float4* __restrict__ A_blk, int b0, int nb, const float* __restrict__ transl,
                     float* __restrict__ verts, int V, int n_vtiles, int vec_ok, const uint32_t* __restrict__ vplan) {
  constexpr int KS = BK / UMMA_K;
  constexpr uint32_t TMEM_COLS = 512;
  using SH = ItemShape<FF_HV>;
  constexpr int PS = FF_PS;                                            // 64-wide slabs of a pose segment
  constexpr int nslab_f = 1 + 2 * PS;                                  // resident: constants+shape, pf_hi, pf_lo
  constexpr int nslab_w = 1 + (USE_LO ? 2 : 1) * PS;                   // streamed per row tile
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  // offset arithmetic on the shared array (not a round trip through an integer) keeps every pointer below in the
  // shared address space: LDS / STS instead of generic accesses
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* f_s = smem;                                          // [nslab_f][16 KB] this CTA's 128 bodies
  unsigned char* w_s = f_s + FF_MAX_SLABS * FF_SLAB;                  // [FF_STAGES][6 KB] this CTA's 48 rows of a slab
  float* tiles = reinterpret_cast<float*>(w_s + FF_STAGES * FF_STAGE_BYTES);       // [12][32][HROW] output staging
  uint32_t* stashes = reinterpret_cast<uint32_t*>(tiles + FF_EPI_WARPS * FF_TILE_WORDS);   // [8][2][160] plan records
  uint64_t* bars = reinterpret_cast<uint64_t*>(stashes + FF_EPI_WARPS * 2 * FF_PLAN_WORDS);
  uint64_t* f_full = bars;
  uint64_t* full_bar = bars + 1;
  uint64_t* empty_bar = full_bar + FF_STAGES;
  uint64_t* tfull_bar = empty_bar + FF_STAGES;      // [2]
  uint64_t* tempty_bar = tfull_bar + 2;             // [2] (the leader's are waited on: 8 arrivals)
  uint64_t* wbars = tempty_bar + 2;                 // [8][2] plan records landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbars + 2 * FF_EPI_WARPS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int piece = (int)(blockIdx.x >> 1);
  const int btile = (int)work.bp[piece] * 2 + (int)rank;              // this CTA's body tile
  const int wt_begin = work.w0[piece], wt_end = work.w1[piece];

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_w);
    prefetch_tmap(&map_f);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(f_full, 1);
    for (int i = 0; i < FF_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 16);                // two epilogue warps per quadrant and tile, both CTAs of the pair
    }
    for (int i = 0; i < 2 * FF_EPI_WARPS; ++i) mbar_init(&wbars[i], 1);
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
  // launched with the PDL attribute behind pose_fwd (which writes the feature rows and the transforms)
  pdl_wait();
  if (threadIdx.x == 0) pdl_trigger();

  if (warp < FF_EPI_WARP0) {
  if (warp == 0) {
    // ===== TMA producer (both CTAs): own body tile once, then own half of every model slab of every row tile =====
    const uint64_t pol_keep = l2_policy_evict_last();       // the model slabs are re-read by every body pair
    if (elect_one()) {
      if (rank == 0) mbar_arrive_expect_tx(f_full, 2u * (uint32_t)nslab_f * FF_SLAB);   // both CTAs' bytes count here
      for (int s = 0; s < nslab_f; ++s) tma_load_2d_pair(f_s + s * FF_SLAB, &map_f, f_full, s * BK, btile * BM, l2_policy_evict_first());
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    for (int wt = wt_begin; wt < wt_end; ++wt)
      for (int s = 0; s < nslab_w; ++s) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elect_one()) {
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * FF_STAGE_BYTES);
          tma_load_2d_pair(w_s + stage * FF_STAGE_BYTES, &map_w, &full_bar[stage], s * BK, wt * FF_BN + (int)rank * FF_BNH, pol_keep);
        }
        __syncwarp();
        if (++stage == FF_STAGES) { stage = 0; phase ^= 1; }
      }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    if (rank == 0) {
      // ===== leader: MMA issuer of the pair.  With 96-column tiles an MMA lasts 48 cycles, so the per-slab issue
      // overhead decides the GEMM's rate: the K schedule is three loops with compile-time structure (no per-slab
      // division / descriptor rebuild; it was ~1000 cycles per slab with the schedule computed at run time) =====
      constexpr uint32_t idesc = make_idesc(2 * BM, FF_BN);
      mbar_wait(f_full, 0);
      const uint64_t da_base = make_sw128_desc(smem_u32(f_s));
      const uint64_t db_base = make_sw128_desc(smem_u32(w_s));
      uint32_t tph0 = 0, tph1 = 0;
      int acc = 0;
      // one model slab against one or two resident feature slabs; `first`: the tile's first MMA overwrites
      auto slab = [&](uint32_t d_tmem, int ks, int f0, int f1, bool first, uint64_t* tfull) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint64_t db = db_base + (uint64_t)(stage * (FF_STAGE_BYTES >> 4));
        if (elect_one()) {
          const uint64_t da0 = da_base + (uint64_t)(f0 * (FF_SLAB >> 4));
#pragma unroll
          for (int k = 0; k < KS; ++k)
            if (k < ks) umma_bf16_2cta(d_tmem, da0 + 2 * k, db + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
          if (f1 >= 0) {
            const uint64_t da1 = da_base + (uint64_t)(f1 * (FF_SLAB >> 4));
#pragma unroll
            for (int k = 0; k < KS; ++k)
              if (k < ks) umma_bf16_2cta(d_tmem, da1 + 2 * k, db + 2 * k, idesc, 1u);
          }
          umma_commit_2cta(&empty_bar[stage]);
          if (tfull != nullptr) umma_commit_2cta(tfull);
        }
        __syncwarp();
        if (++stage == FF_STAGES) { stage = 0; phase ^= 1; }
      };
#pragma unroll 1
      for (int wt = wt_begin; wt < wt_end; ++wt, acc ^= 1) {
        const uint32_t tph = acc ? tph1 : tph0;
        mbar_wait(&tempty_bar[acc], tph ^ 1);           // both CTAs' epilogues have drained this accumulator
        if (acc) tph1 ^= 1; else tph0 ^= 1;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * FF_BN);
        // slab 0: constants + shape features; slabs 1..PS (W_hi[j]): hi AND lo pose features; slabs PS+1..
        // (W_lo[j], fp32 mode): hi pose features
        slab(d_tmem, ksteps_cs, 0, -1, true, nullptr);
#pragma unroll
        for (int j = 0; j < PS; ++j)
          slab(d_tmem, min(KS, FF_KSP - j * KS), 1 + j, 1 + PS + j, false, (!USE_LO && j == PS - 1) ? &tfull_bar[acc] : nullptr);
        if (USE_LO) {
#pragma unroll
          for (int j = 0; j < PS; ++j)
            slab(d_tmem, min(KS, FF_KSP - j * KS), 1 + j, -1, false, j == PS - 1 ? &tfull_bar[acc] : nullptr);
        }
      }
    }
  }
  } else {
    // ===== epilogue (both CTAs): the two warps of a TMEM lane quadrant walk the sequence of HALF tiles (16 vertices =
    // 48 accumulator columns) of the cluster's range, warp r3 taking half r3 of every tile: both warps share each
    // tile, so the epilogue of tile t overlaps the MMAs of tile t + 1 in the other accumulator =====
    const int e = warp - FF_EPI_WARP0, q = warp & 3, r3 = e >> 2;
    float* tile = tiles + e * FF_TILE_WORDS;
    float* my_row = tile + lane * SH::HROW;
    uint32_t* stash = stashes + e * 2 * FF_PLAN_WORDS;
    uint64_t* wbar = wbars + e * 2;
    const bool live = btile < ntiles_n;
    const int g = btile * 4 + q;                                       // slab-local body group of this warp
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t tr_base = lane_base + FF_TR_COL;
    const bool skin = verts != nullptr;
    // ---- the group's transforms -> tensor memory (the two warps of the quadrant take 12 joints each) ----
    if (live && skin) {
      const float4* ap = A_blk + (size_t)g * (NJ * 3 * 32) + lane;
#pragma unroll 1
      for (int j = r3 * (NJ / FF_NW); j < (r3 + 1) * (NJ / FF_NW); ++j) {
        const float4 x0 = ap[(j * 3) * 32], x1 = ap[(j * 3 + 1) * 32], x2 = ap[(j * 3 + 2) * 32];
        tmem_st_x4(tr_base + j * AELEMS, x0);
        tmem_st_x4(tr_base + j * AELEMS + 4, x1);
        tmem_st_x4(tr_base + j * AELEMS + 8, x2);
      }
      tmem_wait_st();
    }
    tc_fence_before();
    asm volatile("bar.sync %0, %1;" ::"r"(1 + q), "n"(32 * FF_NW) : "memory");
    tc_fence_after();
    float tx = 0.f, ty = 0.f, tz = 0.f;
    if (live && transl != nullptr && g * 32 + lane < nb) {
      const float* tp = transl + (size_t)(b0 + g * 32 + lane) * 3;
      tx = tp[0]; ty = tp[1]; tz = tp[2];
    }
    const int nrows = max(0, min(32, nb - g * 32));
    float* v_g = skin ? verts + (size_t)(b0 + g * 32) * V * 3 : nullptr;
    const size_t row_stride = (size_t)V * 3;
    auto release = [&](int acc) {                                      // this warp is done reading the accumulator
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&tempty_bar[acc])) : "memory");
        else remote_arrive(&tempty_bar[acc], 0);
      }
    };
    const int nhalf = 2 * (wt_end - wt_begin);
    auto is_vhalf = [&](int h) { return h < nhalf && wt_begin + (h >> 1) < n_vtiles; };
    auto issue_plan = [&](uint32_t b, int h) {                         // one lane: plan records of half tile h
      mbar_expect_tx(&wbar[b], FF_PLAN_WORDS * 4);
      bulk_g2s(stash + b * FF_PLAN_WORDS, vplan + ((size_t)(wt_begin + (h >> 1)) * 2 + (h & 1)) * FF_PLAN_WORDS,
               FF_PLAN_WORDS * 4, &wbar[b]);
    };
    uint32_t n_plan = 0;
    if (live && skin && is_vhalf(r3) && lane == 0) issue_plan(0u, r3);
    Slots sl;
    sl.zA.r20 = sl.zA.r21 = sl.zA.r22 = sl.zA.t2 = sl.zB.r20 = sl.zB.r21 = sl.zB.r22 = sl.zB.t2 = mk2(0.f, 0.f);
    sl.s0.c0 = sl.s0.c1 = sl.s0.c2 = sl.s0.t = sl.s1.c0 = sl.s1.c1 = sl.s1.c2 = sl.s1.t = mk2(0.f, 0.f);
    sl.s2.c0 = sl.s2.c1 = sl.s2.c2 = sl.s2.t = sl.s3.c0 = sl.s3.c1 = sl.s3.c2 = sl.s3.t = mk2(0.f, 0.f);
#pragma unroll 1
    for (int h = r3; h < nhalf; h += FF_NW) {
      const int ti = h >> 1, half = h & 1, wt = wt_begin + ti, acc = ti & 1;
      mbar_wait(&tfull_bar[acc], (uint32_t)(ti >> 1) & 1u);            // tile ti is the (ti / 2)-th use of its accumulator
      tc_fence_after();
      if (!live) {
        release(acc);
        continue;
      }
      const int row_w = wt * FF_BN + half * (FF_BN / 2);                // first blend row of this half tile
      const uint32_t acc_base = lane_base + (uint32_t)(acc * FF_BN + half * (FF_BN / 2));
      if (skin && wt < n_vtiles) {
        const uint32_t b = n_plan & 1;
        if (is_vhalf(h + FF_NW) && lane == 0) issue_plan(b ^ 1, h + FF_NW);
        mbar_wait(&wbar[b], (n_plan >> 1) & 1);
        const uint32_t* st = stash + b * FF_PLAN_WORDS;
#pragma unroll 1
        for (int sub = 0; sub < FF_WV / FF_HV; ++sub) {
          uint32_t v[24];
          tmem_ld_24(acc_base + (uint32_t)(sub * 24), v);
          if (sub == FF_WV / FF_HV - 1) release(acc);                  // the MMAs of the tile after next may start
#pragma unroll
          for (int u = 0; u < FF_HV / 4; ++u) {
            float P[12];
#pragma unroll
            for (int i = 0; i < 12; ++i)
              P[i] = __uint_as_float(v[u * 12 + i]);
            skin_fwd4_tm(sl, tr_base, plan_meta(st, sub * (FF_HV / 4) + u), plan_wts(st, sub * (FF_HV / 4) + u),
                         (sub == 0 && u == 0) ? (0xFu << 20) : 0u, tx, ty, tz, P, my_row + u * 12);
          }
          __syncwarp();
          {
            const int vbase = wt * TILE_V + half * FF_WV + sub * FF_HV;
            const int ncols = max(0, min(FF_HV, V - vbase)) * 3;
            float* dst0 = v_g + (size_t)vbase * 3;
            if (!vec_ok) tile_to_global_scalar<FF_HV>(tile, dst0, row_stride, nrows, ncols, lane);
            else tile_to_global<FF_HV>(tile, dst0, row_stride, nrows, ncols, lane);
          }
          __syncwarp();                                                // the tile is free again
        }
        ++n_plan;
      } else {
        // virtual (joint) rows, or a call without a vertex output: store the blend rows only
        float4* colbase = vpB + ((size_t)g * nc4 + (row_w >> 2)) * 32 + lane;
#pragma unroll 1
        for (int c0 = 0; c0 < FF_BN / 2; c0 += 24) {
          uint32_t v[24];
          tmem_ld_24(acc_base + (uint32_t)c0, v);
          if (c0 + 24 >= FF_BN / 2) release(acc);
          float4* o = colbase + (size_t)(c0 >> 2) * 32;
#pragma unroll
          for (int i = 0; i < 6; ++i)
            if (row_w + c0 + 4 * i < n_pad)
              o[i * 32] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                      __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
        }
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
// Sw = active slab width (multiple of 128).  Blends every row tile of the model (vertex rows and virtual joint rows)
// for the slab; vertex tiles are skinned into verts when it is given.  vpB receives the virtual rows.
int launch_blend_lbs_fwd(const DevModel& m, int mode, const __nv_bfloat16* feat, int S, int Sw, float* vpT,
                         const float* A_blk, int b0, int nb, const float* transl, float* verts, int num_sms,
                         cudaStream_t st) {
  (void)S;
  const bool use_lo = mode != B200SMPL_MODE_BF16;
  if (m.fl.pseg != FF_PS * BK) return fail(B200SMPL_ERR_INVALID, "fused forward: unexpected pose segment width");
  if (m.n_virt0 != m.ntiles * FF_BN) return fail(B200SMPL_ERR_INVALID, "fused forward: vertex tiles must be 96 rows");
  CUtensorMap map_w, map_f;
  int rc;
  if ((rc = make_map(&map_w, m.Wf, m.fl.pitch, m.n_pad, m.fl.pitch, FF_BNH))) return rc;
  if ((rc = make_map(&map_f, feat, m.fl.pitch, Sw, m.fl.pitch, BM))) return rc;          // rows >= Sw read as zero
  auto kern = use_lo ? blend_lbs_fwd_kernel<true> : blend_lbs_fwd_kernel<false>;
  B200_SMEM_ATTR_ONCE(blend_lbs_fwd_kernel<true>, FF_SMEM);
  B200_SMEM_ATTR_ONCE(blend_lbs_fwd_kernel<false>, FF_SMEM);
  const int wt_total = (m.n_pad + FF_BN - 1) / FF_BN;
  const int ntiles_n = Sw / BM;
  const int bp_total = (ntiles_n + 1) / 2;
  BsWork work;
  const int npieces = build_bs_work(bp_total, wt_total, std::max(1, num_sms / 2), work);
  if (npieces < 0) return fail(B200SMPL_ERR_INVALID, "slab too wide for the fused forward work list");
  const int vec_ok = (verts != nullptr && (m.V & 1) == 0 && (reinterpret_cast<uintptr_t>(verts) & 7) == 0) ? 1 : 0;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * npieces, 1, 1);
  cfg.blockDim = dim3(FF_THREADS, 1, 1);
  cfg.dynamicSmemBytes = FF_SMEM;
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
  LaunchTimer _timer("blend_lbs_fwd", st);
  B200_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, map_w, map_f, (m.fl.k_cs + UMMA_K - 1) / UMMA_K, m.n_pad, ntiles_n, work,
                                   reinterpret_cast<float4*>(vpT), m.n_pad / 4, reinterpret_cast<const float4*>(A_blk), b0, nb,
                                   transl, verts, m.V, m.ntiles, vec_ok, m.vplan));
  B200_LAUNCH_CHECK("blend_lbs_fwd");
  return 0;
}

}  // namespace b200smpl
