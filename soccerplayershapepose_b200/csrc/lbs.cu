// Linear blend skinning of the 6890 vertices, forward and backward (SURVEY.md section 8 row a9;
// smplx.lbs.lbs tail: T = W.A ; v = T.[v_posed;1]).  HBM-roofline kernels.
//
// Mapping: lane = body.  The work is the flat list of (body group, HV-vertex item) units; every CTA owns a
// contiguous range of it, walks it one body group at a time and gives each warp a contiguous run of the
// group's items, so the load is balanced to one item per warp whatever the batch is.  Everything per-vertex (4 joint ids, 4 weights) is
// warp-uniform; everything per-body lives in registers: the 4 cached joint transforms ("slots") are
// (re)loaded -- three coalesced 512-byte float4 loads from A_blk, L1/L2 resident -- only where the packed
// plan says a slot's joint changes (8 times per 32 vertices on the SMPL mesh order).
//
// Data movement: v_posed comes from the blend GEMM group-blocked, [S/32][n/4][32][4], so the v_posed of an
// item is one contiguous block that a single TMA bulk copy (cp.async.bulk, completion on a per-warp
// mbarrier) brings into shared memory together with the item's 160-byte plan records, one item ahead.  The tensors whose layout the
// caller fixes -- (B, 6890, 3) vertices / vertex gradients -- are transposed through a per-warp
// shared-memory tile [32 bodies][100]: the lane = body side uses 128-bit accesses on its own row, the
// global side moves each 384-byte row segment as 8-byte accesses (two rows per three warp
// instructions), every byte read or written exactly once with streaming accesses.  The backward writes
// dv_posed as bf16 hi/lo 16-byte chunks [S/128][n/8][128][8] (512 contiguous bytes per warp store, the operand
// layout of the gradient GEMM) and adds dA / dtransl into the slab accumulators with fp32 REDs.
#include "lbs_tiles.cuh"

namespace b200smpl {


// contiguous range of the flat (group, item) list owned by this CTA; it is walked one group at a time
struct CtaRange {
  int begin, end;
};
__device__ __forceinline__ CtaRange make_cta_range(int ngroups, int nitems) {
  const long long total = (long long)ngroups * nitems;
  CtaRange r;
  r.begin = (int)(total * blockIdx.x / gridDim.x);
  r.end = (int)(total * (blockIdx.x + 1) / gridDim.x);
  return r;
}

// one lane: v_posed block + plan records of item t -> the warp's buffers, completion counted on `bar`
template <int HV>
__device__ __forceinline__ void issue_item(float4* vbuf, uint32_t* stash, uint64_t* bar, const float4* __restrict__ vp_group,
                                           const uint32_t* __restrict__ vplan, int t) {
  using SH = ItemShape<HV>;
  mbar_expect_tx(bar, SH::TX_BYTES);
  bulk_g2s(vbuf, vp_group + (size_t)t * (SH::NCH4 * 32), SH::VP_WORDS * 4, bar);
  bulk_g2s(stash, vplan + (size_t)t * SH::PLAN_WORDS, SH::PLAN_WORDS * 4, bar);
}
template <int HV>
__device__ __forceinline__ void global_to_tile_scalar(float* tile, const float* src0, size_t row_stride, int nrows,
                                                      int ncols, int lane) {
  for (int r = 0; r < 32; ++r)
    for (int c = lane; c < ItemShape<HV>::ROWS; c += 32)
      tile[r * ItemShape<HV>::HROW + c] = (r < nrows && c < ncols) ? src0[(size_t)r * row_stride + c] : 0.f;
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
constexpr int FWD_RUN = 1;                  // consecutive items per warp and round (slots persist inside a run)
constexpr int FWD_HV = 16;
constexpr int FWD_WARPS = 8;
constexpr int FWD_THREADS = FWD_WARPS * 32;
// per warp: output tile | 2 x (v_posed block, plan records) | 2 mbarriers
constexpr int FWD_WARP_WORDS = ItemShape<FWD_HV>::TILE_WORDS + 2 * (ItemShape<FWD_HV>::VP_WORDS + ItemShape<FWD_HV>::PLAN_WORDS) + 4;
constexpr size_t FWD_SMEM = (size_t)(AG_WORDS + FWD_WARPS * FWD_WARP_WORDS) * 4 + 16;

template <bool HI>
__device__ __forceinline__ void load_slot2(SlotXY& s, SlotZ2& z, const float* A_s, int joint, int lane) {
  const float4* p = reinterpret_cast<const float4*>(A_s) + joint * 96 + lane;
  const float4 q0 = p[0], q1 = p[32], q2 = p[64];
  s.c0 = mk2(q0.x, q0.y); s.c1 = mk2(q0.z, q0.w); s.c2 = mk2(q1.x, q1.y); s.t = mk2(q1.z, q1.w);
  z.r20 = set_half<HI>(z.r20, q2.x); z.r21 = set_half<HI>(z.r21, q2.y);
  z.r22 = set_half<HI>(z.r22, q2.z); z.t2 = set_half<HI>(z.t2, q2.w);
}

// 4 vertices: v_posed from the dense block -> skinned coordinates into the lane's row of the output tile
__device__ __forceinline__ void skin_fwd4(Slots& s, const float* A_s, int lane, const uint32_t* meta_s,
                                          const float4* wts_s, uint32_t force, float tx, float ty, float tz,
                                          const float4* vp_s, float* row_out) {
  const uint4 m4 = *reinterpret_cast<const uint4*>(meta_s);
  const uint32_t mts[4] = {m4.x | force, m4.y, m4.z, m4.w};
  float4 ws[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) ws[i] = wts_s[i];
  float P[12], o[12];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float4 v = vp_s[i * 32];
    P[i * 4] = v.x; P[i * 4 + 1] = v.y; P[i * 4 + 2] = v.z; P[i * 4 + 3] = v.w;
  }
  const f2 txy = mk2(tx, ty), tz0 = mk2(tz, 0.f);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t mt = mts[i];
    const float4 w = ws[i];
    if (mt & (0xFu << 20)) {
      if (mt & (1u << 20)) load_slot2<false>(s.s0, s.zA, A_s, mt & 31, lane);
      if (mt & (1u << 21)) load_slot2<true>(s.s1, s.zA, A_s, (mt >> 5) & 31, lane);
      if (mt & (1u << 22)) load_slot2<false>(s.s2, s.zB, A_s, (mt >> 10) & 31, lane);
      if (mt & (1u << 23)) load_slot2<true>(s.s3, s.zB, A_s, (mt >> 15) & 31, lane);
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

__global__ void __launch_bounds__(FWD_THREADS, 1)
lbs_fwd_kernel(const float4* __restrict__ vpB, int nc4, const float4* __restrict__ A_blk, int b0, int nb, int ngroups,
               const float* __restrict__ transl, float* __restrict__ verts, int V, int nitems, int vec_ok,
               const uint32_t* __restrict__ vplan) {
  constexpr int HV = FWD_HV;
  using SH = ItemShape<HV>;
  extern __shared__ __align__(128) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* A_s = smem;                                               // [24][3][32] float4: the group's transforms
  float* wbase = smem + AG_WORDS + warp * FWD_WARP_WORDS;
  float* tile = wbase;                                             // [32][HROW] output staging
  float4* vbufs = reinterpret_cast<float4*>(wbase + SH::TILE_WORDS);                       // [2][NCH4][32]
  uint32_t* stash = reinterpret_cast<uint32_t*>(wbase + SH::TILE_WORDS + 2 * SH::VP_WORDS);  // [2][PLAN_WORDS]
  uint64_t* wbar = reinterpret_cast<uint64_t*>(wbase + SH::TILE_WORDS + 2 * (SH::VP_WORDS + SH::PLAN_WORDS));  // [2]
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + AG_WORDS + FWD_WARPS * FWD_WARP_WORDS);
  if (lane == 0) {
    mbar_init(&wbar[0], 1);
    mbar_init(&wbar[1], 1);
    if (warp == 0) mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();                 // launched behind the blend GEMM with the PDL attribute: v_posed is complete from here on
  if (threadIdx.x == 0) pdl_trigger();     // the joint kernel behind reads nothing this grid writes: it may fill SMs as CTAs exit
  uint32_t a_phase = 0, n_used = 0;                                // n_used: items this warp has pulled so far
  const CtaRange cta = make_cta_range(ngroups, nitems);
  for (int seg0 = cta.begin; seg0 < cta.end;) {
    // ---- one body group at a time per CTA: its 36 KB of transforms come in with one TMA bulk copy ----
    const int g = seg0 / nitems;
    if (threadIdx.x == 0) {
      mbar_expect_tx(bar, AG_WORDS * 4);
      bulk_g2s(A_s, A_blk + (size_t)g * (AG_WORDS / 4), AG_WORDS * 4, bar);
    }
    const int seg1 = min(cta.end, (g + 1) * nitems);
    const int len = seg1 - seg0;
    // the CTA sweeps the group's items in rounds of FWD_WARPS * FWD_RUN consecutive items, FWD_RUN consecutive
    // items per warp: at any time its warps read / write neighbouring pieces of the same 32 body rows
    const int sb = seg0 - g * nitems;
    auto off_at = [&](int n) { const int r = n / FWD_RUN; return (r * FWD_WARPS + warp) * FWD_RUN + (n - r * FWD_RUN); };
    if (off_at(0) < len) {
      const float4* vp_g = vpB + (size_t)g * nc4 * 32;
      float tx = 0.f, ty = 0.f, tz = 0.f;
      if (transl != nullptr && g * 32 + lane < nb) {
        const float* tp = transl + (size_t)(b0 + g * 32 + lane) * 3;
        tx = tp[0]; ty = tp[1]; tz = tp[2];
      }
      const int nrows = min(32, nb - g * 32);
      float* v_g = verts + (size_t)(b0 + g * 32) * V * 3;
      float* my_row = tile + lane * SH::HROW;
      if (lane == 0) {
        const uint32_t b = n_used & 1;
        issue_item<HV>(vbufs + b * (SH::NCH4 * 32), stash + b * SH::PLAN_WORDS, &wbar[b], vp_g, vplan, sb + off_at(0));
      }
      Slots sl;
      sl.zA.r20 = sl.zA.r21 = sl.zA.r22 = sl.zA.t2 = sl.zB.r20 = sl.zB.r21 = sl.zB.r22 = sl.zB.t2 = mk2(0.f, 0.f);
      mbar_wait(bar, a_phase);
      for (int n = 0;; ++n) {
        const int t = sb + off_at(n);
        if (t >= sb + len) break;
        const int tn = sb + off_at(n + 1);
        const uint32_t b = n_used & 1;
        if (tn < sb + len && lane == 0)                            // next item into the other buffers
          issue_item<HV>(vbufs + (b ^ 1) * (SH::NCH4 * 32), stash + (b ^ 1) * SH::PLAN_WORDS, &wbar[b ^ 1], vp_g, vplan, tn);
        mbar_wait(&wbar[b], (n_used >> 1) & 1);                    // this item's v_posed and plan have landed
        const float4* vp_s = vbufs + b * (SH::NCH4 * 32) + lane;
        const uint32_t* st = stash + b * SH::PLAN_WORDS;
#pragma unroll 1
        for (int u = 0; u < HV / 4; ++u)
          skin_fwd4(sl, A_s, lane, plan_meta(st, u), plan_wts(st, u), (u == 0 && n % FWD_RUN == 0) ? (0xFu << 20) : 0u,
                    tx, ty, tz, vp_s + u * 96, my_row + u * 12);
        __syncwarp();
        // flush: each body row of the item is ROWS contiguous floats of the (B, V, 3) output
        {
          const int vbase = t * HV;
          const int ncols = max(0, min(HV, V - vbase)) * 3;
          float* dst0 = v_g + (size_t)vbase * 3;
          if (!vec_ok) tile_to_global_scalar<HV>(tile, dst0, (size_t)V * 3, nrows, ncols, lane);
          else tile_to_global<HV>(tile, dst0, (size_t)V * 3, nrows, ncols, lane);
        }
        __syncwarp();                                              // tile and buffer b are free again
        ++n_used;
      }
    }
    seg0 = seg1;
    a_phase ^= 1;
    if (seg0 < cta.end) __syncthreads();                           // group switch is CTA-wide: A_s is re-filled
  }
}

// ---------------------------------------------------------------------------------------------
// backward:  given dV, v_posed and A:
//   dv_posed = sum_s w_s R_s^T dV            -> bf16 hi (+lo) chunks of dvp (GEMM operand)
//   dA_j    += w_s [dV (x) p | dV]           -> per-slot register accumulators -> fp32 RED into dA_acc
//   dtransl += dV                            -> fp32 RED into dtr_acc
// The gradient rows are 8-byte aligned only (no TMA): they are copied by cp.async one item ahead into the other
// tile of a double-buffered staging tile.
// ---------------------------------------------------------------------------------------------
constexpr int BWD_HV = 8;
constexpr int BWD_WARPS = 8;
constexpr int BWD_THREADS = BWD_WARPS * 32;
constexpr int BWD_NTILE = 2;                // dV rows arrive by cp.async in a double-buffered tile
constexpr int BWD_WARP_WORDS = BWD_NTILE * ItemShape<BWD_HV>::TILE_WORDS + 2 * (ItemShape<BWD_HV>::VP_WORDS + ItemShape<BWD_HV>::PLAN_WORDS) + 4;
constexpr size_t BWD_SMEM = (size_t)(AG_WORDS + BWD_WARPS * BWD_WARP_WORDS) * 4 + 16;

template <bool HI>
__device__ __forceinline__ void load_rot_half(SlotPair& P, const float* A_s, int joint, int lane) {
  const float4* p = reinterpret_cast<const float4*>(A_s) + joint * 96 + lane;
  const float4 q0 = p[0], q1 = p[32], q2 = p[64];
  P.R[0] = set_half<HI>(P.R[0], q0.x); P.R[3] = set_half<HI>(P.R[3], q0.y);
  P.R[1] = set_half<HI>(P.R[1], q0.z); P.R[4] = set_half<HI>(P.R[4], q0.w);
  P.R[2] = set_half<HI>(P.R[2], q1.x); P.R[5] = set_half<HI>(P.R[5], q1.y);
  P.R[6] = set_half<HI>(P.R[6], q2.x); P.R[7] = set_half<HI>(P.R[7], q2.y); P.R[8] = set_half<HI>(P.R[8], q2.z);
}

// 4 vertices: v_posed from the dense buffer, staged dV of the lane's row -> dv_posed written back in place
// (fp32), accumulators updated
__device__ __forceinline__ void skin_bwd4(BwdState& s, const float* A_s, float* __restrict__ dA_g,
                                          int lane, const uint32_t* meta_s, const float4* wts_s, uint32_t force,
                                          const float4* vp_s, float* row_io) {
  const uint4 m4 = *reinterpret_cast<const uint4*>(meta_s);
  const uint32_t mts[4] = {m4.x | force, m4.y, m4.z, m4.w};
  float P[12], G[12];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float4 v = vp_s[i * 32];
    P[i * 4] = v.x; P[i * 4 + 1] = v.y; P[i * 4 + 2] = v.z; P[i * 4 + 3] = v.w;
    const float4 h = *reinterpret_cast<const float4*>(row_io + i * 4);
    G[i * 4] = h.x; G[i * 4 + 1] = h.y; G[i * 4 + 2] = h.z; G[i * 4 + 3] = h.w;
  }
  float4 w = wts_s[0];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t mt = mts[i];
    const float4 wn = wts_s[i < 3 ? i + 1 : 3];            // next vertex's weights, one vertex ahead
    if (mt & (0xFu << 20)) {
      const uint32_t pv = s.prev;
      if (mt & (1u << 20)) { flush_half<false>(s.A, dA_g, pv & 31, lane); load_rot_half<false>(s.A, A_s, mt & 31, lane); }
      if (mt & (1u << 21)) { flush_half<true>(s.A, dA_g, (pv >> 5) & 31, lane); load_rot_half<true>(s.A, A_s, (mt >> 5) & 31, lane); }
      if (mt & (1u << 22)) { flush_half<false>(s.B, dA_g, (pv >> 10) & 31, lane); load_rot_half<false>(s.B, A_s, (mt >> 10) & 31, lane); }
      if (mt & (1u << 23)) { flush_half<true>(s.B, dA_g, (pv >> 15) & 31, lane); load_rot_half<true>(s.B, A_s, (mt >> 15) & 31, lane); }
    }
    s.prev = mt;
    const f2 px = bc2(P[i * 3]), py = bc2(P[i * 3 + 1]), pz = bc2(P[i * 3 + 2]);
    const float gx = G[i * 3], gy = G[i * 3 + 1], gz = G[i * 3 + 2];
    s.sx += gx; s.sy += gy; s.sz += gz;
    const f2 wA = mk2(w.x, w.y), wB = mk2(w.z, w.w);
    const f2 hxA = mul2(wA, bc2(gx)), hyA = mul2(wA, bc2(gy)), hzA = mul2(wA, bc2(gz));
    const f2 hxB = mul2(wB, bc2(gx)), hyB = mul2(wB, bc2(gy)), hzB = mul2(wB, bc2(gz));
    // dv_posed = sum_slots R^T h   (pair lanes = slots, summed at the end); written over the consumed dV
    f2 qx = fma2(s.A.R[0], hxA, fma2(s.A.R[3], hyA, mul2(s.A.R[6], hzA)));
    f2 qy = fma2(s.A.R[1], hxA, fma2(s.A.R[4], hyA, mul2(s.A.R[7], hzA)));
    f2 qz = fma2(s.A.R[2], hxA, fma2(s.A.R[5], hyA, mul2(s.A.R[8], hzA)));
    qx = fma2(s.B.R[0], hxB, fma2(s.B.R[3], hyB, fma2(s.B.R[6], hzB, qx)));
    qy = fma2(s.B.R[1], hxB, fma2(s.B.R[4], hyB, fma2(s.B.R[7], hzB, qy)));
    qz = fma2(s.B.R[2], hxB, fma2(s.B.R[5], hyB, fma2(s.B.R[8], hzB, qz)));
    G[i * 3] = lo2(qx) + hi2(qx); G[i * 3 + 1] = lo2(qy) + hi2(qy); G[i * 3 + 2] = lo2(qz) + hi2(qz);
    // dA += h (x) [p ; 1]
#define B200_ACC(P_, hx_, hy_, hz_)                                                                  \
  P_.D[0] = fma2(hx_, px, P_.D[0]); P_.D[1] = fma2(hx_, py, P_.D[1]); P_.D[2] = fma2(hx_, pz, P_.D[2]);   \
  P_.D[3] = add2(P_.D[3], hx_);                                                                      \
  P_.D[4] = fma2(hy_, px, P_.D[4]); P_.D[5] = fma2(hy_, py, P_.D[5]); P_.D[6] = fma2(hy_, pz, P_.D[6]);   \
  P_.D[7] = add2(P_.D[7], hy_);                                                                      \
  P_.D[8] = fma2(hz_, px, P_.D[8]); P_.D[9] = fma2(hz_, py, P_.D[9]); P_.D[10] = fma2(hz_, pz, P_.D[10]); \
  P_.D[11] = add2(P_.D[11], hz_);
    B200_ACC(s.A, hxA, hyA, hzA)
    B200_ACC(s.B, hxB, hyB, hzB)
#undef B200_ACC
    w = wn;
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
    *reinterpret_cast<float4*>(row_io + i * 4) = make_float4(G[i * 4], G[i * 4 + 1], G[i * 4 + 2], G[i * 4 + 3]);
}

__global__ void __launch_bounds__(BWD_THREADS, 1)
lbs_bwd_kernel(const float4* __restrict__ vpB, int nc4, const float4* __restrict__ A_blk, int b0, int nb, int ngroups,
               const float* __restrict__ grad_verts, int V, int nitems, int vec_ok,
               const uint32_t* __restrict__ vplan,
               __nv_bfloat16* __restrict__ dvp_hi, __nv_bfloat16* __restrict__ dvp_lo,
               float* __restrict__ dA_acc, float* __restrict__ dtr_acc) {
  constexpr int HV = BWD_HV;
  using SH = ItemShape<HV>;
  extern __shared__ __align__(128) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* A_s = smem;                                                           // the group's transforms
  float* wbase = smem + AG_WORDS + warp * BWD_WARP_WORDS;
  float* tiles = wbase;                                                        // [BWD_NTILE][32][HROW]   dV in / dv_posed out
  float4* vbufs = reinterpret_cast<float4*>(wbase + BWD_NTILE * SH::TILE_WORDS);  // [2][NCH4][32]   v_posed
  uint32_t* stash = reinterpret_cast<uint32_t*>(wbase + BWD_NTILE * SH::TILE_WORDS + 2 * SH::VP_WORDS);
  uint64_t* wbar = reinterpret_cast<uint64_t*>(wbase + BWD_NTILE * SH::TILE_WORDS + 2 * (SH::VP_WORDS + SH::PLAN_WORDS));
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + AG_WORDS + BWD_WARPS * BWD_WARP_WORDS);
  if (lane == 0) {
    mbar_init(&wbar[0], 1);
    mbar_init(&wbar[1], 1);
    if (warp == 0) mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) pdl_trigger();     // the joint kernel behind touches disjoint dvp rows (dA by REDs): it may overlap the tail
  uint32_t a_phase = 0, n_used = 0;
  const size_t row_stride = (size_t)V * 3;
  const CtaRange cta = make_cta_range(ngroups, nitems);
  for (int seg0 = cta.begin; seg0 < cta.end;) {
    const int g = seg0 / nitems;
    if (threadIdx.x == 0) {
      mbar_expect_tx(bar, AG_WORDS * 4);
      bulk_g2s(A_s, A_blk + (size_t)g * (AG_WORDS / 4), AG_WORDS * 4, bar);
    }
    const int seg1 = min(cta.end, (g + 1) * nitems);
    const int len = seg1 - seg0;
    const int it0 = seg0 - g * nitems + len * warp / BWD_WARPS;               // this warp's contiguous items
    const int it1 = seg0 - g * nitems + len * (warp + 1) / BWD_WARPS;
    if (it0 < it1) {
      float* dA_g = dA_acc + (size_t)g * AG_WORDS;
      const float4* vp_g = vpB + (size_t)g * nc4 * 32;
      const float* dv_g = grad_verts + (size_t)(b0 + g * 32) * V * 3;
      const int nrows = max(0, min(32, nb - g * 32));
      if (lane == 0) {
        const uint32_t b = n_used & 1;
        issue_item<HV>(vbufs + b * (SH::NCH4 * 32), stash + b * SH::PLAN_WORDS, &wbar[b], vp_g, vplan, it0);
      }
      // first item's gradient rows
      int tb = 0;
      if (vec_ok) issue_rows<HV>(tiles, dv_g + (size_t)it0 * HV * 3, row_stride, nrows, max(0, min(HV, V - it0 * HV)) * 3, lane);
      cp_async_commit();
      if (!vec_ok)
        global_to_tile_scalar<HV>(tiles, dv_g + (size_t)it0 * HV * 3, row_stride, nrows, max(0, min(HV, V - it0 * HV)) * 3, lane);
      BwdState st;
#pragma unroll
      for (int e = 0; e < AELEMS; ++e) st.A.D[e] = st.B.D[e] = mk2(0.f, 0.f);
#pragma unroll
      for (int e = 0; e < 9; ++e) st.A.R[e] = st.B.R[e] = mk2(0.f, 0.f);
      st.prev = 0u;
      st.sx = st.sy = st.sz = 0.f;
      __syncwarp();
      mbar_wait(bar, a_phase);
      for (int t = it0; t < it1; ++t) {
        const bool more = t + 1 < it1;
        const uint32_t b = n_used & 1;
        float* tile = tiles + tb * SH::TILE_WORDS;
        float* my_row = tile + lane * SH::HROW;
        if (more) {                                               // next item: TMA for v_posed + plan, dV rows
          if (lane == 0)
            issue_item<HV>(vbufs + (b ^ 1) * (SH::NCH4 * 32), stash + (b ^ 1) * SH::PLAN_WORDS, &wbar[b ^ 1], vp_g, vplan, t + 1);
          if (vec_ok)
            issue_rows<HV>(tiles + (tb ^ 1) * SH::TILE_WORDS, dv_g + (size_t)(t + 1) * HV * 3, row_stride, nrows,
                           max(0, min(HV, V - (t + 1) * HV)) * 3, lane);
        }
        cp_async_commit();
        cp_async_wait<1>();
        __syncwarp();                                              // this item's dV rows were copied by other lanes
        mbar_wait(&wbar[b], (n_used >> 1) & 1);
        const float4* vp_s = vbufs + b * (SH::NCH4 * 32) + lane;
        const uint32_t* ps = stash + b * SH::PLAN_WORDS;
        // the first vertex of the run (re)loads all four slots; the accumulators are zero there
#pragma unroll 1
        for (int u = 0; u < HV / 4; ++u)
          skin_bwd4(st, A_s, dA_g, lane, plan_meta(ps, u), plan_wts(ps, u), (u == 0 && t == it0) ? (0xFu << 20) : 0u,
                    vp_s + u * 96, my_row + u * 12);
        // ---- the lane's gradient rows -> bf16 hi/lo chunks of dvp (512 contiguous bytes per warp store) ----
        {
          // dvp [S/128][n_pad/8][128][8]: chunk stride 1024 elements, this body at ((g & 3) * 32 + lane) * 8
          const size_t o0 = (((size_t)(g >> 2) * (nc4 >> 1) + t * SH::NCH8) * 128 + (g & 3) * 32 + lane) * 8;
#pragma unroll
          for (int c = 0; c < SH::NCH8; ++c) {
            const float4 x = *reinterpret_cast<const float4*>(my_row + c * 8);
            const float4 y = *reinterpret_cast<const float4*>(my_row + c * 8 + 4);
            const float ch[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
            store_dvp_chunk(ch, dvp_hi + o0 + c * 1024, dvp_lo ? dvp_lo + o0 + c * 1024 : nullptr);
          }
        }
        __syncwarp();                                              // every lane is done with its row of the tile
        if (more && !vec_ok)
          global_to_tile_scalar<HV>(tiles + (tb ^ 1) * SH::TILE_WORDS, dv_g + (size_t)(t + 1) * HV * 3, row_stride, nrows,
                                    max(0, min(HV, V - (t + 1) * HV)) * 3, lane);
        tb ^= 1;
        __syncwarp();                                              // the next item's rows were written by other lanes
        ++n_used;
      }
      bwd_close_group(st, dA_g, dtr_acc + (size_t)g * 96, lane);
    }
    seg0 = seg1;
    a_phase ^= 1;
    if (seg0 < cta.end) __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
static int run_grid(int ngroups, int nitems, int warps, int num_sms) {
  const long long total = (long long)ngroups * nitems;
  return (int)std::max<long long>(1, std::min<long long>(num_sms, (total + warps - 1) / warps));
}

int launch_lbs_fwd(const DevModel& m, const float* vpB, int S, const float* A_blk, int b0, int nb,
                   const float* transl, float* verts, int num_sms, cudaStream_t st) {
  if (nb <= 0) return 0;
  const int groups = (nb + 31) / 32;
  const int nitems = m.ntiles * (TILE_V / FWD_HV);
  const int vec_ok = ((m.V & 1) == 0 && (reinterpret_cast<uintptr_t>(verts) & 7) == 0) ? 1 : 0;
  B200_SMEM_ATTR_ONCE(lbs_fwd_kernel, FWD_SMEM);
  LaunchTimer _timer("lbs_fwd", st);
  B200_CUDA_TRY(launch_k(lbs_fwd_kernel, dim3(run_grid(groups, nitems, FWD_WARPS, num_sms)), dim3(FWD_THREADS), FWD_SMEM, st, true,
                         reinterpret_cast<const float4*>(vpB), m.n_pad / 4, reinterpret_cast<const float4*>(A_blk), b0, nb, groups,
                         transl, verts, m.V, nitems, vec_ok, m.vplan));
  B200_LAUNCH_CHECK("lbs_fwd");
  return 0;
}

// Sw = active slab width (multiple of 32, >= nb): rows of absent bodies get zero dvp
// dA_acc [S/32][288][32] and dtr_acc [S/32][3][32] must be zeroed by the caller; warps add into them
int launch_lbs_bwd(const DevModel& m, const float* vpB, int S, int Sw, const float* A_blk, int b0, int nb,
                   const float* grad_verts, __nv_bfloat16* dvp_hi, __nv_bfloat16* dvp_lo, float* dA_acc,
                   float* dtr_acc, int num_sms, cudaStream_t st) {
  const int groups = Sw / 32;
  const int nitems = m.ntiles * (TILE_V / BWD_HV);
  const int vec_ok = ((m.V & 1) == 0 && (reinterpret_cast<uintptr_t>(grad_verts) & 7) == 0) ? 1 : 0;
  B200_SMEM_ATTR_ONCE(lbs_bwd_kernel, BWD_SMEM);
  LaunchTimer _timer("lbs_bwd", st);
  lbs_bwd_kernel<<<run_grid(groups, nitems, BWD_WARPS, num_sms), BWD_THREADS, BWD_SMEM, st>>>(
      reinterpret_cast<const float4*>(vpB), m.n_pad / 4, reinterpret_cast<const float4*>(A_blk), b0, nb, groups, grad_verts, m.V,
      nitems, vec_ok, m.vplan, dvp_hi, dvp_lo, dA_acc, dtr_acc);
  B200_LAUNCH_CHECK("lbs_bwd");
  return 0;
}

}  // namespace b200smpl
