// Joint outputs (SURVEY.md section 8 rows a2, a5, a10): the 66 non-chain joints of the 90-joint
// superset of models/smpl_official.py:27-41 -- 21 joints picked from vertices (smplx
// VertexJointSelector) and 45 joints regressed from vertices (J_regressor_extra / cocoplus / h36m).
//
// No vertex is re-read: a regressed joint  sum_v Jr[j][v] * skin(v)  is rewritten at pack time as
//   sum_i  A_i . [ q_ji ; c_ji ],   q_ji = sum_v Jr[j][v] w_vi p_v  (linear in the blend features),
// so the q_ji are extra "virtual" rows of the blend GEMM, grouped 32 q-groups (96 rows) per virtual
// tile, and a joint costs a handful of 3x4 transforms.  These kernels are the skinning kernels of
// lbs.cu specialised to virtual tiles: lane = body, CTAs of (body group, a few virtual tiles) with the group's
// transforms in shared memory (one TMA bulk copy), four warps per virtual tile (8 q-groups each), q rows read as
// float4 from the blend output, the warp-uniform plan words held one per lane and broadcast with shuffles, the
// warps' partial sums added through shared tiles and written as contiguous row segments of joints (B, 90, 3);
// the backward emits dq as 16-byte dvp chunks and adds dA / dtransl with fp32 REDs.  The 24 chain joints are written by the pose kernel; reprojection is
// the orthographic kernel.
#include "skin_common.cuh"

namespace b200smpl {

constexpr int JW = 8;                       // warps per CTA
constexpr int JQ = 4;                       // warps per virtual tile: each takes 8 of its 32 q-groups (24 rows = 3 dvp chunks)
constexpr int JTL = JW / JQ;                // virtual tiles per CTA
constexpr int JT = JW * 32;

// 8 q-groups = 24 rows = 6 float4 of one body
__device__ __forceinline__ void load_q24(float (&q)[24], const float4* __restrict__ p) {
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const float4 v = ld_stream4(p + i * 32);
    q[i * 4] = v.x; q[i * 4 + 1] = v.y; q[i * 4 + 2] = v.z; q[i * 4 + 3] = v.w;
  }
}
// transforms from the shared-memory copy of the group (paired layout, skin_common.cuh)
__device__ __forceinline__ void load_slot_s(float (&a)[AELEMS], const float* A_s, int joint, int lane) {
  const float4* p = reinterpret_cast<const float4*>(A_s) + joint * 96 + lane;
  unpack_transform(a, p[0], p[32], p[64]);
}
// the four warps of one virtual tile meet on their own named barrier (0 is __syncthreads)
__device__ __forceinline__ void quartet_sync(int tl) { asm volatile("bar.sync %0, 128;" ::"r"(1 + tl) : "memory"); }

// A virtual tile (32 q-groups) is shared by four warps, eight q-groups each: the per-warp instruction chain is what
// bounds these kernels (they move ~10 KB per body), so four short chains instead of one long one.
// dynamic shared memory: A_s [24][3][32] float4 | JW partial tiles [32][pitch] | mbarrier
__global__ void __launch_bounds__(JT, 1024 / JT)
joints_fwd_kernel(DevModel m, const float4* __restrict__ vpB, int nc4, const float4* __restrict__ A_blk, int b0, int nb,
                  int pitch, const float* __restrict__ transl, float* __restrict__ joints) {
  extern __shared__ __align__(128) float smem[];
  float* A_s = smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tl = warp / JQ, qt = warp % JQ;
  float* my_row = smem + AG_WORDS + warp * 32 * pitch + lane * pitch;   // this warp's partial sums of the lane's body
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + AG_WORDS + JW * 32 * pitch + ((JW * 32 * pitch) & 1));
  const int g = blockIdx.x;
  if (threadIdx.x == 0) fetch_group_transforms(A_s, reinterpret_cast<const float*>(A_blk), g, bar);
  const int tv = blockIdx.y * JTL + tl;
  const bool on = tv < m.ntv;                                // uniform over the tile's four warps
  float q[24];
  uint32_t mt_l = 0;
  float c_l = 0.f;
  int ncols = 0;
  if (on) {
    load_q24(q, vpB + ((size_t)g * nc4 + (m.ntiles + tv) * 24 + qt * 6) * 32 + lane);
    mt_l = __ldg(m.qmeta + tv * 32 + qt * 8 + (lane & 7));   // lane i holds the plan of q-group qt * 8 + (i & 7)
    c_l = __ldg(m.qcoef + tv * 32 + qt * 8 + (lane & 7));
    float tx = 0.f, ty = 0.f, tz = 0.f;
    if (qt == 0 && transl != nullptr && g * 32 + lane < nb) {
      const float* t = transl + (size_t)(b0 + g * 32 + lane) * 3;
      tx = t[0]; ty = t[1]; tz = t[2];
    }
    // every output joint of the tile starts at the translation (first warp) and accumulates its terms in the lane's row
    ncols = m.vt_nj[tv] * 3;
    for (int c = 0; c < ncols; c += 3) { my_row[c] = tx; my_row[c + 1] = ty; my_row[c + 2] = tz; }
  }
  __syncthreads();                                           // barrier init visible to every waiter
  if (on) {
    mbar_wait(bar, 0);
    float a[AELEMS];
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      const uint32_t mt = __shfl_sync(0xffffffffu, mt_l, ii);
      if (!(mt & (1u << 14))) continue;                      // dummy groups pad the END of a tile
      if (ii == 0 || (mt & (1u << 5))) load_slot_s(a, A_s, mt & 31, lane);   // groups are sorted by skinning joint
      const float c = __shfl_sync(0xffffffffu, c_l, ii);
      const float qx = q[ii * 3], qy = q[ii * 3 + 1], qz = q[ii * 3 + 2];
      float* o = my_row + ((mt >> 8) & 31) * 3;
      o[0] += fmaf(a[0], qx, fmaf(a[1], qy, fmaf(a[2], qz, a[3] * c)));
      o[1] += fmaf(a[4], qx, fmaf(a[5], qy, fmaf(a[6], qz, a[7] * c)));
      o[2] += fmaf(a[8], qx, fmaf(a[9], qy, fmaf(a[10], qz, a[11] * c)));
    }
    quartet_sync(tl);
    // flush: this warp sums the four partials of 8 body rows (4 lanes per row) -> 3 nj contiguous floats per body
    const int r = qt * 8 + (lane >> 2);
    if (g * 32 + r < nb) {
      const float* p0 = smem + AG_WORDS + (tl * JQ) * 32 * pitch + r * pitch;
      float* dst = joints + (size_t)(b0 + g * 32 + r) * m.njout * 3 + (size_t)(NJ + m.vt_j0[tv]) * 3;
      for (int c = lane & 3; c < ncols; c += 4)
        dst[c] = (p0[c] + p0[32 * pitch + c]) + (p0[64 * pitch + c] + p0[96 * pitch + c]);
    }
  }
  // launched behind lbs_fwd with the PDL attribute and no wait up front (nothing read here is written by it): the
  // grid must not complete before its predecessor has
  pdl_wait();
}

// backward over virtual tiles.  dJ: total joint gradient (B, NJout, 3).
//   dq -> virtual rows of dvp ; dA, dtransl -> fp32 REDs into the slab accumulators
// dynamic shared memory: A_s | JTL gradient tiles [32][pitch] | mbarrier
__global__ void __launch_bounds__(JT, 768 / JT)
joints_bwd_kernel(DevModel m, const float4* __restrict__ vpB, int nc4, const float4* __restrict__ A_blk, int b0, int nb,
                  int pitch, const float* __restrict__ dJ, __nv_bfloat16* __restrict__ dvp_hi,
                  __nv_bfloat16* __restrict__ dvp_lo, float* __restrict__ dA_acc, float* __restrict__ dtr_acc) {
  extern __shared__ __align__(128) float smem[];
  float* A_s = smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tl = warp / JQ, qt = warp % JQ;
  float* tile = smem + AG_WORDS + tl * 32 * pitch;           // the tile's joint gradients, shared by its four warps
  const float* my_row = tile + lane * pitch;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + AG_WORDS + JTL * 32 * pitch + ((JTL * 32 * pitch) & 1));
  const int g = blockIdx.x;
  if (threadIdx.x == 0) fetch_group_transforms(A_s, reinterpret_cast<const float*>(A_blk), g, bar);
  const int tv = blockIdx.y * JTL + tl;
  const bool on = tv < m.ntv;                                // uniform over the tile's four warps
  float q[24];
  uint32_t mt_l = 0;
  float c_l = 0.f;
  int ncols = 0;
  if (on) {
    load_q24(q, vpB + ((size_t)g * nc4 + (m.ntiles + tv) * 24 + qt * 6) * 32 + lane);
    mt_l = __ldg(m.qmeta + tv * 32 + qt * 8 + (lane & 7));
    c_l = __ldg(m.qcoef + tv * 32 + qt * 8 + (lane & 7));
    ncols = m.vt_nj[tv] * 3;
    {  // stage the gradients of this tile's joints (3 nj floats of each body row): 8 rows per warp, 4 lanes per row
      const int r = qt * 8 + (lane >> 2);
      const bool live = g * 32 + r < nb;
      const float* src = dJ + (size_t)(b0 + g * 32 + r) * m.njout * 3 + (size_t)(NJ + m.vt_j0[tv]) * 3;
      float* trow = tile + r * pitch;
      for (int c0 = lane & 3; c0 < ncols; c0 += 16) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (live && c0 + u * 4 < ncols) ? ld_stream(src + c0 + u * 4) : 0.f;
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (c0 + u * 4 < ncols) trow[c0 + u * 4] = v[u];
      }
    }
  }
  __syncthreads();                                           // barrier init visible; every tile staged
  if (on) {
    mbar_wait(bar, 0);
    if (qt == 0) {                                           // dL/dtransl: every output joint of the tile once
      float sx = 0.f, sy = 0.f, sz = 0.f;
      for (int c = 0; c < ncols; c += 3) { sx += my_row[c]; sy += my_row[c + 1]; sz += my_row[c + 2]; }
      float* dtr_g = dtr_acc + (size_t)g * 96;
      red_add(dtr_g + lane, sx);
      red_add(dtr_g + 32 + lane, sy);
      red_add(dtr_g + 64 + lane, sz);
    }
    float* dA_g = dA_acc + (size_t)g * AG_WORDS;
    float a[AELEMS], d[AELEMS], dq[24];
#pragma unroll
    for (int e = 0; e < AELEMS; ++e) d[e] = 0.f;
    int jcur = 0;
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      const uint32_t mt = __shfl_sync(0xffffffffu, mt_l, ii);
      if (!(mt & (1u << 14))) {                              // dummy slot: its dvp rows must be 0
        dq[ii * 3] = dq[ii * 3 + 1] = dq[ii * 3 + 2] = 0.f;
        continue;
      }
      if (ii == 0 || (mt & (1u << 5))) {                     // next skinning joint: close the accumulators of the last
        if (ii != 0) flush_slot_g(d, dA_g, jcur, lane);
        jcur = mt & 31;
        load_slot_s(a, A_s, jcur, lane);
      }
      const float c = __shfl_sync(0xffffffffu, c_l, ii);
      const float* gj = my_row + ((mt >> 8) & 31) * 3;
      const float gx = gj[0], gy = gj[1], gz = gj[2];
      const float qx = q[ii * 3], qy = q[ii * 3 + 1], qz = q[ii * 3 + 2];
      dq[ii * 3] = fmaf(a[0], gx, fmaf(a[4], gy, a[8] * gz));
      dq[ii * 3 + 1] = fmaf(a[1], gx, fmaf(a[5], gy, a[9] * gz));
      dq[ii * 3 + 2] = fmaf(a[2], gx, fmaf(a[6], gy, a[10] * gz));
      d[0] = fmaf(gx, qx, d[0]); d[1] = fmaf(gx, qy, d[1]); d[2] = fmaf(gx, qz, d[2]); d[3] = fmaf(gx, c, d[3]);
      d[4] = fmaf(gy, qx, d[4]); d[5] = fmaf(gy, qy, d[5]); d[6] = fmaf(gy, qz, d[6]); d[7] = fmaf(gy, c, d[7]);
      d[8] = fmaf(gz, qx, d[8]); d[9] = fmaf(gz, qy, d[9]); d[10] = fmaf(gz, qz, d[10]); d[11] = fmaf(gz, c, d[11]);
    }
    const size_t chunk0 = (size_t)(g >> 2) * (nc4 >> 1) + (size_t)((m.ntiles + tv) * 12 + qt * 3);
    __nv_bfloat16* hi_p = dvp_hi + (chunk0 * 128 + (g & 3) * 32 + lane) * 8;
    __nv_bfloat16* lo_p = dvp_lo ? dvp_lo + (chunk0 * 128 + (g & 3) * 32 + lane) * 8 : nullptr;
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      const float ch[8] = {dq[cc * 8], dq[cc * 8 + 1], dq[cc * 8 + 2], dq[cc * 8 + 3],
                           dq[cc * 8 + 4], dq[cc * 8 + 5], dq[cc * 8 + 6], dq[cc * 8 + 7]};
      const size_t off = (size_t)cc * 128 * 8;
      store_dvp_chunk(ch, hi_p + off, lo_p ? lo_p + off : nullptr);
    }
    if (__shfl_sync(0xffffffffu, mt_l, 0) & (1u << 14)) flush_slot_g(d, dA_g, jcur, lane);   // not for a quarter of padding
  }
  pdl_wait();                 // as in the forward: complete only after lbs_bwd (the gradient GEMM behind needs both)
}

// total joint gradient when a 2D reprojection gradient is present:
//   dJ = grad_joints + [s g2d_x, s g2d_y, 0] ;  dcam = [sum g2d.(xy + t), s sum g2d_x, s sum g2d_y]
__global__ void __launch_bounds__(128)
joint_grad_total_kernel(const float* __restrict__ joints, const float* __restrict__ cam,
                        const float* __restrict__ gj, const float* __restrict__ g2d, float* __restrict__ dJ,
                        float* __restrict__ gcam, int nj) {
  __shared__ float sh[3][4];
  const int b = blockIdx.x;
  const float s = cam[b * 3], tx = cam[b * 3 + 1], ty = cam[b * 3 + 2];
  float gs = 0.f, gtx = 0.f, gty = 0.f;
  for (int j = threadIdx.x; j < nj; j += blockDim.x) {
    const size_t o3 = ((size_t)b * nj + j) * 3, o2 = ((size_t)b * nj + j) * 2;
    const float gu = g2d[o2], gv = g2d[o2 + 1];
    dJ[o3] = (gj ? gj[o3] : 0.f) + s * gu;
    dJ[o3 + 1] = (gj ? gj[o3 + 1] : 0.f) + s * gv;
    dJ[o3 + 2] = gj ? gj[o3 + 2] : 0.f;
    gs += gu * (joints[o3] + tx) + gv * (joints[o3 + 1] + ty);
    gtx += s * gu;
    gty += s * gv;
  }
  float v[3] = {gs, gtx, gty};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = v[k];
  }
  __syncthreads();
  if (gcam != nullptr && threadIdx.x < 3) gcam[b * 3 + threadIdx.x] = sh[threadIdx.x][0] + sh[threadIdx.x][1] + sh[threadIdx.x][2] + sh[threadIdx.x][3];
}

// CTAs per body group: JTL virtual tiles per CTA, four warps each
static int joints_split(int ntv) { return std::max(1, (ntv + JTL - 1) / JTL); }
static size_t joints_smem(int ntiles_s, int pitch) { return (size_t)(AG_WORDS + ntiles_s * 32 * pitch + 1) * 4 + 16; }

// after_lbs: the previous kernel in the stream is the skinning kernel of the same slab -> PDL launch (overlaps its tail)
int launch_joints_fwd(const DevModel& m, const float* vpB, int S, const float* A_blk, int b0, int nb,
                      const float* transl, float* joints, bool after_lbs, cudaStream_t st) {
  if (nb <= 0 || m.ntv == 0) return 0;
  const int groups = (nb + 31) / 32;
  const int pitch = m.vt_maxcols | 1;
  const size_t smem = joints_smem(JW, pitch);
  B200_SMEM_ATTR_ONCE(joints_fwd_kernel, smem);
  LaunchTimer _timer("joints_fwd", st);
  B200_CUDA_TRY(launch_k(joints_fwd_kernel, dim3(groups, joints_split(m.ntv)), dim3(JT), smem, st, after_lbs, m,
                         reinterpret_cast<const float4*>(vpB), m.n_pad / 4, reinterpret_cast<const float4*>(A_blk), b0, nb, pitch,
                         transl, joints));
  B200_LAUNCH_CHECK("joints_fwd");
  return 0;
}

// Sw: active slab width (multiple of 32); absent bodies get zero dvp rows.
int launch_joints_bwd(const DevModel& m, const float* vpB, int S, int Sw, const float* A_blk, int b0, int nb,
                      const float* dJ, __nv_bfloat16* dvp_hi, __nv_bfloat16* dvp_lo, float* dA_acc, float* dtr_acc,
                      bool after_lbs, cudaStream_t st) {
  if (m.ntv == 0) return 0;
  const int groups = Sw / 32;
  const int pitch = m.vt_maxcols | 1;
  const size_t smem = joints_smem(JTL, pitch);
  B200_SMEM_ATTR_ONCE(joints_bwd_kernel, smem);
  LaunchTimer _timer("joints_bwd", st);
  B200_CUDA_TRY(launch_k(joints_bwd_kernel, dim3(groups, joints_split(m.ntv)), dim3(JT), smem, st, after_lbs, m,
                         reinterpret_cast<const float4*>(vpB), m.n_pad / 4, reinterpret_cast<const float4*>(A_blk), b0, nb, pitch,
                         dJ, dvp_hi, dvp_lo, dA_acc, dtr_acc));
  B200_LAUNCH_CHECK("joints_bwd");
  return 0;
}

int launch_joint_grad_total(const float* joints, const float* cam, const float* gj, const float* g2d, float* dJ,
                            float* gcam, int B, int nj, cudaStream_t st) {
  LaunchTimer _timer("joint_grad_total", st);
  joint_grad_total_kernel<<<B, 128, 0, st>>>(joints, cam, gj, g2d, dJ, gcam, nj);
  B200_LAUNCH_CHECK("joint_grad_total");
  return 0;
}

}  // namespace b200smpl
