// Pose stage (SURVEY.md section 8 rows a6, a7 (feature), a8): Rodrigues, rest joints, pose
// feature, the 24-joint kinematic chain and the skinning transforms A = [G_R | G_t - G_R J].
//
// Lane = body: one CTA (16 warps) per 32-body group, each lane holds one body.  The chain G_j = G_parent(j) . L_j
// is walked one tree level at a time (9 levels on the SMPL tree), one warp per joint of the level, instead of the
// reference's 23-iteration Python loop of batched matmuls (smplx.lbs.batch_rigid_transform).  There is no shuffle,
// no divergence and no idle lane.  Per-joint state that is indexed dynamically (local rotations, global transforms,
// rest joints, gradient accumulators) lives in shared memory as [row][lane] (conflict-free); the group-blocked
// operands of the skinning kernels (A_blk, dA) are read / written straight from registers, coalesced; row-major
// per-body tensors (pose, grad_pose) go through a transposing stage.  Rest joints use the pack-time folds
// J_template = J_regressor.v_template, J_shapedirs = J_regressor.shapedirs.
#include "common.cuh"
#include "rodrigues.cuh"
#include "skin_common.cuh"

namespace b200smpl {

// G <- P . G   for 3x4 affine matrices [R|t] (implicit last row 0 0 0 1)
__device__ __forceinline__ void compose(const float P[12], float G[12]) {
  float o[12];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c) o[r * 4 + c] = P[r * 4] * G[c] + P[r * 4 + 1] * G[4 + c] + P[r * 4 + 2] * G[8 + c];
    o[r * 4 + 3] = P[r * 4] * G[3] + P[r * 4 + 1] * G[7] + P[r * 4 + 2] * G[11] + P[r * 4 + 3];
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) G[i] = o[i];
}

__device__ __forceinline__ __nv_bfloat16 bf_hi(float x) { return __float2bfloat16_rn(x); }
__device__ __forceinline__ __nv_bfloat16 bf_lo(float x, __nv_bfloat16 hi) {
  return __float2bfloat16_rn(x - __bfloat162float(hi));
}

constexpr int LB_P = 33;                     // pitch of the transposed staging rows
constexpr int LB_MAXB = 20;                  // betas that fit slab 0 of the feature layout

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

constexpr int LBF_THREADS = 512;
struct LbFwdSmem {
  float R[NJ * 9 * LB_P];        // local rotations [joint * 9 + e][body]
  float AAx[NJ * 3 * LB_P];      // axis-angle input
  float G[NJ * 12 * 32];         // global transforms, row-major [R | t]
  float J[NJ * 3 * 32];          // rest joints
  float B[LB_MAXB * 32];         // betas
  float T[3 * 32];               // translation
  float Jsd[NJ * 3 * LB_MAXB];
  float Jt[NJ * 3];
};

// ---- forward, lane = body.  One CTA (16 warps) per 32-body group:
//   P1 all threads: pose rows (transposed through registers), betas, translation, model constants;
//   P2 all threads: rest joints (and Rodrigues for axis-angle input);
//   P3 level by level, one warp per joint, each lane ITS body: G_j = G_parent . [R_j | Jr_j - Jr_parent];
//   P4 all threads: A = [G_R | G_t - G_R Jr] as coalesced float4, posed joints, the bf16 hi / lo feature row.
template <bool AA>
__global__ void __launch_bounds__(LBF_THREADS, 1)
pose_fwd_lb_kernel(DevModel m, const float* __restrict__ betas, const float* __restrict__ pose, int b0, int nb, int S,
                   __nv_bfloat16* __restrict__ feat, float* __restrict__ featf, float* __restrict__ A_T,
                   const float* __restrict__ transl, float* __restrict__ joints) {
  extern __shared__ __align__(16) unsigned char lbraw_[];
  LbFwdSmem& sm = *reinterpret_cast<LbFwdSmem*>(lbraw_);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = blockIdx.x;
  constexpr int NW = LBF_THREADS / 32;
  const int nlive = max(0, min(32, nb - g * 32));
  const bool live = lane < nlive;
  const FeatLayout fl = m.fl;
  const int nbeta = fl.nb;
  const size_t body0 = (size_t)b0 + (size_t)g * 32;
  (void)S;
  if (tid == 0) pdl_trigger();          // the blend GEMM behind may set itself up; it waits for this grid's completion
  // ---------------- P1 ----------------
  {
    constexpr int PWc = AA ? NJ * 3 : NJ * 9;
    constexpr int PIT = (32 * PWc / 4 + LBF_THREADS - 1) / LBF_THREADS;
    float* dstT = AA ? sm.AAx : sm.R;
    const bool al = (reinterpret_cast<uintptr_t>(pose) & 15) == 0;
    float4 pv[PIT];
    const float4* src4 = reinterpret_cast<const float4*>(pose + body0 * PWc);
    const int n4 = nlive * PWc / 4;
#pragma unroll
    for (int it = 0; it < PIT; ++it) {
      const int i = tid + it * LBF_THREADS;
      pv[it] = (al && i < n4) ? src4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float bv = 0.f, tv = 0.f;
    if (tid < 32 * nbeta && tid / nbeta < nlive) bv = betas[body0 * nbeta + tid];
    if (transl != nullptr && tid < 96 && tid / 3 < nlive) tv = transl[body0 * 3 + tid];
    for (int i = tid; i < NJ * 3 * nbeta; i += LBF_THREADS) sm.Jsd[i] = m.Jsd[i];
    if (tid < NJ * 3) sm.Jt[tid] = m.Jt[tid];
#pragma unroll
    for (int it = 0; it < PIT; ++it) {
      const int i = tid + it * LBF_THREADS;
      if (al && i < n4) {
        const float x[4] = {pv[it].x, pv[it].y, pv[it].z, pv[it].w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = i * 4 + u, body = e / PWc, k = e - body * PWc;
          dstT[k * LB_P + body] = x[u];
        }
      }
    }
    if (!al) {
      const float* src = pose + body0 * PWc;
      for (int i = tid; i < nlive * PWc; i += LBF_THREADS) {
        const int body = i / PWc, k = i - body * PWc;
        dstT[k * LB_P + body] = src[i];
      }
    }
    if (tid < 32 * nbeta) sm.B[(tid % nbeta) * 32 + tid / nbeta] = bv;
    if (tid < 96) sm.T[(tid % 3) * 32 + tid / 3] = tv;
  }
  __syncthreads();
  // ---------------- P2 ----------------
  for (int k = warp; k < NJ * 3; k += NW) {
    float acc = sm.Jt[k];
    for (int l = 0; l < nbeta; ++l) acc = fmaf(sm.Jsd[k * nbeta + l], sm.B[l * 32 + lane], acc);
    sm.J[k * 32 + lane] = acc;
  }
  for (int j = warp; j < NJ; j += NW) {
    if (AA) {
      float r[3] = {0.f, 0.f, 0.f}, R[9];
      if (live) { r[0] = sm.AAx[(j * 3) * LB_P + lane]; r[1] = sm.AAx[(j * 3 + 1) * LB_P + lane]; r[2] = sm.AAx[(j * 3 + 2) * LB_P + lane]; }
      rodrigues_fwd(r, R);
#pragma unroll
      for (int e = 0; e < 9; ++e) sm.R[(j * 9 + e) * LB_P + lane] = R[e];
    } else if (!live) {
#pragma unroll
      for (int e = 0; e < 9; ++e) sm.R[(j * 9 + e) * LB_P + lane] = (e == 0 || e == 4 || e == 8) ? 1.f : 0.f;
    }
  }
  __syncthreads();
  // ---------------- P3: one tree level at a time, one warp per joint of the level (9 levels on the SMPL tree
  // instead of 24 dependent steps on one warp) ----------------
#pragma unroll 1
  for (int dpt = 0; dpt <= m.chain.maxdepth; ++dpt) {
    for (int i = m.chain.level_ptr[dpt] + warp; i < m.chain.level_ptr[dpt + 1]; i += NW) {
      const int j = m.chain.order[i];
      const int p = m.chain.parent[j];
      float G[12];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) G[r * 4 + c] = sm.R[(j * 9 + r * 3 + c) * LB_P + lane];
        G[r * 4 + 3] = sm.J[(j * 3 + r) * 32 + lane];
      }
      if (p >= 0) {
        float P[12];
#pragma unroll
        for (int e = 0; e < 12; ++e) P[e] = sm.G[(p * 12 + e) * 32 + lane];
#pragma unroll
        for (int r = 0; r < 3; ++r) G[r * 4 + 3] -= sm.J[(p * 3 + r) * 32 + lane];
        compose(P, G);
      }
#pragma unroll
      for (int e = 0; e < 12; ++e) sm.G[(j * 12 + e) * 32 + lane] = G[e];
    }
    __syncthreads();
  }
  // ---------------- P4 ----------------
  {
    float4* A4 = reinterpret_cast<float4*>(A_T) + (size_t)g * (NJ * 3 * 32) + lane;
    const float z = live ? 1.f : 0.f;
    for (int j = warp; j < NJ; j += NW) {
      float G[12], Jr[3], t[3];
#pragma unroll
      for (int e = 0; e < 12; ++e) G[e] = sm.G[(j * 12 + e) * 32 + lane];
#pragma unroll
      for (int k = 0; k < 3; ++k) Jr[k] = sm.J[(j * 3 + k) * 32 + lane];
#pragma unroll
      for (int r = 0; r < 3; ++r) t[r] = G[r * 4 + 3] - (G[r * 4] * Jr[0] + G[r * 4 + 1] * Jr[1] + G[r * 4 + 2] * Jr[2]);
      A4[(j * 3 + 0) * 32] = make_float4(z * G[0], z * G[4], z * G[1], z * G[5]);
      A4[(j * 3 + 1) * 32] = make_float4(z * G[2], z * G[6], z * t[0], z * t[1]);
      A4[(j * 3 + 2) * 32] = make_float4(z * G[8], z * G[9], z * G[10], z * t[2]);
      if (joints != nullptr && live) {
        float* o = joints + ((body0 + lane) * m.njout + j) * 3;
        o[0] = G[3] + sm.T[lane]; o[1] = G[7] + sm.T[32 + lane]; o[2] = G[11] + sm.T[64 + lane];
      }
    }
    // feature row: slab 0 = [1 1 1 | betas hi | betas lo | betas hi] (8 chunks), then the pose feature hi / lo
    // segments (pseg / 8 chunk pairs); one item = one 16-byte chunk (or hi / lo pair) of every body of the group
    uint4* frow = reinterpret_cast<uint4*>(feat + ((size_t)g * 32 + lane) * fl.pitch);
    const int pch = fl.pseg / 8;
    for (int item = warp; item < 8 + pch; item += NW) {
      if (item < 8) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int k = item * 8 + i;
          float x = 0.f;
          if (live) {
            if (k < 3) x = 1.f;
            else if (k >= fl.off_s0 && k < fl.off_s0 + nbeta) x = __bfloat162float(bf_hi(sm.B[(k - fl.off_s0) * 32 + lane]));
            else if (k >= fl.off_s1 && k < fl.off_s1 + nbeta) {
              const float be = sm.B[(k - fl.off_s1) * 32 + lane];
              x = be - __bfloat162float(bf_hi(be));
            } else if (k >= fl.off_s2 && k < fl.off_s2 + nbeta) x = __bfloat162float(bf_hi(sm.B[(k - fl.off_s2) * 32 + lane]));
          }
          v[i] = x;
        }
        frow[item] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      } else {
        const int c = item - 8;
        uint32_t h[4], l[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float x[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int idx = c * 8 + i * 2 + u;
            float pf = 0.f;
            if (live && idx < NPOSE) {
              const int e = idx % 9;
              pf = sm.R[(9 + idx) * LB_P + lane] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
            }
            x[u] = pf;
          }
          split2(x[0], x[1], h[i], l[i]);
        }
        frow[8 + c] = make_uint4(h[0], h[1], h[2], h[3]);
        frow[8 + pch + c] = make_uint4(l[0], l[1], l[2], l[3]);
      }
    }
    if (featf != nullptr) {
      float* fr = featf + ((size_t)g * 32 + lane) * fl.nf_pad;
      for (int k = warp; k < fl.nf_pad; k += NW) {
        float x = 0.f;
        if (live) {
          if (k < nbeta) x = sm.B[k * 32 + lane];
          else if (k - nbeta < NPOSE) {
            const int idx = k - nbeta, e = idx % 9;
            x = sm.R[(9 + idx) * LB_P + lane] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
          }
        }
        fr[k] = x;
      }
    }
  }
}

// ---- backward, lane = body.  One CTA (16 warps) per 32-body group:
//   P1 all threads: every input of the group staged into shared memory with coalesced, batched loads (pose rows,
//      betas, the group's A block -> global rotations, dA, the split-K partials of dfeat summed, the chain
//      joints' dJ), accumulators cleared;
//   P2 all threads: rest joints (and Rodrigues for axis-angle input), G_t = A_t + G_R Jr;
//   P3 the reverse walk, deepest level first, one warp per joint, each lane ITS body, shared memory only (the critical path:
//      ~200 instructions per joint);
//   P4 all threads: + pose-blend gradient (Rodrigues backward for axis-angle), betas / transl gradients, coalesced
//      write-out.
constexpr int LBB_THREADS = 512;
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
// rotation part (row-major) of one body's transform stored as (r00 r10 r01 r11) (r02 r12 t0 t1) (r20 r21 r22 t2)
__device__ __forceinline__ void lb_rot_of(const float4* p, float (&R)[9]) {
  const float4 q0 = p[0], q1 = p[32], q2 = p[64];
  R[0] = q0.x; R[3] = q0.y; R[1] = q0.z; R[4] = q0.w; R[2] = q1.x; R[5] = q1.y; R[6] = q2.x; R[7] = q2.y; R[8] = q2.z;
}
struct LbBwdSmem {
  float R[NJ * 9 * LB_P];        // local rotations -> dL/dR
  float AAx[NJ * 3 * LB_P];      // axis-angle input -> its gradient
  float G[NJ * 12 * 32];         // the group's transforms as stored ([joint][3][lane] float4)
  float J[NJ * 3 * 32];          // rest joints
  float B[LB_MAXB * 32];         // betas
  float DA[NJ * 12 * 32];        // dL/dA (sum of the partials)
  float D[NJ * 12 * 32];         // [j]: dL/dG of j's PARENT as far as it comes through j (gathered by the parent)
  float DJ[NJ * 3 * 32];         // dL/dJr, final
  float DJc[NJ * 3 * 32];        // what a joint hands up to its parent's dL/dJr
  float DF[224 * LB_P];          // dL/d[betas | pose feature] (sum of the split-K partials), [k][body]
  float DJo[NJ * 3 * LB_P];      // dL/d(posed chain joints) from the caller
  float Jsd[NJ * 3 * LB_MAXB];
  float Jt[NJ * 3];
};

template <bool AA>
__global__ void __launch_bounds__(LBB_THREADS, 1)
pose_bwd_lb_kernel(DevModel m, const float* __restrict__ betas, const float* __restrict__ pose, int b0, int nb, int S,
                   const float* __restrict__ A_blk, const float* __restrict__ dA_part, int n_dA_parts,
                   const float* __restrict__ dtr_part, const float* __restrict__ dfeat_part, int n_dfeat_parts,
                   const float* __restrict__ dJ, float* __restrict__ grad_betas, float* __restrict__ grad_pose,
                   float* __restrict__ grad_transl) {
  extern __shared__ __align__(16) unsigned char lbraw_[];
  LbBwdSmem& sm = *reinterpret_cast<LbBwdSmem*>(lbraw_);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = blockIdx.x;
  const int nlive = max(0, min(32, nb - g * 32));
  const FeatLayout fl = m.fl;
  const int nbeta = fl.nb, nf = fl.nf_pad, NG = S / 32;
  const size_t body0 = (size_t)b0 + (size_t)g * 32;
  pdl_wait();                           // launched behind the gradient GEMM with the PDL attribute
  // ---------------- P1: stage ----------------
  {
    // (a) straight copies, 16 bytes per cp.async: the group's transforms and dL/dA
    const float4* A4 = reinterpret_cast<const float4*>(A_blk) + (size_t)g * (NJ * 3 * 32);
    const float4* dA4 = reinterpret_cast<const float4*>(dA_part + (size_t)g * (NJ * 12 * 32));
    for (int i = tid; i < NJ * 3 * 32; i += LBB_THREADS) cp_async16(reinterpret_cast<float4*>(sm.G) + i, A4 + i);
    for (int i = tid; i < NJ * 12 * 8; i += LBB_THREADS) cp_async16(reinterpret_cast<float4*>(sm.DA) + i, dA4 + i);
    asm volatile("cp.async.commit_group;" ::: "memory");
    // (b) row-major per-body tensors go through registers and are stored transposed ([k][body]).  All global
    // loads of this block are issued before the first store, so the CTA pays about one memory round trip.
    constexpr int PWc = AA ? NJ * 3 : NJ * 9;
    constexpr int PIT = (32 * PWc / 4 + LBB_THREADS - 1) / LBB_THREADS;     // float4 per thread: pose rows
    constexpr int DIT = (32 * 224 / 4 + LBB_THREADS - 1) / LBB_THREADS;     // float4 per thread: dfeat rows (nf <= 224)
    constexpr int JIT = (32 * NJ * 3 + LBB_THREADS - 1) / LBB_THREADS;      // floats per thread: chain-joint gradient
    float* dstT = AA ? sm.AAx : sm.R;
    const bool al = (reinterpret_cast<uintptr_t>(pose) & 15) == 0;
    float4 pv[PIT];
    {
      const float4* src4 = reinterpret_cast<const float4*>(pose + body0 * PWc);   // PWc * 4 bytes is a multiple of 16
      const int n4 = nlive * PWc / 4;
#pragma unroll
      for (int it = 0; it < PIT; ++it) {
        const int i = tid + it * LBB_THREADS;
        pv[it] = (al && i < n4) ? src4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float4 dv[DIT];
    const int dn4 = 32 * nf / 4;
    {
      const float4* base4 = reinterpret_cast<const float4*>(dfeat_part + (size_t)g * 32 * nf);
      const size_t pstride4 = (size_t)S * nf / 4;
      if (n_dfeat_parts == 4) {                      // the production split count at full slabs: 4 x DIT loads in flight
        float4 w[DIT][4];
#pragma unroll
        for (int it = 0; it < DIT; ++it) {
          const int i = tid + it * LBB_THREADS;
#pragma unroll
          for (int q = 0; q < 4; ++q) w[it][q] = i < dn4 ? base4[(size_t)q * pstride4 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int it = 0; it < DIT; ++it) {
          dv[it].x = (w[it][0].x + w[it][1].x) + (w[it][2].x + w[it][3].x);
          dv[it].y = (w[it][0].y + w[it][1].y) + (w[it][2].y + w[it][3].y);
          dv[it].z = (w[it][0].z + w[it][1].z) + (w[it][2].z + w[it][3].z);
          dv[it].w = (w[it][0].w + w[it][1].w) + (w[it][2].w + w[it][3].w);
        }
      } else {
#pragma unroll
        for (int it = 0; it < DIT; ++it) {
          const int i = tid + it * LBB_THREADS;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (i < dn4) {
            int q = 0;
            for (; q + 4 <= n_dfeat_parts; q += 4) {
              const float4 v0 = base4[(size_t)q * pstride4 + i], v1 = base4[(size_t)(q + 1) * pstride4 + i];
              const float4 v2 = base4[(size_t)(q + 2) * pstride4 + i], v3 = base4[(size_t)(q + 3) * pstride4 + i];
              v.x += (v0.x + v1.x) + (v2.x + v3.x); v.y += (v0.y + v1.y) + (v2.y + v3.y);
              v.z += (v0.z + v1.z) + (v2.z + v3.z); v.w += (v0.w + v1.w) + (v2.w + v3.w);
            }
            for (; q < n_dfeat_parts; ++q) {
              const float4 x = base4[(size_t)q * pstride4 + i];
              v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
            }
          }
          dv[it] = v;
        }
      }
    }
    float jv[JIT];
#pragma unroll
    for (int it = 0; it < JIT; ++it) {
      const int i = tid + it * LBB_THREADS, body = i / (NJ * 3), k = i - body * (NJ * 3);
      jv[it] = (dJ != nullptr && body < nlive) ? dJ[(body0 + body) * m.njout * 3 + k] : 0.f;
    }
    float bv = 0.f;
    if (tid < 32 * nbeta && tid / nbeta < nlive) bv = betas[body0 * nbeta + tid];
    // stores
#pragma unroll
    for (int it = 0; it < PIT; ++it) {
      const int i = tid + it * LBB_THREADS;
      if (al && i < nlive * PWc / 4) {
        const float x[4] = {pv[it].x, pv[it].y, pv[it].z, pv[it].w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = i * 4 + u, body = e / PWc, k = e - body * PWc;
          dstT[k * LB_P + body] = x[u];
        }
      }
    }
    if (!al) {
      const float* src = pose + body0 * PWc;
      for (int i = tid; i < nlive * PWc; i += LBB_THREADS) {
        const int body = i / PWc, k = i - body * PWc;
        dstT[k * LB_P + body] = src[i];
      }
    }
#pragma unroll
    for (int it = 0; it < DIT; ++it) {
      const int i = tid + it * LBB_THREADS;
      if (i < dn4) {
        const int e = i * 4, body = e / nf, k = e - body * nf;                        // nf is a multiple of 4
        sm.DF[k * LB_P + body] = dv[it].x; sm.DF[(k + 1) * LB_P + body] = dv[it].y;
        sm.DF[(k + 2) * LB_P + body] = dv[it].z; sm.DF[(k + 3) * LB_P + body] = dv[it].w;
      }
    }
#pragma unroll
    for (int it = 0; it < JIT; ++it) {
      const int i = tid + it * LBB_THREADS, body = i / (NJ * 3), k = i - body * (NJ * 3);
      if (i < 32 * NJ * 3) sm.DJo[k * LB_P + body] = jv[it];
    }
    if (tid < 32 * nbeta) sm.B[(tid % nbeta) * 32 + tid / nbeta] = bv;
    for (int i = tid; i < NJ * 3 * nbeta; i += LBB_THREADS) sm.Jsd[i] = m.Jsd[i];
    if (tid < NJ * 3) sm.Jt[tid] = m.Jt[tid];
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  __syncthreads();
  // ---------------- P2: rest joints, local rotations ----------------
  for (int k = warp; k < NJ * 3; k += LBB_THREADS / 32) {
    float acc = sm.Jt[k];
    for (int l = 0; l < nbeta; ++l) acc = fmaf(sm.Jsd[k * nbeta + l], sm.B[l * 32 + lane], acc);
    sm.J[k * 32 + lane] = acc;
  }
  if (AA) {
    for (int j = warp; j < NJ; j += LBB_THREADS / 32) {
      float r[3] = {0.f, 0.f, 0.f}, R[9];
      if (lane < nlive) { r[0] = sm.AAx[(j * 3) * LB_P + lane]; r[1] = sm.AAx[(j * 3 + 1) * LB_P + lane]; r[2] = sm.AAx[(j * 3 + 2) * LB_P + lane]; }
      rodrigues_fwd(r, R);
#pragma unroll
      for (int e = 0; e < 9; ++e) sm.R[(j * 9 + e) * LB_P + lane] = R[e];
    }
  }
  __syncthreads();
  // ---------------- P3: reverse walk, one tree level at a time (deepest first), one warp per joint of the level.
  // A joint leaves what it hands up in ITS OWN slots (sm.D[j]: dL/dG of its parent, sm.DJc[j]: the rest-joint term);
  // the parent gathers its children's slots one level later, so the joints of a level never write the same word ----
#pragma unroll 1
  for (int dpt = m.chain.maxdepth; dpt >= 0; --dpt) {
    for (int i = m.chain.level_ptr[dpt] + warp; i < m.chain.level_ptr[dpt + 1]; i += LBB_THREADS / 32) {
      const int j = m.chain.order[i];
      float R[9], GR[9], Jr[3], dAr[12], dGR[9], dGt[3], dJr[3], Dj[12], DJj[3];
#pragma unroll
      for (int e = 0; e < 12; ++e) Dj[e] = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) DJj[c] = 0.f;
      for (int k = 0; k < m.chain.nchild[j]; ++k) {               // what the children handed up
        const int ch = m.chain.child[j][k];
#pragma unroll
        for (int e = 0; e < 12; ++e) Dj[e] += sm.D[(ch * 12 + e) * 32 + lane];
#pragma unroll
        for (int c = 0; c < 3; ++c) DJj[c] -= sm.DJc[(ch * 3 + c) * 32 + lane];
      }
#pragma unroll
      for (int e = 0; e < 9; ++e) R[e] = sm.R[(j * 9 + e) * LB_P + lane];
      lb_rot_of(reinterpret_cast<const float4*>(sm.G) + (j * 3) * 32 + lane, GR);
#pragma unroll
      for (int k = 0; k < 3; ++k) Jr[k] = sm.J[(j * 3 + k) * 32 + lane];
#pragma unroll
      for (int e = 0; e < 12; ++e) dAr[e] = sm.DA[(j * 12 + e) * 32 + lane];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float dat = dAr[r * 4 + 3];
        dGt[r] = Dj[r * 4 + 3] + dat + sm.DJo[(j * 3 + r) * LB_P + lane];
#pragma unroll
        for (int c = 0; c < 3; ++c) dGR[r * 3 + c] = Dj[r * 4 + c] + dAr[r * 4 + c] - dat * Jr[c];
      }
#pragma unroll
      for (int c = 0; c < 3; ++c)
        dJr[c] = DJj[c] - (GR[c] * dAr[3] + GR[3 + c] * dAr[7] + GR[6 + c] * dAr[11]);
      const int p = m.chain.parent[j];
      float dRl[9];
      if (p >= 0) {
        float PR[9], rel[3];
        lb_rot_of(reinterpret_cast<const float4*>(sm.G) + (p * 3) * 32 + lane, PR);
#pragma unroll
        for (int r = 0; r < 3; ++r) rel[r] = Jr[r] - sm.J[(p * 3 + r) * 32 + lane];
        // G_j = G_p . [R_j | rel_j]: hand dL/dG_p up (own slot), keep dL/dR_j and dL/drel_j
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
          for (int c = 0; c < 3; ++c)
            sm.D[(j * 12 + r * 4 + c) * 32 + lane] = dGR[r * 3] * R[c * 3] + dGR[r * 3 + 1] * R[c * 3 + 1] +
                                                     dGR[r * 3 + 2] * R[c * 3 + 2] + dGt[r] * rel[c];
          sm.D[(j * 12 + r * 4 + 3) * 32 + lane] = dGt[r];
        }
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int c = 0; c < 3; ++c) dRl[r * 3 + c] = PR[r] * dGR[c] + PR[3 + r] * dGR[3 + c] + PR[6 + r] * dGR[6 + c];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float drel = PR[c] * dGt[0] + PR[3 + c] * dGt[1] + PR[6 + c] * dGt[2];
          dJr[c] += drel;
          sm.DJc[(j * 3 + c) * 32 + lane] = drel;
        }
      } else {
#pragma unroll
        for (int e = 0; e < 9; ++e) dRl[e] = dGR[e];
#pragma unroll
        for (int c = 0; c < 3; ++c) dJr[c] += dGt[c];
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) sm.DJ[(j * 3 + c) * 32 + lane] = dJr[c];       // final
#pragma unroll
      for (int e = 0; e < 9; ++e) sm.R[(j * 9 + e) * LB_P + lane] = dRl[e];        // chain part of dL/dR_j
    }
    __syncthreads();
  }
  // ---------------- P4: blend part, outputs ----------------
  for (int j = warp; j < NJ; j += LBB_THREADS / 32) {
    float dRl[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) {
      dRl[e] = sm.R[(j * 9 + e) * LB_P + lane];
      if (j >= 1) dRl[e] += sm.DF[(nbeta + (j - 1) * 9 + e) * LB_P + lane];
    }
    if (AA) {
      float r[3] = {0.f, 0.f, 0.f}, dr[3];
      if (lane < nlive) { r[0] = sm.AAx[(j * 3) * LB_P + lane]; r[1] = sm.AAx[(j * 3 + 1) * LB_P + lane]; r[2] = sm.AAx[(j * 3 + 2) * LB_P + lane]; }
      rodrigues_bwd(r, dRl, dr);
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 3; ++k) sm.AAx[(j * 3 + k) * LB_P + lane] = dr[k];
    } else {
#pragma unroll
      for (int e = 0; e < 9; ++e) sm.R[(j * 9 + e) * LB_P + lane] = dRl[e];
    }
  }
  for (int l = warp; l < nbeta; l += LBB_THREADS / 32) {
    float v = sm.DF[l * LB_P + lane];
    for (int k = 0; k < NJ * 3; ++k) v = fmaf(sm.Jsd[k * nbeta + l], sm.DJ[k * 32 + lane], v);
    if (lane < nlive) grad_betas[(body0 + lane) * nbeta + l] = v;
  }
  if (grad_transl != nullptr && warp < 3 && lane < nlive) {
    const int r = warp;
    float t = 0.f;
    for (int j = 0; j < NJ; ++j) t += sm.DJo[(j * 3 + r) * LB_P + lane];
    for (int q = 0; q < n_dA_parts; ++q) t += dtr_part[(((size_t)q * NG + g) * 3 + r) * 32 + lane];
    grad_transl[(body0 + lane) * 3 + r] = t;
  }
  __syncthreads();
  {
    const int PW = AA ? NJ * 3 : NJ * 9;
    const float* srcT = AA ? sm.AAx : sm.R;
    float* dst = grad_pose + body0 * PW;
    const int n = nlive * PW;
    for (int i = tid; i < n; i += LBB_THREADS) {
      const int body = i / PW, k = i - body * PW;
      dst[i] = srcT[k * LB_P + body];
    }
  }
}

constexpr size_t LB_FWD_SMEM = sizeof(LbFwdSmem);
constexpr size_t LB_BWD_SMEM = sizeof(LbBwdSmem);

// pack_model rejects more than MAX_BETAS betas, so every model fits these kernels: one thread per (body, beta)
// stages the betas, slab 0 of the feature layout holds them, and dfeat rows (nf_pad) fit sm.DF
static_assert(MAX_BETAS * 32 <= LBF_THREADS && MAX_BETAS * 32 <= LBB_THREADS, "betas staging: one thread per (body, beta)");
static_assert(MAX_BETAS <= LB_MAXB, "betas staging arrays");
static_assert((MAX_BETAS + NPOSE + 15) / 16 * 16 <= 224, "sm.DF holds nf_pad <= 224 rows");

// Sw = active slab width (multiple of 32, >= nb); columns in [nb, Sw) are written as zeros
int launch_pose_fwd(const DevModel& m, const float* betas, const float* pose, bool axis_angle, int b0, int nb, int S,
                    int Sw, __nv_bfloat16* feat, float* featf, float* A_T, const float* transl, float* joints,
                    cudaStream_t st) {
  const int grid = Sw / 32;
  if (axis_angle) {
    B200_SMEM_ATTR_ONCE(pose_fwd_lb_kernel<true>, LB_FWD_SMEM);
    LaunchTimer _timer("pose_fwd", st);
    pose_fwd_lb_kernel<true><<<grid, LBF_THREADS, LB_FWD_SMEM, st>>>(m, betas, pose, b0, nb, S, feat, featf, A_T, transl, joints);
  } else {
    B200_SMEM_ATTR_ONCE(pose_fwd_lb_kernel<false>, LB_FWD_SMEM);
    LaunchTimer _timer("pose_fwd", st);
    pose_fwd_lb_kernel<false><<<grid, LBF_THREADS, LB_FWD_SMEM, st>>>(m, betas, pose, b0, nb, S, feat, featf, A_T, transl, joints);
  }
  B200_LAUNCH_CHECK("pose_fwd");
  return 0;
}

int launch_pose_bwd(const DevModel& m, const float* betas, const float* pose, bool axis_angle, int b0, int nb, int S,
                    const float* A_blk, const float* dA_part, int n_dA_parts, const float* dtr_part, const float* dfeat_part,
                    int n_dfeat_parts, const float* dJ, float* grad_betas, float* grad_pose,
                    float* grad_transl, cudaStream_t st) {
  if (nb <= 0) return 0;
  const int grid = (nb + 31) / 32;
  if (axis_angle) {
    B200_SMEM_ATTR_ONCE(pose_bwd_lb_kernel<true>, LB_BWD_SMEM);
    LaunchTimer _timer("pose_bwd", st);
    B200_CUDA_TRY(launch_k(pose_bwd_lb_kernel<true>, dim3(grid), dim3(LBB_THREADS), LB_BWD_SMEM, st, true, m, betas, pose, b0, nb,
                           S, A_blk, dA_part, n_dA_parts, dtr_part, dfeat_part, n_dfeat_parts, dJ, grad_betas, grad_pose,
                           grad_transl));
  } else {
    B200_SMEM_ATTR_ONCE(pose_bwd_lb_kernel<false>, LB_BWD_SMEM);
    LaunchTimer _timer("pose_bwd", st);
    B200_CUDA_TRY(launch_k(pose_bwd_lb_kernel<false>, dim3(grid), dim3(LBB_THREADS), LB_BWD_SMEM, st, true, m, betas, pose, b0, nb,
                           S, A_blk, dA_part, n_dA_parts, dtr_part, dfeat_part, n_dfeat_parts, dJ, grad_betas, grad_pose,
                           grad_transl));
  }
  B200_LAUNCH_CHECK("pose_bwd");
  return 0;
}

}  // namespace b200smpl
