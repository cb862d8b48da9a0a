// Small in-tree helpers of the SMPL path (SURVEY.md section 8 rows a13-a18), forward + hand-written
// backward: rot6d_to_rotmat (utils/rigid_transform_utils.py:27-41), orthographic / perspective
// projection (utils/cam_utils.py:5-26, 54-85), undo_keypoint_normalisation
// (utils/joints2d_utils.py:5-10) and the joints2D loss term (losses/multi_task_loss.py:97-113).
// All are tiny element-wise / per-body kernels; they exist so the whole fitting / training step
// stays on hand-written kernels with no eager-op launches in between.
#include "common.cuh"
#include "rodrigues.cuh"

namespace b200smpl {

// smplx.lbs.batch_rodrigues as a standalone op (SURVEY.md section 8 row a6; the reference calls it directly at
// player_recon.py:201,655 and hmr.py:207): one thread per rotation vector
__global__ void rodrigues_fwd_kernel(const float* __restrict__ rv, float* __restrict__ R, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float r[3] = {rv[i * 3], rv[i * 3 + 1], rv[i * 3 + 2]};
  float o[9];
  rodrigues_fwd(r, o);
#pragma unroll
  for (int e = 0; e < 9; ++e) R[i * 9 + e] = o[e];
}
__global__ void rodrigues_bwd_kernel(const float* __restrict__ rv, const float* __restrict__ gR, float* __restrict__ grv,
                                     long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float r[3] = {rv[i * 3], rv[i * 3 + 1], rv[i * 3 + 2]};
  float g[9], d[3];
#pragma unroll
  for (int e = 0; e < 9; ++e) g[e] = gR[i * 9 + e];
  rodrigues_bwd(r, g, d);
  grv[i * 3] = d[0]; grv[i * 3 + 1] = d[1]; grv[i * 3 + 2] = d[2];
}

// F.normalize(v, dim=1, eps=1e-12): v / max(||v||, eps)
__device__ __forceinline__ float safe_norm(const float v[3]) {
  return fmaxf(sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]), 1e-12f);
}

__global__ void rot6d_fwd_kernel(const float* __restrict__ x6, float* __restrict__ R, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* x = x6 + i * 6;
  const float a1[3] = {x[0], x[2], x[4]}, a2[3] = {x[1], x[3], x[5]};
  const float n1 = safe_norm(a1);
  const float b1[3] = {a1[0] / n1, a1[1] / n1, a1[2] / n1};
  const float s = b1[0] * a2[0] + b1[1] * a2[1] + b1[2] * a2[2];
  const float u[3] = {a2[0] - s * b1[0], a2[1] - s * b1[1], a2[2] - s * b1[2]};
  const float n2 = safe_norm(u);
  const float b2[3] = {u[0] / n2, u[1] / n2, u[2] / n2};
  const float b3[3] = {b1[1] * b2[2] - b1[2] * b2[1], b1[2] * b2[0] - b1[0] * b2[2], b1[0] * b2[1] - b1[1] * b2[0]};
  float* o = R + i * 9;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    o[r * 3 + 0] = b1[r];
    o[r * 3 + 1] = b2[r];
    o[r * 3 + 2] = b3[r];
  }
}

__global__ void rot6d_bwd_kernel(const float* __restrict__ x6, const float* __restrict__ gR, float* __restrict__ gx6,
                                 long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* x = x6 + i * 6;
  const float* g = gR + i * 9;
  const float a1[3] = {x[0], x[2], x[4]}, a2[3] = {x[1], x[3], x[5]};
  const float n1 = safe_norm(a1);
  const float b1[3] = {a1[0] / n1, a1[1] / n1, a1[2] / n1};
  const float s = b1[0] * a2[0] + b1[1] * a2[1] + b1[2] * a2[2];
  const float u[3] = {a2[0] - s * b1[0], a2[1] - s * b1[1], a2[2] - s * b1[2]};
  const float n2 = safe_norm(u);
  const float b2[3] = {u[0] / n2, u[1] / n2, u[2] / n2};
  float gb1[3] = {g[0], g[3], g[6]}, gb2[3] = {g[1], g[4], g[7]};
  const float gb3[3] = {g[2], g[5], g[8]};
  // b3 = b1 x b2 :  d/db1 = b2 x g3 ; d/db2 = g3 x b1
  gb1[0] += b2[1] * gb3[2] - b2[2] * gb3[1];
  gb1[1] += b2[2] * gb3[0] - b2[0] * gb3[2];
  gb1[2] += b2[0] * gb3[1] - b2[1] * gb3[0];
  gb2[0] += gb3[1] * b1[2] - gb3[2] * b1[1];
  gb2[1] += gb3[2] * b1[0] - gb3[0] * b1[2];
  gb2[2] += gb3[0] * b1[1] - gb3[1] * b1[0];
  // b2 = u / |u|
  const float d2 = b2[0] * gb2[0] + b2[1] * gb2[1] + b2[2] * gb2[2];
  const float gu[3] = {(gb2[0] - b2[0] * d2) / n2, (gb2[1] - b2[1] * d2) / n2, (gb2[2] - b2[2] * d2) / n2};
  // u = a2 - (b1.a2) b1
  const float gub1 = gu[0] * b1[0] + gu[1] * b1[1] + gu[2] * b1[2];
  const float ga2[3] = {gu[0] - gub1 * b1[0], gu[1] - gub1 * b1[1], gu[2] - gub1 * b1[2]};
#pragma unroll
  for (int k = 0; k < 3; ++k) gb1[k] += -gub1 * a2[k] - s * gu[k];
  // b1 = a1 / |a1|
  const float d1 = b1[0] * gb1[0] + b1[1] * gb1[1] + b1[2] * gb1[2];
  float* o = gx6 + i * 6;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    o[2 * k] = (gb1[k] - b1[k] * d1) / n1;
    o[2 * k + 1] = ga2[k];
  }
}

// ---- orthographic (+ optional pixel de-normalisation) ----------------------------------------
__global__ void ortho_fwd_kernel(const float* __restrict__ pts, const float* __restrict__ cam, float* __restrict__ out,
                                 int n, float pixel_wh) {
  const int b = blockIdx.x;
  const float s = cam[b * 3], tx = cam[b * 3 + 1], ty = cam[b * 3 + 2];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float* p = pts + ((size_t)b * n + i) * 3;
    float u = s * (p[0] + tx), v = s * (p[1] + ty);
    if (pixel_wh > 0.f) {
      u = (u + 1.f) * (pixel_wh / 2.0f);
      v = (v + 1.f) * (pixel_wh / 2.0f);
    }
    out[((size_t)b * n + i) * 2] = u;
    out[((size_t)b * n + i) * 2 + 1] = v;
  }
}

__device__ __forceinline__ float block_sum(float v, float* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  float r = 0.f;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += sh[w];
  return r;
}

__global__ void ortho_bwd_kernel(const float* __restrict__ pts, const float* __restrict__ cam,
                                 const float* __restrict__ gout, float* __restrict__ gpts, float* __restrict__ gcam,
                                 int n, float pixel_wh) {
  __shared__ float sh[32];
  const int b = blockIdx.x;
  const float s = cam[b * 3], tx = cam[b * 3 + 1], ty = cam[b * 3 + 2];
  const float k = pixel_wh > 0.f ? pixel_wh / 2.0f : 1.f;
  float gs = 0.f, gtx = 0.f, gty = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float* p = pts + ((size_t)b * n + i) * 3;
    const float gu = gout[((size_t)b * n + i) * 2] * k, gv = gout[((size_t)b * n + i) * 2 + 1] * k;
    // __fmul_rn is never contracted into the sums: the compiler unswitches this loop on gpts, and a product that is
    // stored in one copy but fused into gtx / gty in the other would give grad_cam other last bits without grad_points
    const float sgu = __fmul_rn(s, gu), sgv = __fmul_rn(s, gv);
    if (gpts != nullptr) {
      float* g = gpts + ((size_t)b * n + i) * 3;
      g[0] = sgu;
      g[1] = sgv;
      g[2] = 0.f;
    }
    gs += gu * (p[0] + tx) + gv * (p[1] + ty);
    gtx += sgu;
    gty += sgv;
  }
  if (gcam != nullptr) {
    gs = block_sum(gs, sh);
    gtx = block_sum(gtx, sh);
    gty = block_sum(gty, sh);
    if (threadIdx.x == 0) {
      gcam[b * 3] = gs;
      gcam[b * 3 + 1] = gtx;
      gcam[b * 3 + 2] = gty;
    }
  }
}

// ---- perspective ------------------------------------------------------------------------------
// intrinsics rows 0 and 1 of the body: from cam_K ([B][3][3], k_stride = 9, or one shared [3][3], k_stride = 0) or
// K = [[f,0,c],[0,f,c],[0,0,1]]
__device__ __forceinline__ void load_intrinsics(float (&K)[6], const float* __restrict__ camK, int k_stride, int b, float f,
                                                float c) {
  if (camK != nullptr) {
#pragma unroll
    for (int i = 0; i < 6; ++i) K[i] = camK[(size_t)b * k_stride + i];
  } else {
    K[0] = f; K[1] = 0.f; K[2] = c; K[3] = 0.f; K[4] = f; K[5] = c;
  }
}

__global__ void persp_fwd_kernel(const float* __restrict__ pts, const float* __restrict__ rot,
                                 const float* __restrict__ trans, float* __restrict__ out, int n, float f, float c,
                                 const float* __restrict__ camK, int k_stride) {
  const int b = blockIdx.x;
  float K[6];
  load_intrinsics(K, camK, k_stride, b, f, c);
  float R[9], t[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = rot[b * 9 + i];
#pragma unroll
  for (int i = 0; i < 3; ++i) t[i] = trans[b * 3 + i];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float* p = pts + ((size_t)b * n + i) * 3;
    const float x = R[0] * p[0] + R[1] * p[1] + R[2] * p[2] + t[0];
    const float y = R[3] * p[0] + R[4] * p[1] + R[5] * p[2] + t[1];
    const float z = R[6] * p[0] + R[7] * p[1] + R[8] * p[2] + t[2];
    // projected = X'/z ; rows 0 and 1 of K . projected (utils/cam_utils.py:79-85)
    const float u = x / z, v = y / z, w = z / z;
    out[((size_t)b * n + i) * 2] = K[0] * u + K[1] * v + K[2] * w;
    out[((size_t)b * n + i) * 2 + 1] = K[3] * u + K[4] * v + K[5] * w;
  }
}

__global__ void persp_bwd_kernel(const float* __restrict__ pts, const float* __restrict__ rot,
                                 const float* __restrict__ trans, const float* __restrict__ gout,
                                 float* __restrict__ gpts, float* __restrict__ grot, float* __restrict__ gtrans, int n,
                                 float f, const float* __restrict__ camK, int k_stride) {
  __shared__ float sh[32];
  const int b = blockIdx.x;
  float K[6];
  load_intrinsics(K, camK, k_stride, b, f, 0.f);
  float R[9], t[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = rot[b * 9 + i];
#pragma unroll
  for (int i = 0; i < 3; ++i) t[i] = trans[b * 3 + i];
  float gR[9], gt[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) gR[i] = 0.f;
  gt[0] = gt[1] = gt[2] = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float* p = pts + ((size_t)b * n + i) * 3;
    const float x = R[0] * p[0] + R[1] * p[1] + R[2] * p[2] + t[0];
    const float y = R[3] * p[0] + R[4] * p[1] + R[5] * p[2] + t[1];
    const float z = R[6] * p[0] + R[7] * p[1] + R[8] * p[2] + t[2];
    const float go0 = gout[((size_t)b * n + i) * 2], go1 = gout[((size_t)b * n + i) * 2 + 1];
    const float gu = K[0] * go0 + K[3] * go1, gv = K[1] * go0 + K[4] * go1;     // d / d (x/z), d / d (y/z)
    const float iz = 1.f / z;
    const float g3[3] = {gu * iz, gv * iz, -(gu * x + gv * y) * iz * iz};
    if (gpts != nullptr) {
      float* g = gpts + ((size_t)b * n + i) * 3;
#pragma unroll
      for (int k = 0; k < 3; ++k) g[k] = R[k] * g3[0] + R[3 + k] * g3[1] + R[6 + k] * g3[2];
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
      for (int k = 0; k < 3; ++k) gR[r * 3 + k] += g3[r] * p[k];
      gt[r] += g3[r];
    }
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const float v = block_sum(gR[i], sh);
    if (grot != nullptr && threadIdx.x == 0) grot[b * 9 + i] = v;
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float v = block_sum(gt[i], sh);
    if (gtrans != nullptr && threadIdx.x == 0) gtrans[b * 3 + i] = v;
  }
}

// ---- fused joints2D loss ------------------------------------------------------------------------
__global__ void count_vis_kernel(const uint8_t* __restrict__ vis, long long n, float* __restrict__ count) {
  __shared__ float sh[32];
  float c = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    c += vis[i] ? 1.f : 0.f;
  c = block_sum(c, sh);
  if (threadIdx.x == 0 && c != 0.f) atomicAdd(count, c);
}

// one CTA per body.  count_ptr: number of (body, joint) pairs in the mean (device scalar) or NULL
__global__ void j2d_loss_kernel(const float* __restrict__ joints, const float* __restrict__ cam,
                                const int32_t* __restrict__ jmap, const float* __restrict__ label,
                                const uint8_t* __restrict__ vis, const float* __restrict__ count_ptr, int batch, int nj,
                                int nmap, float proj_wh, float norm_wh, float log_var, float* __restrict__ loss,
                                float* __restrict__ gjoints, float* __restrict__ gcam) {
  __shared__ float sh[32];
  const int b = blockIdx.x;
  const float s = cam[b * 3], tx = cam[b * 3 + 1], ty = cam[b * 3 + 2];
  const float pairs = count_ptr != nullptr ? *count_ptr : (float)batch * (float)nmap;
  const float inv_count = pairs > 0.f ? 1.f / (2.f * pairs) : 0.f;
  const float ew = expf(-log_var);
  if (gjoints != nullptr)
    for (int i = threadIdx.x; i < nj * 3; i += blockDim.x) gjoints[(size_t)b * nj * 3 + i] = 0.f;
  __syncthreads();
  float lsum = 0.f, gs = 0.f, gtx = 0.f, gty = 0.f;
  for (int i = threadIdx.x; i < nmap; i += blockDim.x) {
    if (vis != nullptr && !vis[(size_t)b * nmap + i]) continue;
    const int J = jmap[i];
    const float* p = joints + ((size_t)b * nj + J) * 3;
    const float t[2] = {tx, ty};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float u = s * (p[k] + t[k]);
      const float pix = (u + 1.f) * (proj_wh / 2.0f);
      const float pn = (2.0f * pix) / norm_wh - 1.0f;
      const float ln = (2.0f * label[((size_t)b * nmap + i) * 2 + k]) / norm_wh - 1.0f;
      const float d = pn - ln;
      lsum += d * d;
      // d loss / d u
      const float gu = 2.f * d * inv_count * ew * (2.0f / norm_wh) * (proj_wh / 2.0f);
      if (gjoints != nullptr) atomicAdd(&gjoints[((size_t)b * nj + J) * 3 + k], s * gu);   // a map may repeat a joint
      gs += gu * (p[k] + t[k]);
      if (k == 0) gtx += s * gu; else gty += s * gu;
    }
  }
  lsum = block_sum(lsum, sh);
  if (gcam != nullptr) {
    gs = block_sum(gs, sh);
    gtx = block_sum(gtx, sh);
    gty = block_sum(gty, sh);
    if (threadIdx.x == 0) {
      gcam[b * 3] = gs;
      gcam[b * 3 + 1] = gtx;
      gcam[b * 3 + 2] = gty;
    }
  }
  if (threadIdx.x == 0) {
    float add = lsum * inv_count * ew;
    if (b == 0) add += log_var;
    atomicAdd(loss, add);
  }
}

}  // namespace b200smpl

using namespace b200smpl;

extern "C" {

int b200smpl_batch_rodrigues(const float* rot_vecs, float* rotmats, int64_t n, void* stream) {
  B200_NVTX("b200smpl_batch_rodrigues");
  if (!rot_vecs || !rotmats || n < 0) return fail(B200SMPL_ERR_INVALID, "bad argument");
  if (n == 0) return 0;
  rodrigues_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rot_vecs, rotmats, n);
  B200_LAUNCH_CHECK("rodrigues_fwd");
  return 0;
}

int b200smpl_batch_rodrigues_backward(const float* rot_vecs, const float* grad_rotmats, float* grad_rot_vecs, int64_t n,
                                      void* stream) {
  B200_NVTX("b200smpl_batch_rodrigues_backward");
  if (!rot_vecs || !grad_rotmats || !grad_rot_vecs || n < 0) return fail(B200SMPL_ERR_INVALID, "bad argument");
  if (n == 0) return 0;
  rodrigues_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rot_vecs, grad_rotmats, grad_rot_vecs, n);
  B200_LAUNCH_CHECK("rodrigues_bwd");
  return 0;
}

int b200smpl_rot6d_to_rotmat(const float* x6, float* rotmats, int64_t n, void* stream) {
  B200_NVTX("b200smpl_rot6d_to_rotmat");
  if (!x6 || !rotmats || n < 0) return fail(B200SMPL_ERR_INVALID, "bad argument");
  if (n == 0) return 0;
  rot6d_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x6, rotmats, n);
  B200_LAUNCH_CHECK("rot6d_fwd");
  return 0;
}

int b200smpl_rot6d_to_rotmat_backward(const float* x6, const float* grad_rotmats, float* grad_x6, int64_t n,
                                      void* stream) {
  B200_NVTX("b200smpl_rot6d_to_rotmat_backward");
  if (!x6 || !grad_rotmats || !grad_x6 || n < 0) return fail(B200SMPL_ERR_INVALID, "bad argument");
  if (n == 0) return 0;
  rot6d_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x6, grad_rotmats, grad_x6, n);
  B200_LAUNCH_CHECK("rot6d_bwd");
  return 0;
}

int b200smpl_orthographic_project(const float* points, const float* cam, float* out, int batch, int n, float pixel_wh,
                                  void* stream) {
  B200_NVTX("b200smpl_orthographic_project");
  if (!points || !cam || !out || batch < 1 || n < 1) return fail(B200SMPL_ERR_INVALID, "bad argument");
  ortho_fwd_kernel<<<batch, 128, 0, (cudaStream_t)stream>>>(points, cam, out, n, pixel_wh);
  B200_LAUNCH_CHECK("ortho_fwd");
  return 0;
}

int b200smpl_orthographic_project_backward(const float* points, const float* cam, const float* grad_out,
                                           float* grad_points, float* grad_cam, int batch, int n, float pixel_wh,
                                           void* stream) {
  B200_NVTX("b200smpl_orthographic_project_backward");
  if (!points || !cam || !grad_out || batch < 1 || n < 1) return fail(B200SMPL_ERR_INVALID, "bad argument");
  ortho_bwd_kernel<<<batch, 128, 0, (cudaStream_t)stream>>>(points, cam, grad_out, grad_points, grad_cam, n, pixel_wh);
  B200_LAUNCH_CHECK("ortho_bwd");
  return 0;
}

int b200smpl_perspective_project(const float* points, const float* rotation, const float* translation, float* out,
                                 int batch, int n, float focal_length, float img_wh, void* stream) {
  B200_NVTX("b200smpl_perspective_project");
  if (!points || !rotation || !translation || !out || batch < 1 || n < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  persp_fwd_kernel<<<batch, 128, 0, (cudaStream_t)stream>>>(points, rotation, translation, out, n, focal_length,
                                                           img_wh / 2.0f, nullptr, 0);
  B200_LAUNCH_CHECK("persp_fwd");
  return 0;
}

int b200smpl_perspective_project_camk(const float* points, const float* rotation, const float* translation,
                                      const float* cam_K, int cam_K_batched, float* out, int batch, int n, void* stream) {
  B200_NVTX("b200smpl_perspective_project_camk");
  if (!points || !rotation || !translation || !cam_K || !out || batch < 1 || n < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  persp_fwd_kernel<<<batch, 128, 0, (cudaStream_t)stream>>>(points, rotation, translation, out, n, 0.f, 0.f, cam_K,
                                                           cam_K_batched ? 9 : 0);
  B200_LAUNCH_CHECK("persp_fwd");
  return 0;
}

int b200smpl_perspective_project_camk_backward(const float* points, const float* rotation, const float* translation,
                                               const float* cam_K, int cam_K_batched, const float* grad_out,
                                               float* grad_points, float* grad_rotation, float* grad_translation,
                                               int batch, int n, void* stream) {
  B200_NVTX("b200smpl_perspective_project_camk_backward");
  if (!points || !rotation || !translation || !cam_K || !grad_out || batch < 1 || n < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  persp_bwd_kernel<<<batch, 128, 0, (cudaStream_t)stream>>>(points, rotation, translation, grad_out, grad_points,
                                                           grad_rotation, grad_translation, n, 0.f, cam_K,
                                                           cam_K_batched ? 9 : 0);
  B200_LAUNCH_CHECK("persp_bwd");
  return 0;
}

int b200smpl_perspective_project_backward(const float* points, const float* rotation, const float* translation,
                                          const float* grad_out, float* grad_points, float* grad_rotation,
                                          float* grad_translation, int batch, int n, float focal_length, float img_wh,
                                          void* stream) {
  B200_NVTX("b200smpl_perspective_project_backward");
  (void)img_wh;
  if (!points || !rotation || !translation || !grad_out || batch < 1 || n < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  persp_bwd_kernel<<<batch, 128, 0, (cudaStream_t)stream>>>(points, rotation, translation, grad_out, grad_points,
                                                           grad_rotation, grad_translation, n, focal_length, nullptr, 0);
  B200_LAUNCH_CHECK("persp_bwd");
  return 0;
}

int b200smpl_joints2d_loss(const float* joints, const float* cam, const int32_t* joint_map, const float* label,
                           const uint8_t* vis, int batch, int num_joints, int nmap, float proj_wh, float norm_wh,
                           float log_var, float* loss, float* grad_joints, float* grad_cam, void* stream) {
  B200_NVTX("b200smpl_joints2d_loss");
  if (!joints || !cam || !joint_map || !label || !loss || batch < 1 || num_joints < 1 || nmap < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const float* count_ptr = nullptr;
  if (vis != nullptr) {
    // loss[1] is used as the visible-pair counter: the caller provides a 2-float buffer in this case
    B200_CUDA_TRY(cudaMemsetAsync(loss + 1, 0, sizeof(float), st));
    const long long n = (long long)batch * nmap;
    count_vis_kernel<<<(unsigned)std::min<long long>((n + 255) / 256, 1024), 256, 0, st>>>(vis, n, loss + 1);
    B200_LAUNCH_CHECK("count_vis");
    count_ptr = loss + 1;
  }
  j2d_loss_kernel<<<batch, 32, 0, st>>>(joints, cam, joint_map, label, vis, count_ptr, batch, num_joints, nmap, proj_wh,
                                        norm_wh, log_var, loss, grad_joints, grad_cam);
  B200_LAUNCH_CHECK("j2d_loss");
  return 0;
}

}  // extern "C"
