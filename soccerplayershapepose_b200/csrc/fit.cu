// Kernels of the batched per-player fitting loop (SURVEY.md section 8f.1; the reference's
// single_view_optimization, PlayerReconstruction/player_recon.py:1172-1294, restated for a batch of
// independent players): per-player reprojection loss with gradients, on-device best-iterate
// tracking (the reference copies the parameters to the host and compares metrics there every
// iteration, player_recon.py:1254-1266 / metrics/train_loss_and_metrics_tracker.py:117-121) and a
// fused masked Adam step (torch.optim.Adam arithmetic, player_recon.py:1199).  Everything reads its
// step counter and flags from device memory so that one iteration can be captured in a CUDA graph
// and replayed.
#include <cstring>

#include "common.cuh"

namespace b200smpl {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One warp per player.  loss_b = mean over the player's visible (joint, coordinate) pairs of the squared
// difference of the normalised 2D keypoints (losses/multi_task_loss.py:97-113 applied to ONE player, as
// the reference's loop does) * exp(-log_var) + log_var  +  shape_weight * mean(beta^2)
// (the shape_params term of multi_task_loss.py:120-124 against a zero label).
__global__ void __launch_bounds__(128)
fit_loss_kernel(const float* __restrict__ joints, const float* __restrict__ cam, const int32_t* __restrict__ jmap,
                const float* __restrict__ label, const uint8_t* __restrict__ vis, const float* __restrict__ betas,
                int batch, int nj, int nmap, int nb, float proj_wh, float norm_wh, float log_var, float shape_weight,
                float* __restrict__ loss, float* __restrict__ gjoints, float* __restrict__ gcam,
                float* __restrict__ gbetas) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= batch) return;
  const float s = cam[b * 3], tx = cam[b * 3 + 1], ty = cam[b * 3 + 2];
  float nvis = 0.f;
  for (int i = lane; i < nmap; i += 32) nvis += (vis == nullptr || vis[(size_t)b * nmap + i]) ? 1.f : 0.f;
  nvis = warp_sum(nvis);
  const float inv_count = nvis > 0.f ? 1.f / (2.f * nvis) : 0.f;
  const float ew = expf(-log_var);
  for (int i = lane; i < nj * 3; i += 32) gjoints[(size_t)b * nj * 3 + i] = 0.f;
  __syncwarp();
  float lsum = 0.f, gs = 0.f, gtx = 0.f, gty = 0.f;
  for (int i = lane; i < nmap; i += 32) {
    if (vis != nullptr && !vis[(size_t)b * nmap + i]) continue;
    const int J = jmap[i];
    const float* p = joints + ((size_t)b * nj + J) * 3;
    const float t[2] = {tx, ty};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float u = s * (p[k] + t[k]);                         // utils/cam_utils.py:5-26
      const float pix = (u + 1.f) * (proj_wh / 2.0f);            // utils/joints2d_utils.py:5-10
      const float pn = (2.0f * pix) / norm_wh - 1.0f;
      const float ln = (2.0f * label[((size_t)b * nmap + i) * 2 + k]) / norm_wh - 1.0f;
      const float d = pn - ln;
      lsum += d * d;
      const float gu = 2.f * d * inv_count * ew * (2.0f / norm_wh) * (proj_wh / 2.0f);   // d loss / d u
      atomicAdd(&gjoints[((size_t)b * nj + J) * 3 + k], s * gu);  // a joint may appear twice in the map
      gs += gu * (p[k] + t[k]);
      if (k == 0) gtx += s * gu; else gty += s * gu;
    }
  }
  lsum = warp_sum(lsum);
  gs = warp_sum(gs); gtx = warp_sum(gtx); gty = warp_sum(gty);
  float bsum = 0.f;
  for (int l = lane; l < nb; l += 32) {
    const float be = betas[(size_t)b * nb + l];
    bsum += be * be;
    if (gbetas != nullptr) gbetas[(size_t)b * nb + l] = shape_weight * 2.f * be / (float)nb;
  }
  bsum = warp_sum(bsum);
  if (lane == 0) {
    loss[b] = lsum * inv_count * ew + log_var + shape_weight * bsum / (float)nb;
    gcam[b * 3] = gs; gcam[b * 3 + 1] = gtx; gcam[b * 3 + 2] = gty;
  }
}

// improved[b] = loss[b] < best_loss[b] (then best_loss / best_iter are updated); thread 0 advances the step counter
__global__ void fit_mark_kernel(const float* __restrict__ loss, float* __restrict__ best_loss,
                                int32_t* __restrict__ best_iter, uint8_t* __restrict__ improved,
                                int32_t* __restrict__ step, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int t = *step + 1;                         // 1-based iteration about to be applied
  if (b < batch) {
    const float l = loss[b];
    const bool imp = l < best_loss[b];
    improved[b] = imp ? 1 : 0;
    if (imp) { best_loss[b] = l; best_iter[b] = t; }
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) step[1] = t;   // step[1] is copied to step[0] by the last Adam kernel
}

// p [B][P]: best-iterate copy (the parameters that produced this iteration's loss) then the Adam update
// (torch.optim.Adam: m, v, bias corrections from the device step counter), elementwise, masked per column.
__global__ void fit_adam_kernel(float* __restrict__ p, const float* __restrict__ g, const float* __restrict__ g2,
                                float* __restrict__ m, float* __restrict__ v, float* __restrict__ best,
                                const uint8_t* __restrict__ improved, const uint8_t* __restrict__ frozen,
                                int32_t* __restrict__ step, int commit_step, int batch, int P, float lr, float beta1,
                                float beta2, float eps) {
  const long long n = (long long)batch * P;
  const int t = step[1];
  __shared__ float coef[2];
  if (threadIdx.x == 0) {                                    // once per CTA: two powf cost more than the update itself
    const float bc1 = 1.f - powf(beta1, (float)t), bc2 = 1.f - powf(beta2, (float)t);
    coef[0] = lr / bc1;
    coef[1] = rsqrtf(bc2);
  }
  __syncthreads();
  const float step_size = coef[0], inv_sqrt_bc2 = coef[1];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / P), c = (int)(i - (long long)b * P);
    const float x = p[i];
    if (improved[b]) best[i] = x;
    if (frozen != nullptr && frozen[c]) continue;
    float gr = g[i];
    if (g2 != nullptr) gr += g2[i];
    const float mi = beta1 * m[i] + (1.f - beta1) * gr;
    const float vi = beta2 * v[i] + (1.f - beta2) * gr * gr;
    m[i] = mi;
    v[i] = vi;
    p[i] = x - step_size * mi / (sqrtf(vi) * inv_sqrt_bc2 + eps);
  }
  if (commit_step && blockIdx.x == 0 && threadIdx.x == 0) step[0] = t;
}

// mark_best + the Adam step of every parameter tensor in ONE launch.  A CTA owns `bpc` whole bodies (as many as
// give every thread at most one element of the concatenated parameter row when that fits): it decides "improved"
// for them from the old best loss (shared memory), then updates their rows of every tensor.  The kernel is a chain
// of dependent memory round trips, not bandwidth: a thread issues the loads of its element (parameter, gradient,
// moments) BEFORE the barrier, next to the loss loads, so the chain is one round trip instead of one per tensor.
// The step counter is double-buffered (read step[parity], write step[1 - parity]) so that no CTA can read a
// counter another CTA has already advanced.
constexpr int FIT_THREADS = 256;
constexpr int FIT_MAX_BPC = 32;
struct FitGroups {
  b200smpl_fit_group g[B200SMPL_FIT_MAX_GROUPS];
  int n;
  int ptot;                   // columns of all groups together
};
struct FitElem {              // one element of one tensor and what the update needs of it
  int k, bl;
  long long i;
  float x, gr, m, v;
  bool live, frozen;
};
__device__ __forceinline__ void fit_elem_load(FitElem& e, const FitGroups& G, int idx, int b0, int batch) {
  e.bl = idx / G.ptot;
  int c = idx - e.bl * G.ptot;
  e.k = 0;
#pragma unroll
  for (int k = 0; k < B200SMPL_FIT_MAX_GROUPS - 1; ++k)      // unrolled: the groups stay in the parameter bank
    if (k + 1 < G.n && e.k == k && c >= G.g[k].cols) { c -= G.g[k].cols; e.k = k + 1; }
  e.live = b0 + e.bl < batch;
  e.frozen = true;
  e.x = e.gr = e.m = e.v = 0.f;
#pragma unroll
  for (int k = 0; k < B200SMPL_FIT_MAX_GROUPS; ++k) {
    if (k != e.k || !e.live) continue;
    const b200smpl_fit_group& q = G.g[k];
    e.i = (long long)(b0 + e.bl) * q.cols + c;
    e.x = q.params[e.i];
    e.frozen = q.frozen_cols != nullptr && q.frozen_cols[c];
    if (!e.frozen) {
      e.gr = q.grad[e.i];
      if (q.grad_extra != nullptr) e.gr += q.grad_extra[e.i];
      e.m = q.exp_avg[e.i];
      e.v = q.exp_avg_sq[e.i];
    }
  }
}
__device__ __forceinline__ void fit_elem_store(const FitElem& e, const FitGroups& G, const uint8_t* imp, float beta1,
                                               float beta2, float step_size, float inv_sqrt_bc2, float eps) {
#pragma unroll
  for (int k = 0; k < B200SMPL_FIT_MAX_GROUPS; ++k) {
    if (k != e.k || !e.live) continue;
    const b200smpl_fit_group& q = G.g[k];
    if (imp[e.bl]) q.best_params[e.i] = e.x;
    if (e.frozen) continue;
    const float mi = beta1 * e.m + (1.f - beta1) * e.gr;
    const float vi = beta2 * e.v + (1.f - beta2) * e.gr * e.gr;
    q.exp_avg[e.i] = mi;
    q.exp_avg_sq[e.i] = vi;
    q.params[e.i] = e.x - step_size * mi / (sqrtf(vi) * inv_sqrt_bc2 + eps);
  }
}
__global__ void __launch_bounds__(FIT_THREADS)
fit_update_kernel(FitGroups G, int bpc, const float* __restrict__ loss, float* __restrict__ best_loss,
                  int32_t* __restrict__ best_iter, float* __restrict__ first_loss, int32_t* __restrict__ step, int parity,
                  int batch, float lr, float beta1, float beta2, float eps) {
  __shared__ uint8_t imp[FIT_MAX_BPC];
  __shared__ float coef[2];
  const int b0 = blockIdx.x * bpc;
  const int nel = bpc * G.ptot;
  FitElem e0;
  e0.live = false;
  e0.k = -1;
  if ((int)threadIdx.x < nel) fit_elem_load(e0, G, threadIdx.x, b0, batch);
  const int t = step[parity] + 1;
  if ((int)threadIdx.x < bpc) {
    const int b = b0 + threadIdx.x;
    bool im = false;
    if (b < batch) {
      const float l = loss[b];
      im = l < best_loss[b];
      if (im) { best_loss[b] = l; best_iter[b] = t; }
      if (t == 1 && first_loss != nullptr) first_loss[b] = l;
    }
    imp[threadIdx.x] = im ? 1 : 0;
  }
  if (threadIdx.x == FIT_THREADS - 1) {                      // the bias corrections once per CTA (two powf are ~300
    const float bc1 = 1.f - powf(beta1, (float)t), bc2 = 1.f - powf(beta2, (float)t);   // instructions: per thread they were
    coef[0] = lr / bc1;                                      // two thirds of the kernel's instruction count)
    coef[1] = rsqrtf(bc2);
  }
  __syncthreads();
  const float step_size = coef[0], inv_sqrt_bc2 = coef[1];
  if ((int)threadIdx.x < nel) fit_elem_store(e0, G, imp, beta1, beta2, step_size, inv_sqrt_bc2, eps);
  for (int idx = threadIdx.x + FIT_THREADS; idx < nel; idx += FIT_THREADS) {   // rows longer than the CTA
    FitElem e;
    fit_elem_load(e, G, idx, b0, batch);
    fit_elem_store(e, G, imp, beta1, beta2, step_size, inv_sqrt_bc2, eps);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) step[1 - parity] = t;
}

}  // namespace b200smpl

using namespace b200smpl;

extern "C" {

int b200smpl_fit_loss(const float* joints, const float* cam, const int32_t* joint_map, const float* label,
                      const uint8_t* vis, const float* betas, int batch, int num_joints, int nmap, int num_betas,
                      float proj_wh, float norm_wh, float log_var, float shape_weight, float* loss_per_body,
                      float* grad_joints, float* grad_cam, float* grad_betas, void* stream) {
  B200_NVTX("b200smpl_fit_loss");
  if (!joints || !cam || !joint_map || !label || !betas || !loss_per_body || !grad_joints || !grad_cam || batch < 1 ||
      nmap < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  // mean(beta^2) over no betas would be 0 / 0 = NaN for every body, whatever shape_weight is
  if (num_joints < 1 || num_betas < 1) return fail(B200SMPL_ERR_INVALID, "num_joints and num_betas must be >= 1");
  LaunchTimer _timer("fit_loss", (cudaStream_t)stream);
  fit_loss_kernel<<<(batch + 3) / 4, 128, 0, (cudaStream_t)stream>>>(joints, cam, joint_map, label, vis, betas, batch,
                                                                     num_joints, nmap, num_betas, proj_wh, norm_wh, log_var,
                                                                     shape_weight, loss_per_body, grad_joints, grad_cam,
                                                                     grad_betas);
  B200_LAUNCH_CHECK("fit_loss");
  return 0;
}

int b200smpl_fit_mark_best(const float* loss_per_body, float* best_loss, int32_t* best_iter, uint8_t* improved,
                           int32_t* step, int batch, void* stream) {
  B200_NVTX("b200smpl_fit_mark_best");
  if (!loss_per_body || !best_loss || !best_iter || !improved || !step || batch < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  fit_mark_kernel<<<(batch + 255) / 256, 256, 0, (cudaStream_t)stream>>>(loss_per_body, best_loss, best_iter, improved,
                                                                         step, batch);
  B200_LAUNCH_CHECK("fit_mark");
  return 0;
}

int b200smpl_fit_adam_step(float* params, const float* grad, const float* grad_extra, float* exp_avg, float* exp_avg_sq,
                           float* best_params, const uint8_t* improved, const uint8_t* frozen_cols, int32_t* step,
                           int commit_step, int batch, int cols, float lr, float beta1, float beta2, float eps,
                           void* stream) {
  B200_NVTX("b200smpl_fit_adam_step");
  if (!params || !grad || !exp_avg || !exp_avg_sq || !best_params || !improved || !step || batch < 1 || cols < 1)
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  const long long n = (long long)batch * cols;
  const unsigned grid = (unsigned)std::min<long long>((n + 255) / 256, 148 * 8);
  fit_adam_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(params, grad, grad_extra, exp_avg, exp_avg_sq, best_params,
                                                          improved, frozen_cols, step, commit_step, batch, cols, lr, beta1,
                                                          beta2, eps);
  B200_LAUNCH_CHECK("fit_adam");
  return 0;
}

int b200smpl_fit_update(const b200smpl_fit_group* groups, int ngroups, const float* loss_per_body, float* best_loss,
                        int32_t* best_iter, float* first_loss, int32_t* step, int parity, int batch, float lr, float beta1,
                        float beta2, float eps, void* stream) {
  B200_NVTX("b200smpl_fit_update");
  if (!groups || ngroups < 1 || ngroups > B200SMPL_FIT_MAX_GROUPS || !loss_per_body || !best_loss || !best_iter || !step ||
      batch < 1 || (parity != 0 && parity != 1))
    return fail(B200SMPL_ERR_INVALID, "bad argument");
  FitGroups G;
  memset(&G, 0, sizeof(G));
  G.n = ngroups;
  for (int k = 0; k < ngroups; ++k) {
    const b200smpl_fit_group& q = groups[k];
    if (!q.params || !q.grad || !q.exp_avg || !q.exp_avg_sq || !q.best_params || q.cols < 1)
      return fail(B200SMPL_ERR_INVALID, "bad parameter group");
    G.g[k] = q;
    G.ptot += q.cols;
  }
  const int bpc = std::max(1, std::min(FIT_MAX_BPC, FIT_THREADS / G.ptot));
  LaunchTimer _timer("fit_update", (cudaStream_t)stream);
  fit_update_kernel<<<(batch + bpc - 1) / bpc, FIT_THREADS, 0, (cudaStream_t)stream>>>(G, bpc, loss_per_body, best_loss, best_iter,
                                                                                      first_loss, step, parity, batch, lr, beta1,
                                                                                      beta2, eps);
  B200_LAUNCH_CHECK("fit_update");
  return 0;
}

}  // extern "C"
