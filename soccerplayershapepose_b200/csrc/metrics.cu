// Reconstruction errors on the device: per body, the mean Euclidean distance between predicted and target points
// (PVE on the vertices, MPJPE on mapped joint rows), plain, scale-corrected (SC) and Procrustes-aligned (PA).  The
// reference computes them on the host after a device -> host copy (metrics/train_loss_and_metrics_tracker.py over
// utils/eval_utils.py, one numpy SVD per body).  The definition is stated once in DESIGN.md section 13 and restated
// in fp64 by oracle/metrics_oracle.py:
//
//   E(P, Q)  = (1/N) sum_i |p_i - q_i|
//   SC       p_i' = (p_i - mu_P) r_Q / r_P + mu_Q,           r = sqrt(sum |p_i - mu|^2 / N)
//   PA       p_i' = s R (p_i - mu_P) + mu_Q,  R in SO(3) maximising tr(R K), K = sum x_i y_i^T,
//            s = tr(R K) / sum |x_i|^2    (x, y the centred points)
//   all predicted points coincident: p_i' = mu_Q;  a non-finite input point: NaN in the three columns of its set
//
// Design: one CTA per body, so every reduction runs in a fixed order inside one CTA and a body's result does not
// depend on its batch position or on the launch.  Pass 1 streams the body's points once and accumulates the plain
// distance and, in fp64, the moments of the points shifted by the set's first point (sum a, sum |a|^2, sum a b^T with
// a = p - p_0, b = q - q_0; p - p_0 of two fp32 values is exact in fp64, so coincident points give exactly zero
// spread and the moments do not cancel at large translations).  Thread 0 solves the vertex transforms and thread 32
// the joint transforms, concurrently, in fp64: SC is a ratio, PA is Horn's quaternion method (top eigenvector of the
// 4x4 symmetric matrix built from K, by cyclic Jacobi), which yields a proper rotation by construction.  Pass 2
// re-reads the points from L2 (measured against staging them in shared memory: DESIGN.md section 13), centres them in
// fp64, and forms the SC and PA distances in fp32 from the centred coordinates.  Loads are scalar and coalesced (a
// warp reads 32 consecutive 12-byte points with three 4-byte loads), so any 4-byte-aligned input works.
#include <cmath>

#include "common.cuh"

namespace b200smpl {
namespace {

constexpr int RE_THREADS = 256;
constexpr int RE_WARPS = RE_THREADS / 32;
constexpr int RE_NMOM = 17;                   // sum a (3), sum b (3), sum |a|^2, sum |b|^2, sum a b^T (9)
constexpr int RE_JACOBI_SWEEPS = 12;

struct ReArgs {
  int V, NJ, M;
  const float* pv;
  const float* tv;
  const float* pj;
  const float* tj;
  const int32_t* map;
  float* out;
};

// one point set of a body: point i is rows[idx(i)] of pred / tgt
struct PointSet {
  const float* p;
  const float* q;
  const int32_t* map;                         // NULL: identity
  int n;
  __device__ __forceinline__ int row(int i) const { return map ? __ldg(map + i) : i; }
};

// the transforms of one set, as pass 2 reads them
struct Xform {
  double mp[3], mq[3];                        // mu_P, mu_Q
  float ssc;                                  // r_Q / r_P (0 when degenerate)
  float sr[9];                                // s R, row-major
  int finite;
};

__device__ __forceinline__ void load3(const float* base, int r, float v[3]) {
  v[0] = __ldg(base + 3 * (size_t)r);
  v[1] = __ldg(base + 3 * (size_t)r + 1);
  v[2] = __ldg(base + 3 * (size_t)r + 2);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// CTA sum of n per-thread values into dst[0..n): a butterfly inside each warp, then warps in index order
template <int N>
__device__ __forceinline__ void block_sum(double (&v)[N], double (*part)[RE_WARPS], double* dst) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    const double s = warp_sum(v[k]);
    if (lane == 0) part[k][warp] = s;
  }
  __syncthreads();
  if (threadIdx.x < N) {
    double s = 0.0;
    for (int w = 0; w < RE_WARPS; ++w) s += part[threadIdx.x][w];
    dst[threadIdx.x] = s;
  }
  __syncthreads();
}

// pass 1 of one set: [0] plain distance sum, [1..18) the shifted moments
__device__ __forceinline__ void moments(const PointSet& s, double (*part)[RE_WARPS], double* dst, float (*first)[3]) {
  float p0[3], q0[3];
  load3(s.p, s.row(0), p0);
  load3(s.q, s.row(0), q0);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      first[0][c] = p0[c];
      first[1][c] = q0[c];
    }
  }
  double acc[1 + RE_NMOM];
#pragma unroll
  for (int k = 0; k < 1 + RE_NMOM; ++k) acc[k] = 0.0;
  for (int i = threadIdx.x; i < s.n; i += RE_THREADS) {
    const int r = s.row(i);
    float p[3], q[3];
    load3(s.p, r, p);
    load3(s.q, r, q);
    const float dx = p[0] - q[0], dy = p[1] - q[1], dz = p[2] - q[2];
    acc[0] += (double)sqrtf(dx * dx + dy * dy + dz * dz);
    double a[3], b[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      a[c] = (double)p[c] - (double)p0[c];
      b[c] = (double)q[c] - (double)q0[c];
      acc[1 + c] += a[c];
      acc[4 + c] += b[c];
      acc[7] = fma(a[c], a[c], acc[7]);
      acc[8] = fma(b[c], b[c], acc[8]);
    }
#pragma unroll
    for (int r2 = 0; r2 < 3; ++r2)
#pragma unroll
      for (int c = 0; c < 3; ++c) acc[9 + 3 * r2 + c] = fma(a[r2], b[c], acc[9 + 3 * r2 + c]);
  }
  block_sum(acc, part, dst);
}

// cyclic Jacobi on the symmetric 4x4 matrix with upper triangle a (row-major, 10 entries; destroyed): returns the
// largest eigenvalue and its unit eigenvector in q.  A fixed sweep cap bounds the time a NaN input takes.
__device__ __forceinline__ constexpr int ut(int i, int j) { return i <= j ? i * 4 - i * (i - 1) / 2 + (j - i)
                                                                          : j * 4 - j * (j - 1) / 2 + (i - j); }

__device__ __forceinline__ double top_eigenvector4(double (&a)[10], double q[4]) {
  double V[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) V[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < RE_JACOBI_SWEEPS; ++sweep) {
    double off = 0.0, diag = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      diag += a[ut(i, i)] * a[ut(i, i)];
#pragma unroll
      for (int j = i + 1; j < 4; ++j) off += a[ut(i, j)] * a[ut(i, j)];
    }
    if (!(off > 1e-30 * diag)) break;                     // converged (or all zero)
#pragma unroll
    for (int p = 0; p < 3; ++p)
#pragma unroll
      for (int r = p + 1; r < 4; ++r) {
        const double apr = a[ut(p, r)];
        if (apr == 0.0) continue;
        const double theta = (a[ut(r, r)] - a[ut(p, p)]) / (2.0 * apr);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
        const double c = rsqrt(fma(t, t, 1.0)), s = t * c;
        a[ut(p, p)] -= t * apr;
        a[ut(r, r)] += t * apr;
        a[ut(p, r)] = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (k == p || k == r) continue;
          const double akp = a[ut(k, p)], akr = a[ut(k, r)];
          a[ut(k, p)] = c * akp - s * akr;
          a[ut(k, r)] = s * akp + c * akr;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const double vkp = V[k][p], vkr = V[k][r];
          V[k][p] = c * vkp - s * vkr;
          V[k][r] = s * vkp + c * vkr;
        }
      }
  }
  double top = a[ut(0, 0)];
#pragma unroll
  for (int k = 0; k < 4; ++k) q[k] = V[k][0];
#pragma unroll
  for (int i = 1; i < 4; ++i)
    if (a[ut(i, i)] > top) {
      top = a[ut(i, i)];
#pragma unroll
      for (int k = 0; k < 4; ++k) q[k] = V[k][i];
    }
  return top;
}

// the SC and PA transforms of one set from its pass-1 sums m[0..18)
__device__ __forceinline__ void solve(const double* m, const float p0[3], const float q0[3], int n, Xform* x) {
  const double inv_n = 1.0 / (double)n;
  double sa[3], sb[3];
  bool finite = true;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    sa[c] = m[1 + c];
    sb[c] = m[4 + c];
    x->mp[c] = (double)p0[c] + sa[c] * inv_n;
    x->mq[c] = (double)q0[c] + sb[c] * inv_n;
    finite = finite && isfinite(x->mp[c]) && isfinite(x->mq[c]);
  }
  // centred second moments: sum |x|^2, sum |y|^2, K = sum x y^T
  const double sxx = fmax(m[7] - (sa[0] * sa[0] + sa[1] * sa[1] + sa[2] * sa[2]) * inv_n, 0.0);
  const double syy = fmax(m[8] - (sb[0] * sb[0] + sb[1] * sb[1] + sb[2] * sb[2]) * inv_n, 0.0);
  double K[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) K[r][c] = m[9 + 3 * r + c] - sa[r] * sb[c] * inv_n;
  // Horn: for x -> y the unit quaternion maximising sum y.(R x) is the top eigenvector of N(K)
  double N[10] = {K[0][0] + K[1][1] + K[2][2], K[1][2] - K[2][1], K[2][0] - K[0][2], K[0][1] - K[1][0],
                  K[0][0] - K[1][1] - K[2][2], K[0][1] + K[1][0], K[2][0] + K[0][2],
                  -K[0][0] + K[1][1] - K[2][2], K[1][2] + K[2][1],
                  -K[0][0] - K[1][1] + K[2][2]};
  double q[4];
  const double trRK = top_eigenvector4(N, q);               // the top eigenvalue is max tr(R K)
  const double qq = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  const double w = q[0], i = q[1], j = q[2], k = q[3];
  const double R[3][3] = {{w * w + i * i - j * j - k * k, 2 * (i * j - w * k), 2 * (i * k + w * j)},
                          {2 * (j * i + w * k), w * w - i * i + j * j - k * k, 2 * (j * k - w * i)},
                          {2 * (k * i - w * j), 2 * (k * j + w * i), w * w - i * i - j * j + k * k}};
  // all predicted points coincident (sxx is exactly zero then): p' = mu_Q
  const double spa = sxx > 0.0 ? trRK / sxx : 0.0;
  x->ssc = sxx > 0.0 ? (float)sqrt(syy / sxx) : 0.f;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) x->sr[3 * r + c] = (float)(spa * R[r][c] / qq);
  x->finite = finite;
}

// pass 2 of one set: [0] SC distance sum, [1] PA distance sum
__device__ __forceinline__ void aligned_sums(const PointSet& s, const Xform& x, double (*part)[RE_WARPS],
                                             double* dst) {
  double acc[2] = {0.0, 0.0};
  const float ssc = x.ssc;
  float sr[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) sr[k] = x.sr[k];
  for (int i = threadIdx.x; i < s.n; i += RE_THREADS) {
    const int r = s.row(i);
    float p[3], q[3], xc[3], yc[3];
    load3(s.p, r, p);
    load3(s.q, r, q);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      xc[c] = (float)((double)p[c] - x.mp[c]);
      yc[c] = (float)((double)q[c] - x.mq[c]);
    }
    float d2 = 0.f, e2 = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float d = fmaf(ssc, xc[c], -yc[c]);
      const float e = fmaf(sr[3 * c], xc[0], fmaf(sr[3 * c + 1], xc[1], fmaf(sr[3 * c + 2], xc[2], -yc[c])));
      d2 = fmaf(d, d, d2);
      e2 = fmaf(e, e, e2);
    }
    acc[0] += (double)sqrtf(d2);
    acc[1] += (double)sqrtf(e2);
  }
  block_sum(acc, part, dst);
}

__global__ void __launch_bounds__(RE_THREADS, 2) recon_errors(ReArgs a) {
  __shared__ double part[1 + RE_NMOM][RE_WARPS];
  __shared__ double mom[2][1 + RE_NMOM];
  __shared__ double fin[2][2];
  __shared__ float first[2][2][3];            // [set][pred / target][xyz]
  __shared__ Xform xf[2];
  const int b = blockIdx.x;
  PointSet sets[2];
  sets[0] = PointSet{a.pv ? a.pv + (size_t)b * a.V * 3 : nullptr, a.tv ? a.tv + (size_t)b * a.V * 3 : nullptr,
                     nullptr, a.V};
  sets[1] = PointSet{a.pj ? a.pj + (size_t)b * a.NJ * 3 : nullptr, a.tj ? a.tj + (size_t)b * a.NJ * 3 : nullptr,
                     a.map, a.M};
  const bool on[2] = {a.pv != nullptr, a.pj != nullptr};
#pragma unroll
  for (int k = 0; k < 2; ++k)
    if (on[k]) moments(sets[k], part, mom[k], first[k]);
  if ((threadIdx.x & 31) == 0 && threadIdx.x < 64) {       // thread 0: vertices, thread 32: joints
    const int k = threadIdx.x >> 5;
    if (k ? on[1] : on[0]) solve(mom[k], first[k][0], first[k][1], k ? a.M : a.V, &xf[k]);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 2; ++k)
    if (on[k]) aligned_sums(sets[k], xf[k], part, fin[k]);
  if (threadIdx.x < 2 && (threadIdx.x ? on[1] : on[0])) {
    const int k = threadIdx.x;
    const double inv_n = 1.0 / (double)(k ? a.M : a.V);
    float* o = a.out + (size_t)b * 6 + 3 * k;
    const float nan = __int_as_float(0x7fc00000);
    o[0] = xf[k].finite ? (float)(mom[k][0] * inv_n) : nan;
    o[1] = xf[k].finite ? (float)(fin[k][0] * inv_n) : nan;
    o[2] = xf[k].finite ? (float)(fin[k][1] * inv_n) : nan;
  }
}

}  // namespace
}  // namespace b200smpl

using namespace b200smpl;

extern "C" {

int b200smpl_reconstruction_errors(const b200smpl_recon_error_args* args, float* out, void* stream) {
  B200_NVTX("b200smpl_reconstruction_errors");
  if (!args) return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: args is NULL");
  const b200smpl_recon_error_args& p = *args;
  if (p.batch < 1) return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: need batch >= 1");
  if (!out) return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: out is NULL");
  if ((p.pred_vertices == nullptr) != (p.target_vertices == nullptr) ||
      (p.pred_joints == nullptr) != (p.target_joints == nullptr))
    return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: a prediction and its target must both be given or "
                                      "both be NULL");
  const bool verts = p.pred_vertices != nullptr, joints = p.pred_joints != nullptr;
  if (!verts && !joints) return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: nothing to do");
  if (verts && p.num_verts < 1) return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: need num_verts >= 1");
  if (joints && (p.num_joints < 1 || p.num_map < 1))
    return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: need num_joints >= 1 and num_map >= 1");
  if (joints && !p.joint_map) return fail(B200SMPL_ERR_INVALID, "reconstruction_errors: joint_map is NULL");
  ReArgs a;
  a.V = verts ? p.num_verts : 0;
  a.NJ = joints ? p.num_joints : 0;
  a.M = joints ? p.num_map : 0;
  a.pv = p.pred_vertices;
  a.tv = p.target_vertices;
  a.pj = p.pred_joints;
  a.tj = p.target_joints;
  a.map = joints ? p.joint_map : nullptr;
  a.out = out;
  LaunchTimer _timer("recon_errors", (cudaStream_t)stream);
  recon_errors<<<(unsigned)p.batch, RE_THREADS, 0, (cudaStream_t)stream>>>(a);
  B200_LAUNCH_CHECK("recon_errors");
  return 0;
}

}  // extern "C"
