// The regressor's input, the 1 + K channel "proxy representation" of a detection, built on the device: channel 0 is
// the binary mask resized by nearest neighbour, channels 1 + j are Gaussian heatmaps of the K keypoints (the
// reference builds it on the host per crop: create_proxy_representation, predict_3D.py:67-81, over
// convert_2Djoints_to_gaussian_heatmaps, label_conversions.py:58-87).  The definition is stated once in DESIGN.md
// section 12 and restated in fp64 by oracle/proxy_oracle.py:
//
//   mask      out[0][y][x] = mask[(y in) / out][(x in) / out] != 0   (exact integer division)
//   centre    (cu, cv) = trunc(kp * (out / in)), in double precision; zero channel when vis = 0, the keypoint is not
//             finite or a truncated centre leaves the int16 range
//   heatmap   out[1 + j][v][u] = exp(-((u - cu) / std)^2 / 2) * exp(-((v - cv) / std)^2 / 2)
//
// Design: the kernel reads ~1/18 of what it writes, so it is bound by HBM writes.  One CTA per (body, band of
// PX_TH rows, tile of PX_TW columns).  The CTA computes the keypoint centres and the separable Gaussian factors of
// its columns and rows into shared memory, then its warps stream the tile out: each warp takes one contiguous span
// of the output at a time -- one (channel, row) segment in NCHW, one row of pixels x channels in NHWC -- and writes
// it with 16-byte streaming stores, with scalar stores for the unaligned head and tail of the span.
#include <cmath>

#include "common.cuh"

namespace b200smpl {
namespace {

constexpr int PX_THREADS = 256;
constexpr int PX_WARPS = PX_THREADS / 32;
constexpr int PX_TW = 256;                    // columns per tile
constexpr int PX_TH = 32;                     // rows per tile (16: 5 % slower at B = 256, 8: 11 %)
constexpr int PX_MAX_K = B200SMPL_PROXY_MAX_KEYPOINTS;
constexpr int PX_MAX_WH = 16384;

struct ProxyArgs {
  int B, in_wh, S, K, C, ntx, nty;
  float inv_std;
  double scale;                               // out_wh / in_wh
  const uint8_t* masks;
  const float* kp;
  const uint8_t* vis;
};

// Gaussian factor exp(-(d / std)^2 / 2) of an integer offset d (exact in fp32 for the sizes the entry admits)
__device__ __forceinline__ float gauss(int d, float inv_std) {
  const float t = (float)d * inv_std;
  return expf(-0.5f * t * t);
}

// CL = false (NCHW): gx[j][i] at j * PX_TW + i.  CL = true (NHWC): gx[i][j] at i * K + j, so that a span's
// consecutive elements read consecutive words.  gy[r][j] at r * K + j in both.
template <bool CL>
__global__ void __launch_bounds__(PX_THREADS) proxy_rep(ProxyArgs a, float* __restrict__ out) {
  __shared__ __align__(16) float gx[PX_MAX_K * PX_TW];
  __shared__ float gy[PX_TH * PX_MAX_K];
  __shared__ int sx[PX_TW];                   // source column of each tile column
  __shared__ int cu[PX_MAX_K], cv[PX_MAX_K], ok[PX_MAX_K];
  const int tile = blockIdx.x % (a.ntx * a.nty);
  const int b = blockIdx.x / (a.ntx * a.nty);
  const int x0 = (tile % a.ntx) * PX_TW, y0 = (tile / a.ntx) * PX_TH;
  const int nx = min(PX_TW, a.S - x0), ny = min(PX_TH, a.S - y0);
  const int K = a.K, C = a.C;
  if (threadIdx.x < K) {
    const int j = threadIdx.x;
    const float kx = a.kp[((size_t)b * K + j) * 2], ky = a.kp[((size_t)b * K + j) * 2 + 1];
    const double u = (double)kx * a.scale, v = (double)ky * a.scale;
    // NaN fails both comparisons; a truncated centre in [-32768, 32767] is what an int16 cast keeps
    const bool in16 = u > -32769.0 && u < 32768.0 && v > -32769.0 && v < 32768.0;
    ok[j] = in16 && (a.vis == nullptr || a.vis[(size_t)b * K + j] != 0);
    cu[j] = in16 ? (int)u : 0;                // (int) truncates toward zero, as astype(np.int16)
    cv[j] = in16 ? (int)v : 0;
  }
  for (int i = threadIdx.x; i < nx; i += PX_THREADS) sx[i] = (int)(((long long)(x0 + i) * a.in_wh) / a.S);
  __syncthreads();
  for (int e = threadIdx.x; e < K * nx; e += PX_THREADS) {
    const int j = e / nx, i = e - j * nx;
    const float g = ok[j] ? gauss(x0 + i - cu[j], a.inv_std) : 0.f;
    gx[CL ? i * K + j : j * PX_TW + i] = g;
  }
  for (int e = threadIdx.x; e < K * ny; e += PX_THREADS) {
    const int r = e / K, j = e - r * K;
    gy[e] = ok[j] ? gauss(y0 + r - cv[j], a.inv_std) : 0.f;
  }
  __syncthreads();

  const uint8_t* mask = a.masks + (size_t)b * a.in_wh * a.in_wh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t plane = (size_t)a.S * a.S;
  // spans: NCHW (channel, row) segments of nx floats, channel-major; NHWC rows of nx * C floats
  const int nspan = CL ? ny : C * ny;
  const int len = CL ? nx * C : nx;
  for (int s = warp; s < nspan; s += PX_WARPS) {
    const int c = CL ? 0 : s / ny;
    const int r = CL ? s : s - c * ny;
    const int y = y0 + r;
    const uint8_t* mrow = mask + (size_t)(((long long)y * a.in_wh) / a.S) * a.in_wh;
    const float* gyr = gy + r * K;
    float* p = CL ? out + (size_t)b * C * plane + ((size_t)y * a.S + x0) * C
                  : out + ((size_t)b * C + c) * plane + (size_t)y * a.S + x0;
    // element i of the span
    auto value = [&](int i) -> float {
      if (CL) {
        const int px = i / C, ch = i - px * C;
        return ch == 0 ? (mrow[sx[px]] ? 1.f : 0.f) : gx[px * K + ch - 1] * gyr[ch - 1];
      }
      return c == 0 ? (mrow[sx[i]] ? 1.f : 0.f) : gx[(c - 1) * PX_TW + i] * gyr[c - 1];
    };
    const int head = min(len, (int)(((16u - ((unsigned)(uintptr_t)p & 15u)) & 15u) >> 2));
    const int nvec = (len - head) >> 2;
    const int tail = head + 4 * nvec;
    if (lane < head) p[lane] = value(lane);
    if (lane < len - tail) p[tail + lane] = value(tail + lane);
    float4* pv = reinterpret_cast<float4*>(p + head);
    if (!CL && c > 0 && head == 0) {          // aligned NCHW heatmap segment: 16-byte shared loads as well
      const float4* gv = reinterpret_cast<const float4*>(gx + (c - 1) * PX_TW);
      const float f = gyr[c - 1];
      for (int v = lane; v < nvec; v += 32) {
        const float4 g = gv[v];
        __stcs(pv + v, make_float4(g.x * f, g.y * f, g.z * f, g.w * f));
      }
    } else if (CL) {                          // one division per 16 bytes, then step through pixel x channel
      for (int v = lane; v < nvec; v += 32) {
        const int i = head + 4 * v;
        int px = i / C, ch = i - px * C;
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          o[k] = ch == 0 ? (mrow[sx[px]] ? 1.f : 0.f) : gx[px * K + ch - 1] * gyr[ch - 1];
          if (++ch == C) { ch = 0; ++px; }
        }
        __stcs(pv + v, make_float4(o[0], o[1], o[2], o[3]));
      }
    } else {
      for (int v = lane; v < nvec; v += 32) {
        const int i = head + 4 * v;
        __stcs(pv + v, make_float4(value(i), value(i + 1), value(i + 2), value(i + 3)));
      }
    }
  }
}

}  // namespace
}  // namespace b200smpl

using namespace b200smpl;

extern "C" {

int b200smpl_proxy_representation(const b200smpl_proxy_args* args, float* out, void* stream) {
  B200_NVTX("b200smpl_proxy_representation");
  if (!args) return fail(B200SMPL_ERR_INVALID, "proxy_representation: args is NULL");
  const b200smpl_proxy_args& p = *args;
  if (p.batch < 1 || p.in_wh < 1 || p.in_wh > PX_MAX_WH || p.out_wh < 1 || p.out_wh > PX_MAX_WH ||
      p.num_keypoints < 1 || p.num_keypoints > PX_MAX_K)
    return fail(B200SMPL_ERR_INVALID, "proxy_representation: need batch >= 1, 1 <= in_wh, out_wh <= 16384 and "
                                      "1 <= num_keypoints <= " + std::to_string(PX_MAX_K));
  if (!(p.std > 0.f) || !std::isfinite(p.std))
    return fail(B200SMPL_ERR_INVALID, "proxy_representation: need a finite std > 0");
  if (p.channels_last != 0 && p.channels_last != 1)
    return fail(B200SMPL_ERR_INVALID, "proxy_representation: channels_last must be 0 or 1");
  if (!p.masks || !p.keypoints || !out) return fail(B200SMPL_ERR_INVALID, "proxy_representation: NULL pointer");
  ProxyArgs a;
  a.B = p.batch;
  a.in_wh = p.in_wh;
  a.S = p.out_wh;
  a.K = p.num_keypoints;
  a.C = 1 + p.num_keypoints;
  a.ntx = (p.out_wh + PX_TW - 1) / PX_TW;
  a.nty = (p.out_wh + PX_TH - 1) / PX_TH;
  a.inv_std = 1.f / p.std;
  a.scale = (double)p.out_wh / (double)p.in_wh;
  a.masks = p.masks;
  a.kp = p.keypoints;
  a.vis = p.vis;
  const long long grid = (long long)p.batch * a.ntx * a.nty;
  if (grid > 0x7fffffffLL) return fail(B200SMPL_ERR_INVALID, "proxy_representation: batch too large for one launch");
  const char* name = p.channels_last ? "proxy_rep_nhwc" : "proxy_rep_nchw";
  LaunchTimer _timer(name, (cudaStream_t)stream);
  if (p.channels_last)
    proxy_rep<true><<<(unsigned)grid, PX_THREADS, 0, (cudaStream_t)stream>>>(a, out);
  else
    proxy_rep<false><<<(unsigned)grid, PX_THREADS, 0, (cudaStream_t)stream>>>(a, out);
  B200_LAUNCH_CHECK(name);
  return 0;
}

}  // extern "C"
