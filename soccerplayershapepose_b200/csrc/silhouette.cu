// Batched silhouette rasteriser for posed SMPL meshes: hard (binary) coverage, the SoftRas / SoftSilhouetteShader
// soft silhouette, its hand-written backward and a fused loss for the fitting loop (the reference renders the posed
// mesh with its neural renderer every iteration, player_recon.py:1226-1229, 1084-1087).  The definition is stated
// once in DESIGN.md section 11 and restated densely in fp64 by oracle/silhouette_oracle.py:
//
//   camera    R = I, t = cam_t[b], K = [[f,0,S/2],[0,f,S/2],[0,0,1]]:  u = f (x+tx)/(z+tz) + S/2, v likewise with y;
//             image element [i][j] is the pixel centred at (u, v) = (j + 0.5, i + 0.5), no vertical flip
//   dropped   faces with a vertex at z + tz <= 1e-3 or with |projected signed area| < 1e-8 px^2; winding ignored
//   hard      sigma == 0: 1 where the pixel centre lies inside or on the boundary of a kept face
//   soft      sigma  > 0: D_f = sigmoid(+-d^2/sigma) (+ inside, - outside), d = distance to the face's nearest edge
//             segment; an outside face with d^2 > sigma ln(1/eps - 1), eps = 1e-4, contributes nothing;
//             alpha = 1 - prod_f (1 - D_f)
//
// Design: one CTA per body (the forward may split a body's row bands over several CTAs so that small batches fill
// the GPU).  The CTA projects the body's vertices into shared memory, then walks bands of 32 image rows: it compacts
// the faces whose bounding box (grown by the blur radius) meets the band into a shared list -- in face order, so the
// per-pixel products and sums are deterministic -- and each warp evaluates 32x8-pixel tiles (lane = column, 8 rows
// per lane) against the band list, filtered per tile 32 faces at a time with a ballot.
// The backward keeps, per pixel, the product of the unsaturated factors (1 - D_f) and the count of saturated ones,
// so that prod_{g != f} (1 - D_g) is exact without dividing by a vanishing factor.  d alpha / d(u, v) is reduced
// over the warp and accumulated per vertex in shared memory; the flush applies the chain rule through the
// projection, writes grad_vertices without global atomics and reduces grad_t over the block.
// The gradient-free loss runs the forward's per-pixel pass and sums (alpha - target)^2 instead of writing alpha; when
// it splits a body's bands, the CTAs form a cluster whose partial sums are added in rank order.
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace b200smpl {
namespace {

constexpr int SIL_THREADS = 512;
constexpr int SIL_WARPS = SIL_THREADS / 32;
constexpr int SIL_TW = 32;          // tile width (lane = column)
constexpr int SIL_TH = 8;           // tile height (rows per lane)
constexpr int SIL_BAND = 32;        // rows per band
constexpr float SIL_EPS = 1e-4f;    // contribution cut-off of an outside face
constexpr float SIL_ZMIN = 1e-3f;   // a face with a vertex at z + tz <= ZMIN is dropped
constexpr float SIL_AREA_MIN = 1e-8f;
constexpr float SIL_SAT = 1e-30f;   // 1 - D_f below this counts as saturated (exactly 0 in the products)
constexpr float SIL_SLACK = 1e-2f;  // px added to every culling box (the per-pixel tests are exact)
constexpr int SIL_MAX_CLUSTER = 8;  // CTAs per body of sil_loss_value (the portable cluster size)

struct SilArgs {
  int V, F, S;
  float f, c, sigma, inv_sigma, r2, rad;
  const float* verts;
  const float* cam_t;
  const int32_t* faces;
};

struct Face {
  float ax, ay, bx, by, cx, cy;
  float e0x, e0y, e1x, e1y, e2x, e2y;   // A->B, B->C, C->A
  float i0, i1, i2;                     // 1 / |e|^2
  float xmin, xmax, ymin, ymax;
};

__device__ __forceinline__ void face_setup(Face& F, const float2* P, const uint16_t* L, int k) {
  const float2 A = P[L[3 * k]], B = P[L[3 * k + 1]], C = P[L[3 * k + 2]];
  F.ax = A.x; F.ay = A.y; F.bx = B.x; F.by = B.y; F.cx = C.x; F.cy = C.y;
  F.e0x = B.x - A.x; F.e0y = B.y - A.y;
  F.e1x = C.x - B.x; F.e1y = C.y - B.y;
  F.e2x = A.x - C.x; F.e2y = A.y - C.y;
  F.i0 = 1.f / (F.e0x * F.e0x + F.e0y * F.e0y);
  F.i1 = 1.f / (F.e1x * F.e1x + F.e1y * F.e1y);
  F.i2 = 1.f / (F.e2x * F.e2x + F.e2y * F.e2y);
  F.xmin = fminf(A.x, fminf(B.x, C.x)); F.xmax = fmaxf(A.x, fmaxf(B.x, C.x));
  F.ymin = fminf(A.y, fminf(B.y, C.y)); F.ymax = fmaxf(A.y, fmaxf(B.y, C.y));
}

__device__ __forceinline__ bool face_inside(const Face& F, float px, float py) {
  const float w0 = F.e0x * (py - F.ay) - F.e0y * (px - F.ax);
  const float w1 = F.e1x * (py - F.by) - F.e1y * (px - F.bx);
  const float w2 = F.e2x * (py - F.cy) - F.e2y * (px - F.cx);
  return (w0 >= 0.f && w1 >= 0.f && w2 >= 0.f) || (w0 <= 0.f && w1 <= 0.f && w2 <= 0.f);
}

// squared distance from p to segment (s, s + e); t = clamped parameter of the nearest point, q = p - nearest point
__device__ __forceinline__ float seg_d2(float px, float py, float sx, float sy, float ex, float ey, float inv, float& t,
                                        float& qx, float& qy) {
  const float dx = px - sx, dy = py - sy;
  t = fminf(fmaxf((dx * ex + dy * ey) * inv, 0.f), 1.f);
  qx = dx - t * ex;
  qy = dy - t * ey;
  return qx * qx + qy * qy;
}

// Soft term of face F at pixel p.  Returns false when the face contributes nothing (outside beyond the cut-off).
// D = D_f, om = 1 - D_f (both computed from one exp), sgn = +1 inside / -1 outside, ke / t / q describe the nearest
// edge (edge ke runs from vertex ke to vertex (ke + 1) % 3).
__device__ __forceinline__ bool soft_term(const Face& F, const SilArgs& a, float px, float py, float& D, float& om,
                                          float& sgn, int& ke, float& t, float& qx, float& qy) {
  if (px < F.xmin - a.rad || px > F.xmax + a.rad || py < F.ymin - a.rad || py > F.ymax + a.rad) return false;
  const bool in = face_inside(F, px, py);
  float t1, q1x, q1y, t2, q2x, q2y;
  float d2 = seg_d2(px, py, F.ax, F.ay, F.e0x, F.e0y, F.i0, t, qx, qy);
  ke = 0;
  const float d21 = seg_d2(px, py, F.bx, F.by, F.e1x, F.e1y, F.i1, t1, q1x, q1y);
  const float d22 = seg_d2(px, py, F.cx, F.cy, F.e2x, F.e2y, F.i2, t2, q2x, q2y);
  if (d21 < d2) { d2 = d21; ke = 1; t = t1; qx = q1x; qy = q1y; }
  if (d22 < d2) { d2 = d22; ke = 2; t = t2; qx = q2x; qy = q2y; }
  if (!in && d2 > a.r2) return false;
  sgn = in ? 1.f : -1.f;
  const float x = sgn * d2 * a.inv_sigma;
  D = 1.f / (1.f + expf(-x));
  om = 1.f / (1.f + expf(x));
  return true;
}

__device__ __forceinline__ bool tile_hit(const float2* P, const uint16_t* L, int k, float x0, float x1, float y0,
                                         float y1, float pad) {
  const float2 A = P[L[3 * k]], B = P[L[3 * k + 1]], C = P[L[3 * k + 2]];
  return fmaxf(A.x, fmaxf(B.x, C.x)) + pad >= x0 && fminf(A.x, fminf(B.x, C.x)) - pad <= x1 &&
         fmaxf(A.y, fmaxf(B.y, C.y)) + pad >= y0 && fminf(A.y, fminf(B.y, C.y)) - pad <= y1;
}

__device__ void project_body(const SilArgs& a, int b, float2* P) {
  const float tx = a.cam_t[3 * b], ty = a.cam_t[3 * b + 1], tz = a.cam_t[3 * b + 2];
  const float* X = a.verts + (size_t)b * a.V * 3;
  for (int v = threadIdx.x; v < a.V; v += blockDim.x) {
    const float x = X[3 * v], y = X[3 * v + 1], Z = X[3 * v + 2] + tz;
    P[v] = Z > SIL_ZMIN ? make_float2(a.f * (x + tx) / Z + a.c, a.f * (y + ty) / Z + a.c) : make_float2(NAN, NAN);
  }
}

// Faces that are kept and whose box grown by `pad` meets pixel centres [0.5, S - 0.5] x [y0, y1], compacted into L
// as vertex-index triples in face order.  Returns the count (block-uniform).
__device__ int band_list(const SilArgs& a, const float2* P, uint16_t* L, int* wcnt, float y0, float y1, float pad) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float x0 = 0.5f, x1 = a.S - 0.5f;
  int total = 0;
  for (int base = 0; base < a.F; base += blockDim.x) {
    const int f = base + threadIdx.x;
    bool hit = false;
    int i0 = 0, i1 = 0, i2 = 0;
    if (f < a.F) {
      i0 = a.faces[3 * f]; i1 = a.faces[3 * f + 1]; i2 = a.faces[3 * f + 2];
      if ((unsigned)i0 < (unsigned)a.V && (unsigned)i1 < (unsigned)a.V && (unsigned)i2 < (unsigned)a.V) {
        const float2 A = P[i0], B = P[i1], C = P[i2];
        const float area = 0.5f * ((B.x - A.x) * (C.y - A.y) - (B.y - A.y) * (C.x - A.x));
        hit = fabsf(area) >= SIL_AREA_MIN &&    // false for NaN: a vertex behind the near limit
              fmaxf(A.x, fmaxf(B.x, C.x)) + pad >= x0 && fminf(A.x, fminf(B.x, C.x)) - pad <= x1 &&
              fmaxf(A.y, fmaxf(B.y, C.y)) + pad >= y0 && fminf(A.y, fminf(B.y, C.y)) - pad <= y1;
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) wcnt[warp] = __popc(m);
    __syncthreads();
    int off = total, all = 0;
    for (int w = 0; w < SIL_WARPS; ++w) {
      const int cw = wcnt[w];
      off += w < warp ? cw : 0;
      all += cw;
    }
    if (hit) {
      const int k = off + __popc(m & ((1u << lane) - 1u));
      L[3 * k] = (uint16_t)i0; L[3 * k + 1] = (uint16_t)i1; L[3 * k + 2] = (uint16_t)i2;
    }
    total += all;
    __syncthreads();
  }
  return total;
}

// ---- forward -----------------------------------------------------------------------------------------------------
// VALUE = false: writes the tile's alpha.  VALUE = true: writes nothing and returns the lane's share of
// sum (alpha - target)^2 (the same per-pixel alpha and the same summation order as pass 1 of the fused loss).
template <bool VALUE>
__device__ float tile_fwd(const SilArgs& a, const float2* P, const uint16_t* L, int n, int row0, int col0,
                          float* __restrict__ alpha, const uint8_t* __restrict__ target) {
  const int lane = threadIdx.x & 31;
  const float px = col0 + lane + 0.5f;
  const float x0 = col0 + 0.5f, x1 = col0 + SIL_TW - 0.5f, y0 = row0 + 0.5f, y1 = row0 + SIL_TH - 0.5f;
  const float pad = a.rad + SIL_SLACK;
  const bool soft = a.sigma > 0.f;
  float prod[SIL_TH];
  int nsat[SIL_TH];
#pragma unroll
  for (int r = 0; r < SIL_TH; ++r) { prod[r] = 1.f; nsat[r] = 0; }
  for (int c0 = 0; c0 < n; c0 += 32) {
    const bool hit = c0 + lane < n && tile_hit(P, L, c0 + lane, x0, x1, y0, y1, pad);
    unsigned m = __ballot_sync(0xffffffffu, hit);
    while (m) {
      const int k = c0 + __ffs(m) - 1;
      m &= m - 1;
      Face F;
      face_setup(F, P, L, k);
#pragma unroll
      for (int r = 0; r < SIL_TH; ++r) {
        const float py = row0 + r + 0.5f;
        if (soft) {
          float D, om, sgn, t, qx, qy;
          int ke;
          if (soft_term(F, a, px, py, D, om, sgn, ke, t, qx, qy)) {
            if (om < SIL_SAT) ++nsat[r]; else prod[r] *= om;
          }
        } else if (px >= F.xmin && px <= F.xmax && py >= F.ymin && py <= F.ymax && face_inside(F, px, py)) {
          nsat[r] = 1;
        }
      }
    }
  }
  float lsum = 0.f;
  const int col = col0 + lane;
  if (col >= a.S) return lsum;
#pragma unroll
  for (int r = 0; r < SIL_TH; ++r) {
    const int row = row0 + r;
    if (row >= a.S) continue;
    const float al = nsat[r] ? 1.f : 1.f - prod[r];
    if (VALUE) {
      const float d = al - (target[(size_t)row * a.S + col] ? 1.f : 0.f);
      lsum += d * d;
    } else {
      alpha[(size_t)row * a.S + col] = al;
    }
  }
  return lsum;
}

__global__ void __launch_bounds__(SIL_THREADS, 1) sil_fwd(SilArgs a, float* __restrict__ alpha) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int wcnt[SIL_WARPS];
  float2* P = reinterpret_cast<float2*>(smem);
  uint16_t* L = reinterpret_cast<uint16_t*>(smem + (size_t)a.V * sizeof(float2));
  const int b = blockIdx.x;
  project_body(a, b, P);
  __syncthreads();
  float* out = alpha + (size_t)b * a.S * a.S;
  const int nbands = (a.S + SIL_BAND - 1) / SIL_BAND, ntc = (a.S + SIL_TW - 1) / SIL_TW;
  const int warp = threadIdx.x >> 5;
  for (int band = blockIdx.y; band < nbands; band += gridDim.y) {
    const int r0 = band * SIL_BAND;
    const int rows = min(SIL_BAND, a.S - r0);
    const int n = band_list(a, P, L, wcnt, r0 + 0.5f, r0 + rows - 0.5f, a.rad + SIL_SLACK);
    const int ntr = (rows + SIL_TH - 1) / SIL_TH;
    for (int tile = warp; tile < ntr * ntc; tile += SIL_WARPS)
      tile_fwd<false>(a, P, L, n, r0 + (tile / ntc) * SIL_TH, (tile % ntc) * SIL_TW, out, nullptr);
    __syncthreads();                                      // the next band rewrites L
  }
}

// ---- backward and fused loss -------------------------------------------------------------------------------------
// LOSS = false: g = grad_alpha.  LOSS = true: alpha is evaluated first, g = 2 weight (alpha - target) / S^2 and the
// lane's share of sum (alpha - target)^2 is returned.
template <bool LOSS>
__device__ float tile_bwd(const SilArgs& a, const float2* P, const uint16_t* L, int n, int row0, int col0,
                          const float* __restrict__ galpha, const uint8_t* __restrict__ target, float gscale,
                          float2* G) {
  const int lane = threadIdx.x & 31;
  const int col = col0 + lane;
  const float px = col + 0.5f;
  const float x0 = col0 + 0.5f, x1 = col0 + SIL_TW - 0.5f, y0 = row0 + 0.5f, y1 = row0 + SIL_TH - 0.5f;
  const float pad = a.rad + SIL_SLACK;
  float g[SIL_TH], prod[SIL_TH];
  int nsat[SIL_TH];
  bool need = false;
#pragma unroll
  for (int r = 0; r < SIL_TH; ++r) {
    prod[r] = 1.f;
    nsat[r] = 0;
    g[r] = 0.f;
    const int row = row0 + r;
    if (!LOSS && row < a.S && col < a.S) g[r] = galpha[(size_t)row * a.S + col];
    need |= LOSS || g[r] != 0.f;
  }
  float lsum = 0.f;
  if (!__any_sync(0xffffffffu, need)) return lsum;
  // pass 1: per pixel, the product of the unsaturated (1 - D_f) and the number of saturated faces
  for (int c0 = 0; c0 < n; c0 += 32) {
    const bool hit = c0 + lane < n && tile_hit(P, L, c0 + lane, x0, x1, y0, y1, pad);
    unsigned m = __ballot_sync(0xffffffffu, hit);
    while (m) {
      const int k = c0 + __ffs(m) - 1;
      m &= m - 1;
      Face F;
      face_setup(F, P, L, k);
#pragma unroll
      for (int r = 0; r < SIL_TH; ++r) {
        float D, om, sgn, t, qx, qy;
        int ke;
        if (soft_term(F, a, px, row0 + r + 0.5f, D, om, sgn, ke, t, qx, qy)) {
          if (om < SIL_SAT) ++nsat[r]; else prod[r] *= om;
        }
      }
    }
  }
  if (LOSS) {
    need = false;
#pragma unroll
    for (int r = 0; r < SIL_TH; ++r) {
      const int row = row0 + r;
      if (row < a.S && col < a.S) {
        const float alpha = nsat[r] ? 1.f : 1.f - prod[r];
        const float d = alpha - (target[(size_t)row * a.S + col] ? 1.f : 0.f);
        lsum += d * d;
        g[r] = gscale * d;
        need |= g[r] != 0.f;
      }
    }
    if (!__any_sync(0xffffffffu, need)) return lsum;
  }
  // pass 2: d loss / d(u, v) of the three vertices of every face, reduced over the warp
  for (int c0 = 0; c0 < n; c0 += 32) {
    const bool hit = c0 + lane < n && tile_hit(P, L, c0 + lane, x0, x1, y0, y1, pad);
    unsigned m = __ballot_sync(0xffffffffu, hit);
    while (m) {
      const int k = c0 + __ffs(m) - 1;
      m &= m - 1;
      Face F;
      face_setup(F, P, L, k);
      float gax = 0.f, gay = 0.f, gbx = 0.f, gby = 0.f, gcx = 0.f, gcy = 0.f;
#pragma unroll
      for (int r = 0; r < SIL_TH; ++r) {
        if (g[r] == 0.f) continue;
        float D, om, sgn, t, qx, qy;
        int ke;
        if (!soft_term(F, a, px, row0 + r + 0.5f, D, om, sgn, ke, t, qx, qy)) continue;
        // prod_{g != f} (1 - D_g) from the unsaturated product and the saturated count
        const float others = om < SIL_SAT ? (nsat[r] == 1 ? prod[r] : 0.f) : (nsat[r] == 0 ? prod[r] / om : 0.f);
        // alpha = 1 - prod (1 - D): d alpha / d D_f = others;  d D / d d^2 = sgn D (1 - D) / sigma
        const float gd2 = g[r] * others * sgn * D * om * a.inv_sigma;
        // d^2 = |p - (1 - t) S - t E|^2 (t at its optimum or clamped): d/dS = -2 (1 - t) q, d/dE = -2 t q
        const float cx = -2.f * gd2 * qx, cy = -2.f * gd2 * qy;
        const float ws = 1.f - t;
        const float wa = ke == 0 ? ws : (ke == 2 ? t : 0.f);
        const float wb = ke == 0 ? t : (ke == 1 ? ws : 0.f);
        const float wc = ke == 1 ? t : (ke == 2 ? ws : 0.f);
        gax += wa * cx; gay += wa * cy;
        gbx += wb * cx; gby += wb * cy;
        gcx += wc * cx; gcy += wc * cy;
      }
      const bool nz = gax != 0.f || gay != 0.f || gbx != 0.f || gby != 0.f || gcx != 0.f || gcy != 0.f;
      if (!__any_sync(0xffffffffu, nz)) continue;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        gax += __shfl_xor_sync(0xffffffffu, gax, o); gay += __shfl_xor_sync(0xffffffffu, gay, o);
        gbx += __shfl_xor_sync(0xffffffffu, gbx, o); gby += __shfl_xor_sync(0xffffffffu, gby, o);
        gcx += __shfl_xor_sync(0xffffffffu, gcx, o); gcy += __shfl_xor_sync(0xffffffffu, gcy, o);
      }
      if (lane == 0) {
        const int ia = L[3 * k], ib = L[3 * k + 1], ic = L[3 * k + 2];
        atomicAdd(&G[ia].x, gax); atomicAdd(&G[ia].y, gay);
        atomicAdd(&G[ib].x, gbx); atomicAdd(&G[ib].y, gby);
        atomicAdd(&G[ic].x, gcx); atomicAdd(&G[ic].y, gcy);
      }
    }
  }
  return lsum;
}

template <bool LOSS>
__device__ void sil_bwd_body(const SilArgs& a, const float* __restrict__ grad_alpha, const uint8_t* __restrict__ target,
                             float weight, float* __restrict__ loss, float* __restrict__ grad_verts,
                             float* __restrict__ grad_t) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int wcnt[SIL_WARPS];
  __shared__ float red[SIL_WARPS][4];
  float2* P = reinterpret_cast<float2*>(smem);
  float2* G = P + a.V;
  uint16_t* L = reinterpret_cast<uint16_t*>(smem + 2 * (size_t)a.V * sizeof(float2));
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  project_body(a, b, P);
  for (int v = threadIdx.x; v < a.V; v += blockDim.x) G[v] = make_float2(0.f, 0.f);
  __syncthreads();
  const size_t img = (size_t)a.S * a.S;
  const float gscale = 2.f * weight / (float)img;
  const int nbands = (a.S + SIL_BAND - 1) / SIL_BAND, ntc = (a.S + SIL_TW - 1) / SIL_TW;
  float lsum = 0.f;
  for (int band = 0; band < nbands; ++band) {
    const int r0 = band * SIL_BAND;
    const int rows = min(SIL_BAND, a.S - r0);
    const int n = band_list(a, P, L, wcnt, r0 + 0.5f, r0 + rows - 0.5f, a.rad + SIL_SLACK);
    const int ntr = (rows + SIL_TH - 1) / SIL_TH;
    for (int tile = warp; tile < ntr * ntc; tile += SIL_WARPS)
      lsum += tile_bwd<LOSS>(a, P, L, n, r0 + (tile / ntc) * SIL_TH, (tile % ntc) * SIL_TW,
                             LOSS ? nullptr : grad_alpha + b * img, LOSS ? target + b * img : nullptr, gscale, G);
    __syncthreads();
  }
  // flush: chain rule through u = f (x + tx) / Z + c, v = f (y + ty) / Z + c, Z = z + tz
  const float tx = a.cam_t[3 * b], ty = a.cam_t[3 * b + 1], tz = a.cam_t[3 * b + 2];
  const float* X = a.verts + (size_t)b * a.V * 3;
  float* GX = grad_verts + (size_t)b * a.V * 3;
  float gtx = 0.f, gty = 0.f, gtz = 0.f;
  for (int v = threadIdx.x; v < a.V; v += blockDim.x) {
    const float Z = X[3 * v + 2] + tz;
    float gx = 0.f, gy = 0.f, gz = 0.f;
    if (Z > SIL_ZMIN) {
      const float2 g = G[v];
      const float fz = a.f / Z;
      gx = g.x * fz;
      gy = g.y * fz;
      gz = -(g.x * (X[3 * v] + tx) + g.y * (X[3 * v + 1] + ty)) * fz / Z;
    }
    GX[3 * v] = gx; GX[3 * v + 1] = gy; GX[3 * v + 2] = gz;
    gtx += gx; gty += gy; gtz += gz;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    gtx += __shfl_xor_sync(0xffffffffu, gtx, o);
    gty += __shfl_xor_sync(0xffffffffu, gty, o);
    gtz += __shfl_xor_sync(0xffffffffu, gtz, o);
    lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
  }
  if (lane == 0) { red[warp][0] = gtx; red[warp][1] = gty; red[warp][2] = gtz; red[warp][3] = lsum; }
  __syncthreads();
  if (threadIdx.x < 4) {
    float s = 0.f;
    for (int w = 0; w < SIL_WARPS; ++w) s += red[w][threadIdx.x];
    if (threadIdx.x < 3) grad_t[3 * b + threadIdx.x] = s;
    else if (LOSS) loss[b] += weight * s / (float)img;
  }
}

__global__ void __launch_bounds__(SIL_THREADS, 1) sil_bwd(SilArgs a, const float* __restrict__ grad_alpha,
                                                          float* __restrict__ grad_verts, float* __restrict__ grad_t) {
  sil_bwd_body<false>(a, grad_alpha, nullptr, 0.f, nullptr, grad_verts, grad_t);
}

__global__ void __launch_bounds__(SIL_THREADS, 1) sil_loss(SilArgs a, const uint8_t* __restrict__ target, float weight,
                                                           float* __restrict__ loss, float* __restrict__ grad_verts,
                                                           float* __restrict__ grad_t) {
  sil_bwd_body<true>(a, nullptr, target, weight, loss, grad_verts, grad_t);
}

// ---- gradient-free loss ------------------------------------------------------------------------------------------
// loss[b] += weight * mean (alpha - target)^2 without the backward's pass 2 or its accumulator G, so the shared
// memory is that of sil_fwd.  Grid (B, split), cluster (1, split, 1): the CTAs of one cluster share a body's bands
// as sil_fwd's do, and rank 0 adds their partial sums in rank order through distributed shared memory, so the
// result is deterministic for a given split and needs neither global atomics nor a workspace.
__global__ void __launch_bounds__(SIL_THREADS, 1) sil_loss_value(SilArgs a, const uint8_t* __restrict__ target,
                                                                 float weight, float* __restrict__ loss) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int wcnt[SIL_WARPS];
  __shared__ float red[SIL_WARPS];
  __shared__ float part;
  cg::cluster_group cluster = cg::this_cluster();
  float2* P = reinterpret_cast<float2*>(smem);
  uint16_t* L = reinterpret_cast<uint16_t*>(smem + (size_t)a.V * sizeof(float2));
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  project_body(a, b, P);
  __syncthreads();
  const size_t img = (size_t)a.S * a.S;
  const uint8_t* tg = target + b * img;
  const int nbands = (a.S + SIL_BAND - 1) / SIL_BAND, ntc = (a.S + SIL_TW - 1) / SIL_TW;
  float lsum = 0.f;
  for (int band = blockIdx.y; band < nbands; band += gridDim.y) {
    const int r0 = band * SIL_BAND;
    const int rows = min(SIL_BAND, a.S - r0);
    const int n = band_list(a, P, L, wcnt, r0 + 0.5f, r0 + rows - 0.5f, a.rad + SIL_SLACK);
    const int ntr = (rows + SIL_TH - 1) / SIL_TH;
    for (int tile = warp; tile < ntr * ntc; tile += SIL_WARPS)
      lsum += tile_fwd<true>(a, P, L, n, r0 + (tile / ntc) * SIL_TH, (tile % ntc) * SIL_TW, nullptr, tg);
    __syncthreads();                                      // the next band rewrites L
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
  if (lane == 0) red[warp] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < SIL_WARPS; ++w) s += red[w];
    part = s;
  }
  cluster.sync();
  if (cluster.block_rank() == 0 && threadIdx.x == 0) {
    float s = 0.f;
    for (unsigned r = 0; r < cluster.num_blocks(); ++r) s += *cluster.map_shared_rank(&part, r);
    loss[b] += weight * s / (float)img;
  }
  cluster.sync();                                         // every partial stays readable until rank 0 has read it
}

size_t sil_smem(const b200smpl_silhouette_args* p, bool bwd) {
  return (size_t)p->num_verts * sizeof(float2) * (bwd ? 2 : 1) + (size_t)p->num_faces * 3 * sizeof(uint16_t);
}

// argument checks shared by the entry points; fills the kernel arguments
int sil_prepare(const b200smpl_silhouette_args* p, bool bwd, SilArgs& a, size_t& smem) {
  if (!p) return fail(B200SMPL_ERR_INVALID, "silhouette: args is NULL");
  if (p->batch < 1 || p->num_verts < 3 || p->num_verts > 65535 || p->num_faces < 1 || p->img_wh < 1 ||
      p->img_wh > 16384)
    return fail(B200SMPL_ERR_INVALID, "silhouette: need batch >= 1, 3 <= num_verts <= 65535, num_faces >= 1, "
                                      "1 <= img_wh <= 16384");
  if (!(p->focal_length > 0.f) || !std::isfinite(p->focal_length) || !(p->sigma >= 0.f) || !std::isfinite(p->sigma))
    return fail(B200SMPL_ERR_INVALID, "silhouette: need focal_length > 0 and a finite sigma >= 0");
  if (!p->vertices || !p->cam_t || !p->faces) return fail(B200SMPL_ERR_INVALID, "silhouette: NULL input pointer");
  smem = sil_smem(p, bwd);
  int dev = 0, optin = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  B200_CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if (smem + 1024 > (size_t)optin)
    return fail(B200SMPL_ERR_INVALID, "silhouette: mesh too large for the shared-memory rasteriser (" +
                                          std::to_string(smem) + " bytes of shared memory needed)");
  a.V = p->num_verts;
  a.F = p->num_faces;
  a.S = p->img_wh;
  a.f = p->focal_length;
  a.c = 0.5f * (float)p->img_wh;
  a.sigma = p->sigma;
  a.inv_sigma = p->sigma > 0.f ? 1.f / p->sigma : 0.f;
  a.r2 = p->sigma * logf(1.f / SIL_EPS - 1.f);
  a.rad = sqrtf(a.r2);
  a.verts = p->vertices;
  a.cam_t = p->cam_t;
  a.faces = p->faces;
  return 0;
}

}  // namespace
}  // namespace b200smpl

using namespace b200smpl;

extern "C" {

size_t b200smpl_silhouette_workspace_bytes(const b200smpl_silhouette_args* args) {
  (void)args;
  return 0;
}

int b200smpl_silhouette_render(const b200smpl_silhouette_args* args, float* alpha, void* stream) {
  B200_NVTX("b200smpl_silhouette_render");
  SilArgs a;
  size_t smem = 0;
  if (int rc = sil_prepare(args, false, a, smem)) return rc;
  if (!alpha) return fail(B200SMPL_ERR_INVALID, "silhouette_render: alpha is NULL");
  int dev = 0, sms = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  B200_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  // small batches: split a body's bands over several CTAs so that the grid covers the SMs
  const int nbands = (a.S + SIL_BAND - 1) / SIL_BAND;
  const int split = std::max(1, std::min(nbands, (sms + args->batch - 1) / args->batch));
  B200_SMEM_ATTR_ONCE(sil_fwd, smem);
  LaunchTimer _timer("sil_fwd", (cudaStream_t)stream);
  sil_fwd<<<dim3(args->batch, split), SIL_THREADS, smem, (cudaStream_t)stream>>>(a, alpha);
  B200_LAUNCH_CHECK("sil_fwd");
  return 0;
}

int b200smpl_silhouette_render_backward(const b200smpl_silhouette_args* args, const float* grad_alpha,
                                        float* grad_vertices, float* grad_t, void* stream) {
  B200_NVTX("b200smpl_silhouette_render_backward");
  SilArgs a;
  size_t smem = 0;
  if (int rc = sil_prepare(args, true, a, smem)) return rc;
  if (!(args->sigma > 0.f))
    return fail(B200SMPL_ERR_INVALID, "silhouette_render_backward: the hard silhouette (sigma = 0) has no gradient");
  if (!grad_alpha || !grad_vertices || !grad_t)
    return fail(B200SMPL_ERR_INVALID, "silhouette_render_backward: NULL pointer");
  B200_SMEM_ATTR_ONCE(sil_bwd, smem);
  LaunchTimer _timer("sil_bwd", (cudaStream_t)stream);
  sil_bwd<<<args->batch, SIL_THREADS, smem, (cudaStream_t)stream>>>(a, grad_alpha, grad_vertices, grad_t);
  B200_LAUNCH_CHECK("sil_bwd");
  return 0;
}

int b200smpl_silhouette_loss(const b200smpl_silhouette_args* args, const uint8_t* target, float weight,
                             float* loss_per_body, float* grad_vertices, float* grad_t, void* stream) {
  B200_NVTX("b200smpl_silhouette_loss");
  SilArgs a;
  size_t smem = 0;
  if (int rc = sil_prepare(args, true, a, smem)) return rc;
  if (!(args->sigma > 0.f))
    return fail(B200SMPL_ERR_INVALID, "silhouette_loss: the hard silhouette (sigma = 0) has no gradient");
  if (!target || !loss_per_body || !grad_vertices || !grad_t || !std::isfinite(weight))
    return fail(B200SMPL_ERR_INVALID, "silhouette_loss: NULL pointer or non-finite weight");
  B200_SMEM_ATTR_ONCE(sil_loss, smem);
  LaunchTimer _timer("sil_loss", (cudaStream_t)stream);
  sil_loss<<<args->batch, SIL_THREADS, smem, (cudaStream_t)stream>>>(a, target, weight, loss_per_body, grad_vertices,
                                                                     grad_t);
  B200_LAUNCH_CHECK("sil_loss");
  return 0;
}

int b200smpl_silhouette_loss_value(const b200smpl_silhouette_args* args, const uint8_t* target, float weight,
                                   float* loss_per_body, void* stream) {
  B200_NVTX("b200smpl_silhouette_loss_value");
  SilArgs a;
  size_t smem = 0;
  if (int rc = sil_prepare(args, false, a, smem)) return rc;
  if (!target || !loss_per_body || !std::isfinite(weight))
    return fail(B200SMPL_ERR_INVALID, "silhouette_loss_value: NULL pointer or non-finite weight");
  int dev = 0, sms = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  B200_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  // small batches: a cluster of CTAs per body, as many as fill the SMs (sil_fwd's split, capped at a portable cluster)
  const int nbands = (a.S + SIL_BAND - 1) / SIL_BAND;
  const int split = std::max(1, std::min({SIL_MAX_CLUSTER, nbands, (sms + args->batch - 1) / args->batch}));
  B200_SMEM_ATTR_ONCE(sil_loss_value, smem);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(args->batch, split, 1);
  cfg.blockDim = dim3(SIL_THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = split;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  LaunchTimer _timer("sil_loss_value", (cudaStream_t)stream);
  B200_CUDA_TRY(cudaLaunchKernelEx(&cfg, sil_loss_value, a, target, weight, loss_per_body));
  B200_LAUNCH_CHECK("sil_loss_value");
  return 0;
}

}  // extern "C"
