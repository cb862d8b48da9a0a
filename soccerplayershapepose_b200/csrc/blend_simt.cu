// Plain fp32 FFMA versions of the two blend-shape contractions (B200SMPL_MODE_FP32_SIMT).
// Verification mode only: exact fp32 arithmetic to triangulate the tcgen05 kernels against the
// oracle.  Not tuned; the tensor-core kernels in blend_umma.cu are the product path.
#include "common.cuh"

namespace b200smpl {

// vpT[n][s] = W32[0][n] + sum_f featf[b0+s][f] * W32[1+f][n]      (smplx.lbs: v_template +
// blend_shapes + pose_offsets, rows a4/a7 of SURVEY.md section 8)
// block (32, 8): tile of 32 bodies x 32 rows; each thread 4 rows.
__global__ void __launch_bounds__(256)
blend_fwd_simt_kernel(const float* __restrict__ W32, int n_pad, int nf, const float* __restrict__ featf,
                      int nf_pad, int S, float* __restrict__ vpT, int row0) {
  __shared__ float sW[32][33];   // [f][n]
  __shared__ float sF[32][33];   // [b][f]
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int n0 = row0 + blockIdx.x * 32;
  const int s0 = blockIdx.y * 32;
  float acc[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i] = W32[n0 + ty * 4 + i];
  for (int f0 = 0; f0 < nf; f0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int f = f0 + ty * 4 + i;
      sW[ty * 4 + i][tx] = f < nf ? W32[(size_t)(1 + f) * n_pad + n0 + tx] : 0.f;
      // sF[b][f]: tx indexes f (contiguous in memory), ty*4+i indexes the body
      const int fb = f0 + tx;
      sF[ty * 4 + i][tx] = fb < nf ? featf[(size_t)(s0 + ty * 4 + i) * nf_pad + fb] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int f = 0; f < 32; ++f) {
      const float x = sF[tx][f];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(x, sW[f][ty * 4 + i], acc[i]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {   // vpB [S/32][n_pad/4][32][4] (skin_common.cuh)
    const size_t n = (size_t)(n0 + ty * 4 + i);
    vpT[(((size_t)(s0 >> 5) * (n_pad >> 2) + (n >> 2)) * 32 + tx) * 4 + (n & 3)] = acc[i];
  }
}

int launch_blend_fwd_simt(const DevModel& m, const float* featf, int S, int Sw, float* vpT, int row_begin,
                          int row_end, cudaStream_t st) {
  if (row_begin >= row_end) return 0;        // joints only, and the model has no virtual joint rows
  dim3 grid((row_end - row_begin) / 32, Sw / 32);
  LaunchTimer _timer_46("blend_fwd_simt", st);
  blend_fwd_simt_kernel<<<grid, dim3(32, 8), 0, st>>>(m.W32, m.n_pad, m.fl.nf, featf, m.fl.nf_pad, S, vpT,
                                                      row_begin);
  B200_LAUNCH_CHECK("blend_fwd_simt");
  return 0;
}

// dfeat[b0+s][f] = sum_{n in [row_begin, row_end)} (hi + lo)[s][n] * W32[1+f][n]
// one block per (8 features, 32 bodies); threads reduce over n with a shared-memory tile.
__global__ void __launch_bounds__(256)
blend_bwd_simt_kernel(const float* __restrict__ W32, int n_pad, int nf, const __nv_bfloat16* __restrict__ dvp_hi,
                      const __nv_bfloat16* __restrict__ dvp_lo, int S, float* __restrict__ dfeat, int nf_pad,
                      int row_begin, int row_end) {
  __shared__ float sD[32][33];   // [s][n]
  __shared__ float sW[8][33];    // [f][n]
  const int tx = threadIdx.x, ty = threadIdx.y;   // tx: body, ty: feature
  const int f = blockIdx.x * 8 + ty;
  const int s0 = blockIdx.y * 32;
  float acc = 0.f;
  for (int n0 = row_begin; n0 < row_end; n0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int s = ty * 4 + i;
      const size_t nn = (size_t)(n0 + tx);   // dvp [S/128][n_pad/8][128][8] (skin_common.cuh)
      const size_t o = (((size_t)(s0 >> 7) * (n_pad >> 3) + (nn >> 3)) * 128 + (s0 & 127) + s) * 8 + (nn & 7);
      float v = 0.f;
      if (n0 + tx < row_end) {
        v = __bfloat162float(dvp_hi[o]);
        if (dvp_lo != nullptr) v += __bfloat162float(dvp_lo[o]);
      }
      sD[s][tx] = v;
    }
    sW[ty][tx] = (f < nf && n0 + tx < row_end) ? W32[(size_t)(1 + f) * n_pad + n0 + tx] : 0.f;
    __syncthreads();
#pragma unroll 8
    for (int n = 0; n < 32; ++n) acc = fmaf(sD[tx][n], sW[ty][n], acc);
    __syncthreads();
  }
  if (f < nf_pad) dfeat[(size_t)(s0 + tx) * nf_pad + f] = (f < nf) ? acc : 0.f;
}

int launch_blend_bwd_simt(const DevModel& m, const __nv_bfloat16* dvp_hi, const __nv_bfloat16* dvp_lo, int S, int Sw,
                          float* dfeat, int row_begin, int row_end, cudaStream_t st) {
  dim3 grid(m.fl.nf_pad / 8, Sw / 32);
  LaunchTimer _timer_88("blend_bwd_simt", st);
  blend_bwd_simt_kernel<<<grid, dim3(32, 8), 0, st>>>(m.W32, m.n_pad, m.fl.nf, dvp_hi, dvp_lo, S, dfeat,
                                                      m.fl.nf_pad, row_begin, row_end);
  B200_LAUNCH_CHECK("blend_bwd_simt");
  return 0;
}

}  // namespace b200smpl
