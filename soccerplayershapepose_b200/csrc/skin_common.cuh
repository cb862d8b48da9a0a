// Helpers shared by the skinning kernels (lbs.cu: real vertex tiles; joints.cu: virtual joint tiles).
//
// Slab-local layouts, all blocked by body group (32 consecutive bodies; lane = body everywhere) so that a
// warp streams through one contiguous block per group:
//   vpB   [S/32][n_pad/4][32][4] fp32   blend output: element (row n, body s) at
//                                ((s >> 5) * (n_pad/4) + (n >> 2)) * 128 + (s & 31) * 4 + (n & 3)
//   dvp   [S/128][n_pad/8][128][8] bf16 gradient-GEMM operand (hi and lo arrays): element (body s, row n) at
//                                ((s >> 7) * (n_pad/8) + (n >> 3)) * 1024 + (s & 127) * 8 + (n & 7) -- 16-byte
//                                chunks = rows of the UMMA no-swizzle K-major core matrices; a K slab of 64 rows
//                                of one 128-body tile is 16 contiguous KB = one bulk copy of the GEMM
//   A_blk [S/32][24][3][32][4]   skinning transforms: one float4 = row r of [R | t] of one body
//   dA    [S/32][24*12][32]      gradient of A, accumulated with fp32 REDs
#pragma once

#include "common.cuh"

namespace b200smpl {

constexpr int AG_WORDS = NJ * AELEMS * 32;       // 9216 floats = 36 KB: one group's skinning transforms

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_addr(bar)), "r"(parity)
        : "memory");
    if (done) break;
    if (++spins > (1u << 26)) __trap();   // a lost completion must fail loudly, not hang the GPU
  }
}
// global -> shared bulk-async copy (TMA unit), completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}

// one thread: initialise the barrier and pull the group's transforms (36 KB, contiguous) into smem
__device__ __forceinline__ void fetch_group_transforms(float* A_s, const float* A_blk, int g, uint64_t* bar) {
  mbar_init(bar, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  mbar_expect_tx(bar, AG_WORDS * 4);
  bulk_g2s(A_s, A_blk + (size_t)g * AG_WORDS, AG_WORDS * 4, bar);
}

// streaming global accesses: read-once inputs bypass L1, written-once outputs are not kept hot
__device__ __forceinline__ float ld_stream(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_stream4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream(float* p, float v) {
  asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void st_stream2(float* p, float2 v) {
  asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream_u4(void* p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
// fire-and-forget fp32 add into global memory (resolved in L2)
__device__ __forceinline__ void red_add(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// ---- packed fp32 pairs (Blackwell FFMA2 / FMUL2 / FADD2: two fp32 lanes per instruction) -------------------
typedef unsigned long long f2;
__device__ __forceinline__ f2 mk2(float lo, float hi) {
  f2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ float lo2(f2 v) {
  float lo;
  [[maybe_unused]] float hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
  return lo;
}
__device__ __forceinline__ float hi2(f2 v) {
  [[maybe_unused]] float lo;
  float hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
  return hi;
}
__device__ __forceinline__ f2 bc2(float x) { return mk2(x, x); }   // ptxas folds this into the scalar-broadcast operand form
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) {
  f2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f2 mul2(f2 a, f2 b) {
  f2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f2 add2(f2 a, f2 b) {
  f2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
template <bool HI>
__device__ __forceinline__ f2 set_half(f2 v, float x) { return HI ? mk2(lo2(v), x) : mk2(x, hi2(v)); }
template <bool HI>
__device__ __forceinline__ float get_half(f2 v) { return HI ? hi2(v) : lo2(v); }

// ---- transforms: [joint][3][lane] float4 = (r00 r10 r01 r11) (r02 r12 t0 t1) (r20 r21 r22 t2) of that lane's body
// (the same indexing serves the shared-memory copy of one group and the global A_blk + group offset)
__device__ __forceinline__ void unpack_transform(float (&a)[AELEMS], const float4& q0, const float4& q1, const float4& q2) {
  a[0] = q0.x; a[4] = q0.y; a[1] = q0.z; a[5] = q0.w;
  a[2] = q1.x; a[6] = q1.y; a[3] = q1.z; a[7] = q1.w;
  a[8] = q2.x; a[9] = q2.y; a[10] = q2.z; a[11] = q2.w;
}
// add a slot's gradient accumulators into the group's dA rows [joint * 12 + e][32] and clear them
__device__ __forceinline__ void flush_slot_g(float (&d)[AELEMS], float* dA_g, int joint, int lane) {
  float* p = dA_g + (size_t)joint * AELEMS * 32 + lane;
#pragma unroll
  for (int e = 0; e < AELEMS; ++e) {
    red_add(p + e * 32, d[e]);
    d[e] = 0.f;
  }
}

// (x0, x1) -> packed bf16 hi pair and bf16 lo pair (x ~ hi + lo to 16 mantissa bits); low half = x0
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
  const float r0 = x0 - __uint_as_float(hi << 16);
  const float r1 = x1 - __uint_as_float(hi & 0xFFFF0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r1), "f"(r0));
}
// eight consecutive gradient rows of one body -> one 16-byte chunk of dvp_hi (and dvp_lo)
__device__ __forceinline__ void store_dvp_chunk(const float (&q)[8], __nv_bfloat16* hi_p, __nv_bfloat16* lo_p) {
  uint4 h, l;
  split2(q[0], q[1], h.x, l.x);
  split2(q[2], q[3], h.y, l.y);
  split2(q[4], q[5], h.z, l.z);
  split2(q[6], q[7], h.w, l.w);
  st_stream_u4(hi_p, h);
  if (lo_p != nullptr) st_stream_u4(lo_p, l);
}

}  // namespace b200smpl
