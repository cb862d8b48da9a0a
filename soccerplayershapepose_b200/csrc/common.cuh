// Shared definitions of the B200-native SMPL kernels (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/b200smpl.h"

namespace b200smpl {

constexpr int NJ = 24;             // SMPL chain joints (compile-time)
constexpr int NPOSE = 9 * (NJ - 1);  // 207 pose-corrective features
constexpr int AELEMS = 12;         // per-joint skinning transform, row-major 3x4 [R | t]
constexpr int TILE_V = 32;         // vertices per skinning tile (= output flush granularity)
constexpr int MAX_CHILD = 4;
constexpr int MAX_BETAS = 16;

// vmeta bit layout (one u32 per vertex in processing order)
//  [0:5) j0  [5:10) j1  [10:15) j2  [15:20) j3   slot joint ids
//  [20:24) reload mask (slot s must be (re)loaded before this vertex)
//  [24:29) position of the vertex inside its tile in ORIGINAL order (ol)
//  [29]    valid (vertex index < V)
constexpr uint32_t VMETA_VALID = 1u << 29;

struct ChainTables {
  int8_t parent[NJ];
  int8_t depth[NJ];
  int8_t nchild[NJ];
  int8_t child[NJ][MAX_CHILD];
  int8_t maxchild_at[NJ];   // [d]: max number of children a joint of depth d-1 has (bounds the gather of round d)
  int8_t order[NJ];         // joints sorted by depth (stable): the joints of one level are independent of each other
  int8_t level_ptr[NJ + 1]; // order[level_ptr[d] .. level_ptr[d + 1]) = joints of depth d
  int32_t maxdepth;
};

// K layout of the two forward blend operands (elements; 64-element slabs = one 128-byte swizzle row each).
//   feature row of a body:  [1 1 1 | b_hi b_lo b_hi | 0.. ]  [pf_hi (207) | 0..]  [pf_lo (207) | 0..]
//   model row n:            [t_hi t_lo t_lo2 | S_hi S_hi S_lo | 0..]  [P_hi (207) | 0..]  [P_lo (207) | 0..]
// Slab 0 pairs position by position (template exact 3-way split, shape terms error-compensated).  The pose
// segments are multiplied crosswise by the kernel: pf_hi x P_hi + pf_lo x P_hi ("bf16 mode": bf16 model operand,
// 16-bit features) + pf_hi x P_lo ("fp32 mode": bf16x3 split, ~2^-16 relative, fp32 accumulate) -- each operand
// segment is stored and streamed once and used by two of the three products.
struct FeatLayout {
  int nb;       // betas
  int off_s0, off_s1, off_s2;   // 3, 3+nb, 3+2nb  (inside slab 0)
  int k_cs;     // used extent of slab 0 = 3 + 3 nb
  int pseg;     // elements per pose segment = roundup64(207)
  int off_p0;   // 64: first pose segment  (features: pf_hi, model: P_hi)
  int off_p1;   // 64 + pseg: second       (features: pf_lo, model: P_lo)
  int pitch;    // 64 + 2 pseg (elements; *2 bytes is a multiple of 128)
  int nf;       // nb + 207 gradient features
  int nf_pad;   // roundup16(nf)
};

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

inline FeatLayout make_feat_layout(int nb) {
  FeatLayout L;
  L.nb = nb;
  L.off_s0 = 3;
  L.off_s1 = 3 + nb;
  L.off_s2 = 3 + 2 * nb;
  L.k_cs = 3 + 3 * nb;          // <= 51 for nb <= 16
  L.pseg = round_up(NPOSE, 64);
  L.off_p0 = 64;
  L.off_p1 = 64 + L.pseg;
  L.pitch = 64 + 2 * L.pseg;
  L.nf = nb + NPOSE;
  L.nf_pad = round_up(L.nf, 16);
  return L;
}

// Device-side view of a packed model (all pointers are device pointers).
struct DevModel {
  int V;          // vertices
  int ntiles;     // ceil(V / 32) rounded up to a multiple of 4
  int n_real;     // 3V
  int nq;         // virtual q-groups (3 rows each) appended after the real rows
  int n_rows;     // n_virt0 + 3nq
  int n_virt0;    // first virtual row = ntiles*96 (multiple of 128)
  int n_pad;      // n_rows rounded up to 128
  int njout;      // 24 + nvj + nreg
  int nterms;
  int ntv;        // virtual (joint) tiles of 32 q-groups appended after the vertex tiles
  int vt_maxcols; // max over virtual tiles of 3 * (output joints of the tile)
  FeatLayout fl;
  ChainTables chain;
  const __nv_bfloat16* Wf;     // [n_pad][fl.pitch]         forward operand, K-major
  const __nv_bfloat16* Wb_hi;  // [fl.nf_pad][n_pad]        backward operand (K = n), hi part
  const __nv_bfloat16* Wb_lo;  // [fl.nf_pad][n_pad]        lo part
  const float* W32;            // [1 + nf][n_pad]           fp32 rows: template, shapedirs, posedirs
  const uint32_t* vmeta;       // [ntiles*32]
  const float4* vwts;          // [ntiles*32]
  const uint32_t* vplan;       // [ntiles*4][40]: per 8 vertices, 8 float4 weights then 8 plan words (one 160 B TMA record)
  const float* Jt;             // [24][3]   J_regressor . v_template
  const float* Jsd;            // [24][3][nb]  J_regressor . shapedirs
  const int32_t* term_ptr;     // [njout-24+1]
  const uint8_t* term_joint;   // [nterms] skinning joint of the term
  const int32_t* term_qrow;    // [nterms] first of the 3 blend rows holding q
  const float* term_c;         // [nterms]
  const uint32_t* qmeta;       // [ntv*32] virtual-tile plan (groups sorted by skinning joint): joint | reload<<5 | jl<<8 | valid<<14
  const float* qcoef;          // [ntv*32] homogeneous coefficient c of the q-group
  const int32_t* vt_j0;        // [ntv] first output joint (index into joints 24..) of the tile
  const int32_t* vt_nj;        // [ntv] output joints covered by the tile
};

struct HostArrays {
  std::vector<__nv_bfloat16> Wf, Wb_hi, Wb_lo;
  std::vector<float> W32, Jt, Jsd, term_c;
  std::vector<uint32_t> vmeta;
  std::vector<float> vwts;     // 4 per vertex
  std::vector<uint32_t> vplan; // 40 words per 8 vertices
  std::vector<int32_t> term_ptr, term_qrow, vt_j0, vt_nj;
  std::vector<int8_t> chain_order, chain_level_ptr;   // copies of ChainTables::order / level_ptr (debug / tests)
  std::vector<uint32_t> qmeta;
  std::vector<float> qcoef;
  std::vector<uint8_t> term_joint;
};

}  // namespace b200smpl

struct b200smpl_model {
  int device = -1;
  b200smpl::DevModel dm{};       // device pointers (null for host-only)
  b200smpl::HostArrays host;     // kept for host-only handles / debug queries
  std::vector<void*> allocs;
  int nvj = 0, nreg = 0;
  int num_sms = 148;
};

namespace b200smpl {

// error plumbing ------------------------------------------------------------------------------
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);
void count_launch(int n = 1);

// optional per-launch device timing (bench.py roofline); see b200smpl_timing_enable
// NVTX range over a C-ABI entry point / a kernel launch (SURVEY.md section 5 "Tracing"; no-ops unless a tool such
// as Nsight Systems has injected its NVTX library into the process)
struct NvtxRange {
  explicit NvtxRange(const char* name);
  ~NvtxRange();
};
#define B200_NVTX(name) ::b200smpl::NvtxRange _nvtx_range(name)

struct LaunchTimer {
  LaunchTimer(const char* name, cudaStream_t st);
  ~LaunchTimer();
  const char* name_;
  cudaStream_t st_;
  cudaEvent_t start_ = nullptr;
  NvtxRange nvtx_;
};

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------
// Consecutive kernels of the forward / backward chains are launched with the programmatic-stream-serialization
// attribute: a dependent grid may become resident while its predecessor drains, runs its prologue (barrier init,
// TMEM allocation, descriptor prefetch) and blocks in pdl_wait() until the predecessor grid has completed and
// flushed.  pdl_trigger() in the predecessor marks the point after which dependents may be scheduled.
// B200_PDL=0 disables the attribute (the device instructions are then no-ops).
bool pdl_enabled();
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// kernel<<<grid, block, smem, st>>>(args...) with the PDL attribute when `pdl` (and B200_PDL != 0)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                            Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl && pdl_enabled()) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(std::forward<Args>(args))...);
}
#endif

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) only when the kernel needs more than it has been granted on this
// device so far (the size can depend on the model), instead of on every launch
#define B200_SMEM_ATTR_ONCE(kern, bytes)                                                          \
  do {                                                                                            \
    static int _granted[64] = {};                                                                 \
    int _dev = 0;                                                                                 \
    B200_CUDA_TRY(cudaGetDevice(&_dev));                                                          \
    if (_dev < 0 || _dev >= 64 || (int)(bytes) > _granted[_dev]) {                                \
      B200_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
      if (_dev >= 0 && _dev < 64) _granted[_dev] = (int)(bytes);                                  \
    }                                                                                             \
  } while (0)

#define B200_CUDA_TRY(expr)                                                                       \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return ::b200smpl::fail(B200SMPL_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
  } while (0)

#define B200_LAUNCH_CHECK(name)                                                                   \
  do {                                                                                            \
    cudaError_t _e = cudaGetLastError();                                                          \
    if (_e != cudaSuccess)                                                                        \
      return ::b200smpl::fail(B200SMPL_ERR_CUDA, std::string("launch ") + name + ": " + cudaGetErrorString(_e)); \
    ::b200smpl::count_launch();                                                                   \
  } while (0)

// host pack (pack.cpp)
int pack_model(const b200smpl_model_desc* d, HostArrays& h, DevModel& dm, std::string& err);

// kernel launchers ----------------------------------------------------------------------------
// The batch is processed in slabs of at most S bodies.  Every scratch array is slab-local: its
// body index is the slab column (body - b0) and its body pitch is S.  nb = live bodies of the
// slab, Sw = nb rounded up to 128 (columns in [nb, Sw) are kept zero / finite).
int launch_pose_fwd(const DevModel& m, const float* betas, const float* pose, bool axis_angle, int b0, int nb, int S,
                    int Sw, __nv_bfloat16* feat, float* featf, float* A_blk, const float* transl, float* joints,
                    cudaStream_t st);
int launch_pose_bwd(const DevModel& m, const float* betas, const float* pose, bool axis_angle, int b0, int nb, int S,
                    const float* A_blk, const float* dA_part, int n_dA_parts, const float* dtr_part, const float* dfeat_part,
                    int n_dfeat_parts, const float* dJ, float* grad_betas, float* grad_pose,
                    float* grad_transl, cudaStream_t st);

int launch_blend_fwd_simt(const DevModel& m, const float* featf, int S, int Sw, float* vpT, int row_begin,
                          int row_end, cudaStream_t st);
int launch_blend_bwd_simt(const DevModel& m, const __nv_bfloat16* dvp_hi, const __nv_bfloat16* dvp_lo, int S, int Sw,
                          float* dfeat, int row_begin, int row_end, cudaStream_t st);
int launch_blend_fwd_umma(const DevModel& m, int mode, const __nv_bfloat16* feat, int S, int Sw, float* vpT,
                          int row_begin, int row_end, int num_sms, cudaStream_t st);
int launch_blend_bwd_umma(const DevModel& m, int mode, const __nv_bfloat16* dvp_hi, const __nv_bfloat16* dvp_lo,
                          int S, int Sw, float* dfeat_part, int nsplit, int row_begin, int row_end,
                          cudaStream_t st);
int blend_bwd_umma_splits(const DevModel& m, int S, int num_sms);
// blend GEMM with the skinning in its epilogue (fused_fwd.cu); forward-only calls
int launch_blend_lbs_fwd(const DevModel& m, int mode, const __nv_bfloat16* feat, int S, int Sw, float* vpT,
                         const float* A_blk, int b0, int nb, const float* transl, float* verts, int num_sms,
                         cudaStream_t st);

int launch_lbs_fwd(const DevModel& m, const float* vpT, int S, const float* A_T, int b0, int nb,
                   const float* transl, float* verts, int num_sms, cudaStream_t st);
int launch_lbs_bwd(const DevModel& m, const float* vpT, int S, int Sw, const float* A_T, int b0, int nb,
                   const float* grad_verts, __nv_bfloat16* dvp_hi, __nv_bfloat16* dvp_lo, float* dA_acc,
                   float* dtr_acc, int num_sms, cudaStream_t st);

int launch_joints_fwd(const DevModel& m, const float* vpB, int S, const float* A_blk, int b0, int nb,
                      const float* transl, float* joints, bool after_lbs, cudaStream_t st);
int launch_joints_bwd(const DevModel& m, const float* vpB, int S, int Sw, const float* A_blk, int b0, int nb,
                      const float* dJ, __nv_bfloat16* dvp_hi, __nv_bfloat16* dvp_lo, float* dA_part, float* dtr_part,
                      bool after_lbs, cudaStream_t st);
int launch_joint_grad_total(const float* joints, const float* cam, const float* gj, const float* g2d, float* dJ,
                            float* gcam, int B, int nj, cudaStream_t st);

}  // namespace b200smpl
