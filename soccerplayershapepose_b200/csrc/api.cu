// C-ABI entry points (include/b200smpl.h): model lifetime, workspace planning, and the slab
// pipelines that chain the kernels for forward and backward.
#include <atomic>
#include <cstring>
#include <map>
#include <mutex>

#include <nvtx3/nvToolsExt.h>

#include "common.cuh"
#include "umma_common.cuh"

namespace b200smpl {

bool pdl_enabled() {
  static const bool on = getenv("B200_PDL") == nullptr || atoi(getenv("B200_PDL")) != 0;
  return on;
}

NvtxRange::NvtxRange(const char* name) { nvtxRangePushA(name); }
NvtxRange::~NvtxRange() { nvtxRangePop(); }

static thread_local std::string g_last_error;
static std::atomic<long long> g_launches{0};

void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- per-launch timing ------------------------------------------------------------------------
static std::atomic<int> g_timing{0};
static std::mutex g_timing_mu;
struct TimingRec { const char* name; cudaEvent_t a, b; };
static std::vector<TimingRec> g_timing_recs;

LaunchTimer::LaunchTimer(const char* name, cudaStream_t st) : name_(name), st_(st), nvtx_(name) {
  if (g_timing.load(std::memory_order_relaxed)) {
    if (cudaEventCreate(&start_) == cudaSuccess) cudaEventRecord(start_, st_);
    else start_ = nullptr;
  }
}
LaunchTimer::~LaunchTimer() {
  if (start_ == nullptr) return;
  cudaEvent_t stop = nullptr;
  if (cudaEventCreate(&stop) != cudaSuccess) return;
  cudaEventRecord(stop, st_);
  std::lock_guard<std::mutex> lk(g_timing_mu);
  g_timing_recs.push_back({name_, start_, stop});
}

// The public modes name the precision of the FORWARD blend GEMM.  The gradient GEMM of the bf16-GEMM mode runs the
// bf16x3 split like the fp32 mode: with single bf16 products grad_betas is 2.2e-3 relative off the fp64 oracle
// (BASELINE.json north_star: 1e-4), with the split it is 2e-5 for +9 % step time.  The single-product backward stays
// available as B200SMPL_MODE_BF16_FAST.
static int fwd_gemm_mode(int mode) { return mode == B200SMPL_MODE_BF16_FAST ? B200SMPL_MODE_BF16 : mode; }
static int bwd_gemm_mode(int mode) {
  return mode == B200SMPL_MODE_BF16 ? B200SMPL_MODE_FP32 : (mode == B200SMPL_MODE_BF16_FAST ? B200SMPL_MODE_BF16 : mode);
}

constexpr int DEFAULT_SLAB = 4096;   // bodies per pass (vpT slab = n_pad * S * 4 B)
// widest slab: the forward GEMMs' work lists hold BS_MAX_WORK pairs of 128-body tiles.  Wider requests are cut to it;
// results do not depend on the slab width.
constexpr int MAX_SLAB = 40960;
static_assert(MAX_SLAB == 2 * BM * BS_MAX_WORK, "slab cap = the forward GEMMs' work-list capacity");
// fewest 64-row K slabs one split of a row-range gradient GEMM (joints only / vertices only) may get.  Fitting
// iteration at 1024 players: 74.3 us with 8, 71.3 with 4, 73.6 with 2
constexpr int MIN_SLABS_PER_SPLIT = 4;

struct Plan {
  int S;                 // slab pitch (multiple of 128)
  int k_splits;          // split-K partials of the backward GEMM
  size_t off_feat, off_featf, off_A, off_jposed, off_vpT;
  size_t off_dvp_hi, off_dvp_lo, off_dA, off_dtr, off_dJtot, off_dfeat;
  size_t total;
  size_t saved_slab_bytes;   // per slab: A_blk [S/32][24][3][32][4] then vpB [S/32][n_pad/4][32][4]
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static Plan make_plan(const b200smpl_model* m, int batch, int mode, int slab_bodies, bool backward) {
  const DevModel& d = m->dm;
  Plan p{};
  const int Bp = round_up(std::max(batch, 1), 128);
  const int S = slab_bodies > 0 ? round_up(std::min(slab_bodies, MAX_SLAB), 128) : DEFAULT_SLAB;
  p.S = std::min(S, Bp);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off = align_up(off + bytes, 1024);
    return o;
  };
  const size_t S_ = (size_t)p.S;
  p.off_feat = take(S_ * d.fl.pitch * 2);
  p.off_featf = take(mode == B200SMPL_MODE_FP32_SIMT ? S_ * d.fl.nf_pad * 4 : 0);
  p.off_A = take((size_t)NJ * AELEMS * S_ * 4);
  p.off_jposed = take((size_t)NJ * 3 * S_ * 4);
  p.off_vpT = take((size_t)d.n_pad * S_ * 4);
  p.saved_slab_bytes = align_up((size_t)NJ * AELEMS * S_ * 4, 1024) + align_up((size_t)d.n_pad * S_ * 4, 1024);
  if (backward) {
    const int bmode = bwd_gemm_mode(mode);
    p.k_splits = bmode == B200SMPL_MODE_FP32_SIMT ? 1 : blend_bwd_umma_splits(d, p.S, m->num_sms);
    p.off_dvp_hi = take(S_ * d.n_pad * 2);
    p.off_dvp_lo = take(bmode == B200SMPL_MODE_BF16 ? 0 : S_ * d.n_pad * 2);
    // dA accumulator [S/32][288][32] directly followed by the dtransl accumulator [S/32][3][32]
    p.off_dA = take((size_t)(NJ * AELEMS + 3) * S_ * 4);
    p.off_dtr = p.off_dA + (size_t)NJ * AELEMS * S_ * 4;
    p.off_dJtot = take((size_t)std::max(batch, 1) * d.njout * 3 * 4);
    p.off_dfeat = take((size_t)p.k_splits * S_ * d.fl.nf_pad * 4);   // split-K partials of the gradient GEMM
  }
  p.total = off + 1024;   // slack for aligning the caller's base pointer
  return p;
}

static int check_common(const b200smpl_model* m, int batch, int mode, const void* ws) {
  if (m == nullptr) return fail(B200SMPL_ERR_INVALID, "null model handle");
  if (m->device < 0) return fail(B200SMPL_ERR_CUDA, "host-only model handle: no CUDA device (there is no CPU fallback)");
  if (batch < 1) return fail(B200SMPL_ERR_INVALID, "batch must be >= 1");
  if (mode != B200SMPL_MODE_FP32 && mode != B200SMPL_MODE_BF16 && mode != B200SMPL_MODE_FP32_SIMT &&
      mode != B200SMPL_MODE_BF16_FAST)
    return fail(B200SMPL_ERR_INVALID, "unknown mode");
  if (ws == nullptr) return fail(B200SMPL_ERR_WORKSPACE, "null workspace");
  return 0;
}

}  // namespace b200smpl

using namespace b200smpl;

extern "C" {

int b200smpl_abi_version(void) { return B200SMPL_ABI_VERSION; }
const char* b200smpl_last_error(void) { return g_last_error.c_str(); }
int64_t b200smpl_launch_count(void) { return (int64_t)g_launches.load(); }

void b200smpl_timing_enable(int enable) { g_timing.store(enable ? 1 : 0); }

size_t b200smpl_timing_report(char* buf, size_t cap) {
  std::vector<TimingRec> recs;
  {
    std::lock_guard<std::mutex> lk(g_timing_mu);
    recs.swap(g_timing_recs);
  }
  std::map<std::string, std::pair<long long, double>> agg;
  for (auto& r : recs) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      auto& e = agg[r.name];
      e.first += 1;
      e.second += ms;
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  std::string out;
  for (auto& kv : agg) out += kv.first + " " + std::to_string(kv.second.first) + " " + std::to_string(kv.second.second) + "\n";
  if (buf != nullptr && cap > 0) {
    const size_t n = std::min(cap - 1, out.size());
    memcpy(buf, out.data(), n);
    buf[n] = 0;
  }
  return out.size() + 1;
}

int b200smpl_model_create(const b200smpl_model_desc* desc, int device, b200smpl_model** out) {
  B200_NVTX("b200smpl_model_create");
  if (desc == nullptr || out == nullptr) return fail(B200SMPL_ERR_INVALID, "null argument");
  *out = nullptr;
  b200smpl_model* m = new b200smpl_model();
  std::string err;
  int rc = pack_model(desc, m->host, m->dm, err);
  if (rc != 0) {
    delete m;
    return fail(rc, err);
  }
  m->nvj = desc->num_vertex_joints;
  m->nreg = desc->num_regressed_joints;
  m->device = device;
  if (device < 0) {
    *out = m;
    return 0;
  }
  auto cleanup = [&]() {
    for (void* p : m->allocs) cudaFree(p);
    delete m;
  };
  int prev = 0;
  cudaError_t e = cudaGetDevice(&prev);
  if (e == cudaSuccess) e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    cleanup();
    return fail(B200SMPL_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
    m->num_sms = prop.multiProcessorCount;
    if (prop.major != 10) {
      cleanup();
      cudaSetDevice(prev);
      return fail(B200SMPL_ERR_CUDA, "this library is built for sm_100a (B200) only; device is sm_" +
                                         std::to_string(prop.major) + std::to_string(prop.minor));
    }
  }
  auto upload = [&](const void* src, size_t bytes, const void** dst) -> bool {
    void* p = nullptr;
    if (cudaMalloc(&p, std::max<size_t>(bytes, 16)) != cudaSuccess) return false;
    m->allocs.push_back(p);
    if (bytes && cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice) != cudaSuccess) return false;
    *dst = p;
    return true;
  };
  HostArrays& h = m->host;
  DevModel& d = m->dm;
  bool ok = true;
#define UP(field, vec) ok = ok && upload((vec).data(), (vec).size() * sizeof((vec)[0]), (const void**)&d.field)
  UP(Wf, h.Wf);
  UP(Wb_hi, h.Wb_hi);
  UP(Wb_lo, h.Wb_lo);
  UP(W32, h.W32);
  UP(vmeta, h.vmeta);
  UP(vwts, h.vwts);
  UP(vplan, h.vplan);
  UP(Jt, h.Jt);
  UP(Jsd, h.Jsd);
  UP(term_ptr, h.term_ptr);
  UP(term_joint, h.term_joint);
  UP(term_qrow, h.term_qrow);
  UP(term_c, h.term_c);
  UP(qmeta, h.qmeta);
  UP(qcoef, h.qcoef);
  UP(vt_j0, h.vt_j0);
  UP(vt_nj, h.vt_nj);
#undef UP
  cudaSetDevice(prev);
  if (!ok) {
    e = cudaGetLastError();
    cleanup();
    return fail(B200SMPL_ERR_CUDA, std::string("model upload failed: ") + cudaGetErrorString(e));
  }
  *out = m;
  return 0;
}

void b200smpl_model_destroy(b200smpl_model* m) {
  if (m == nullptr) return;
  for (void* p : m->allocs) cudaFree(p);
  delete m;
}

int b200smpl_model_get_info(const b200smpl_model* m, b200smpl_model_info* info) {
  if (m == nullptr || info == nullptr) return fail(B200SMPL_ERR_INVALID, "null argument");
  info->num_verts = m->dm.V;
  info->num_joints_out = m->dm.njout;
  info->num_betas = m->dm.fl.nb;
  info->num_blend_rows = m->dm.n_rows;
  info->num_blend_rows_padded = m->dm.n_pad;
  info->feature_pitch = m->dm.fl.pitch;
  info->num_virtual_groups = m->dm.nq;
  info->device = m->device;
  return 0;
}

int b200smpl_model_debug_array(const b200smpl_model* m, const char* name, const void** data, size_t* bytes) {
  if (m == nullptr || name == nullptr || data == nullptr || bytes == nullptr)
    return fail(B200SMPL_ERR_INVALID, "null argument");
  const HostArrays& h = m->host;
  const std::string n(name);
#define RET(key, vec)                          \
  if (n == key) {                              \
    *data = (vec).data();                      \
    *bytes = (vec).size() * sizeof((vec)[0]);  \
    return 0;                                  \
  }
  RET("Wf", h.Wf) RET("Wb_hi", h.Wb_hi) RET("Wb_lo", h.Wb_lo) RET("W32", h.W32) RET("vmeta", h.vmeta)
  RET("vwts", h.vwts) RET("term_ptr", h.term_ptr) RET("term_joint", h.term_joint) RET("term_qrow", h.term_qrow)
  RET("term_c", h.term_c) RET("Jt", h.Jt) RET("Jsd", h.Jsd) RET("qmeta", h.qmeta) RET("qcoef", h.qcoef)
  RET("vt_j0", h.vt_j0) RET("vt_nj", h.vt_nj) RET("chain_order", h.chain_order) RET("chain_level_ptr", h.chain_level_ptr)
#undef RET
  return fail(B200SMPL_ERR_INVALID, "unknown debug array: " + n);
}

size_t b200smpl_saved_bytes(const b200smpl_model* m, int batch, int slab_bodies) {
  if (m == nullptr) return 0;
  const Plan p = make_plan(m, batch, B200SMPL_MODE_FP32, slab_bodies, false);
  const size_t nslabs = ((size_t)std::max(batch, 1) + p.S - 1) / p.S;
  return nslabs * p.saved_slab_bytes + 1024;
}
size_t b200smpl_forward_workspace_bytes(const b200smpl_model* m, int batch, int mode, int slab_bodies) {
  if (m == nullptr) return 0;
  return make_plan(m, batch, mode, slab_bodies, false).total;
}
size_t b200smpl_backward_workspace_bytes(const b200smpl_model* m, int batch, int mode, int slab_bodies) {
  if (m == nullptr) return 0;
  return make_plan(m, batch, mode, slab_bodies, true).total;
}

int b200smpl_forward(const b200smpl_model* m, const b200smpl_forward_args* a, void* stream) {
  B200_NVTX("b200smpl_forward");
  if (a == nullptr) return fail(B200SMPL_ERR_INVALID, "null args");
  int rc = check_common(m, a->batch, a->mode, a->workspace);
  if (rc) return rc;
  if (!a->betas || !a->pose || !a->joints) return fail(B200SMPL_ERR_INVALID, "betas, pose and joints are required");
  if (a->joints2d && !a->cam) return fail(B200SMPL_ERR_INVALID, "joints2d requires cam");
  const Plan p = make_plan(m, a->batch, a->mode, a->slab_bodies, false);
  if (a->workspace_bytes < p.total) return fail(B200SMPL_ERR_WORKSPACE, "forward workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const DevModel& d = m->dm;
  char* ws = (char*)align_up((size_t)a->workspace, 1024);
  __nv_bfloat16* feat = (__nv_bfloat16*)(ws + p.off_feat);
  float* featf = a->mode == B200SMPL_MODE_FP32_SIMT ? (float*)(ws + p.off_featf) : nullptr;
  float* A_T = (float*)(ws + p.off_A);
  float* vpT = (float*)(ws + p.off_vpT);
  const int S = p.S, B = a->batch;
  const bool aa = a->pose_is_axis_angle != 0;
  // joints-only calls blend only the virtual (joint) rows, also when the products are kept for the backward:
  // without a vertices output no grad_vertices can arrive, and b200smpl_backward rejects that combination
  const int row_begin = a->vertices ? 0 : d.n_virt0;
  char* saved = nullptr;
  if (a->saved) {
    if (a->saved_bytes < b200smpl_saved_bytes(m, B, a->slab_bodies)) return fail(B200SMPL_ERR_WORKSPACE, "saved buffer too small");
    saved = (char*)align_up((size_t)a->saved, 1024);
  }
  for (int b0 = 0; b0 < B; b0 += S) {
    const int nb = std::min(S, B - b0);
    const int Sw = round_up(nb, 128);
    if (saved) {
      A_T = (float*)(saved + (size_t)(b0 / S) * p.saved_slab_bytes);
      vpT = (float*)((char*)A_T + align_up((size_t)NJ * AELEMS * S * 4, 1024));
    }
    if ((rc = launch_pose_fwd(d, a->betas, a->pose, aa, b0, nb, S, Sw, feat, featf, A_T, a->transl, a->joints, st)))
      return rc;
    // forward-only calls that want vertices (no products kept for a backward): the blend GEMM skins in its epilogue
    // and v_posed never touches HBM (188 us against 108 + 136 us at B = 4096).  When the products are kept the
    // fused kernel would have to write v_posed AND the vertices (658 MB of pure writes, 242 us): no faster than the
    // two kernels, so that case stays on them.  Below ~512 bodies a call is launch-latency bound and the two kernels
    // (PDL-chained) are as fast or faster (53 vs 47 us at B = 64, 57 vs 65 us at B = 512, 0.211 vs 0.263 ms at
    // B = 4096).
    const bool fused = a->vertices != nullptr && a->mode != B200SMPL_MODE_FP32_SIMT && saved == nullptr && nb >= 512;
    if (fused) {
      rc = launch_blend_lbs_fwd(d, fwd_gemm_mode(a->mode), feat, S, Sw, vpT, A_T, b0, nb, a->transl, a->vertices,
                                m->num_sms, st);
    } else if (a->mode == B200SMPL_MODE_FP32_SIMT) {
      rc = launch_blend_fwd_simt(d, featf, S, Sw, vpT, row_begin, d.n_pad, st);
    } else {
      rc = launch_blend_fwd_umma(d, fwd_gemm_mode(a->mode), feat, S, Sw, vpT, row_begin, d.n_pad, m->num_sms, st);
    }
    if (rc) return rc;
    if (a->vertices && !fused)
      if ((rc = launch_lbs_fwd(d, vpT, S, A_T, b0, nb, a->transl, a->vertices, m->num_sms, st))) return rc;
    // behind the fused kernel the joint kernel reads rows its predecessor writes: plain stream order
    if ((rc = launch_joints_fwd(d, vpT, S, A_T, b0, nb, a->transl, a->joints, a->vertices != nullptr && !fused, st))) return rc;
  }
  if (a->joints2d)   // reprojection of all joints: utils/cam_utils.py:5-26
    if ((rc = b200smpl_orthographic_project(a->joints, a->cam, a->joints2d, B, d.njout, 0.f, stream))) return rc;
  return 0;
}

int b200smpl_backward(const b200smpl_model* m, const b200smpl_backward_args* a, void* stream) {
  B200_NVTX("b200smpl_backward");
  if (a == nullptr) return fail(B200SMPL_ERR_INVALID, "null args");
  int rc = check_common(m, a->batch, a->mode, a->workspace);
  if (rc) return rc;
  if (!a->betas || !a->pose || !a->grad_betas || !a->grad_pose)
    return fail(B200SMPL_ERR_INVALID, "betas, pose, grad_betas and grad_pose are required");
  if (a->grad_joints2d && (!a->cam || !a->joints))
    return fail(B200SMPL_ERR_INVALID, "grad_joints2d requires cam and the forward joints");
  const Plan p = make_plan(m, a->batch, a->mode, a->slab_bodies, true);
  if (a->workspace_bytes < p.total) return fail(B200SMPL_ERR_WORKSPACE, "backward workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const DevModel& d = m->dm;
  const int S = p.S, B = a->batch, nbeta = d.fl.nb;
  const bool aa = a->pose_is_axis_angle != 0;
  const bool have_v = a->grad_vertices != nullptr;
  const bool have_j = a->grad_joints != nullptr || a->grad_joints2d != nullptr;
  if (a->grad_cam && !a->grad_joints2d) B200_CUDA_TRY(cudaMemsetAsync(a->grad_cam, 0, (size_t)B * 3 * 4, st));
  if (!have_v && !have_j) {
    B200_CUDA_TRY(cudaMemsetAsync(a->grad_betas, 0, (size_t)B * nbeta * 4, st));
    B200_CUDA_TRY(cudaMemsetAsync(a->grad_pose, 0, (size_t)B * (aa ? 72 : 216) * 4, st));
    if (a->grad_transl) B200_CUDA_TRY(cudaMemsetAsync(a->grad_transl, 0, (size_t)B * 3 * 4, st));
    return 0;
  }
  char* ws = (char*)align_up((size_t)a->workspace, 1024);
  __nv_bfloat16* feat = (__nv_bfloat16*)(ws + p.off_feat);
  float* featf = a->mode == B200SMPL_MODE_FP32_SIMT ? (float*)(ws + p.off_featf) : nullptr;
  float* A_T = (float*)(ws + p.off_A);
  float* vpT = (float*)(ws + p.off_vpT);
  __nv_bfloat16* dvp_hi = (__nv_bfloat16*)(ws + p.off_dvp_hi);
  const int bmode = bwd_gemm_mode(a->mode);
  __nv_bfloat16* dvp_lo = bmode == B200SMPL_MODE_BF16 ? nullptr : (__nv_bfloat16*)(ws + p.off_dvp_lo);
  float* dA_part = (float*)(ws + p.off_dA);
  float* dtr_part = (float*)(ws + p.off_dtr);
  float* dJtot = (float*)(ws + p.off_dJtot);
  float* dfeat_part = (float*)(ws + p.off_dfeat);
  // total joint gradient: grad_joints itself, or grad_joints + reprojected 2D gradient (also yields dcam)
  const float* dJ = a->grad_joints;
  if (a->grad_joints2d) {
    if ((rc = launch_joint_grad_total(a->joints, a->cam, a->grad_joints, a->grad_joints2d, dJtot, a->grad_cam, B,
                                      d.njout, st)))
      return rc;
    dJ = dJtot;
  }
  const int row_begin = have_v ? 0 : d.n_virt0;
  const int row_end = have_j ? d.n_rows : d.n_virt0;
  int k_splits = 1;
  if (a->mode != B200SMPL_MODE_FP32_SIMT) {
    const int slabs = (row_end + 63) / 64 - row_begin / 64;
    k_splits = std::max(1, std::min(p.k_splits, slabs / MIN_SLABS_PER_SPLIT));
  }
  const char* saved = nullptr;
  if (a->saved) {
    if (a->saved_bytes < b200smpl_saved_bytes(m, B, a->slab_bodies)) return fail(B200SMPL_ERR_WORKSPACE, "saved buffer too small");
    saved = (const char*)align_up((size_t)a->saved, 1024);
  }
  for (int b0 = 0; b0 < B; b0 += S) {
    const int nb = std::min(S, B - b0);
    const int Sw = round_up(nb, 128);
    // the skinning / joint kernels accumulate dL/dA and dL/dtransl of this slab with fp32 REDs
    B200_CUDA_TRY(cudaMemsetAsync(dA_part, 0, (size_t)(NJ * AELEMS + 3) * S * 4, st));
    if (saved) {   // forward kept the transforms and the blend output of this slab: nothing to recompute
      A_T = (float*)(saved + (size_t)(b0 / S) * p.saved_slab_bytes);
      vpT = (float*)((char*)A_T + align_up((size_t)NJ * AELEMS * S * 4, 1024));
    } else {
      if ((rc = launch_pose_fwd(d, a->betas, a->pose, aa, b0, nb, S, Sw, feat, featf, A_T, nullptr, nullptr, st)))
        return rc;
      if (a->mode == B200SMPL_MODE_FP32_SIMT)
        rc = launch_blend_fwd_simt(d, featf, S, Sw, vpT, row_begin, d.n_pad, st);
      else
        rc = launch_blend_fwd_umma(d, fwd_gemm_mode(a->mode), feat, S, Sw, vpT, row_begin, d.n_pad, m->num_sms, st);
      if (rc) return rc;
    }
    {  // the gradient GEMM reads whole 64-row K slabs: rows between row_end and the slab boundary must be finite
      const size_t c0 = (size_t)row_end / 8, c1 = (size_t)round_up(row_end, 64) / 8;
      if (c1 > c0) {   // dvp [S/128][n_pad/8][128][8]: the same chunk range of every 128-body tile
        const size_t pitch = (size_t)(d.n_pad / 8) * 2048, width = (c1 - c0) * 2048;
        B200_CUDA_TRY(cudaMemset2DAsync(dvp_hi + c0 * 1024, pitch, 0, width, (size_t)Sw / 128, st));
        if (dvp_lo) B200_CUDA_TRY(cudaMemset2DAsync(dvp_lo + c0 * 1024, pitch, 0, width, (size_t)Sw / 128, st));
      }
    }
    if (have_v)
      if ((rc = launch_lbs_bwd(d, vpT, S, Sw, A_T, b0, nb, a->grad_vertices, dvp_hi, dvp_lo, dA_part, dtr_part,
                               m->num_sms, st)))
        return rc;
    if (have_j)
      if ((rc = launch_joints_bwd(d, vpT, S, Sw, A_T, b0, nb, dJ, dvp_hi, dvp_lo, dA_part, dtr_part, have_v, st))) return rc;
    if (a->mode == B200SMPL_MODE_FP32_SIMT)
      rc = launch_blend_bwd_simt(d, dvp_hi, dvp_lo, S, Sw, dfeat_part, row_begin, row_end, st);
    else
      rc = launch_blend_bwd_umma(d, bmode, dvp_hi, dvp_lo, S, Sw, dfeat_part, k_splits, row_begin, row_end, st);
    if (rc) return rc;
    if ((rc = launch_pose_bwd(d, a->betas, a->pose, aa, b0, nb, S, A_T, dA_part, 1, dtr_part, dfeat_part, k_splits,
                              have_j ? dJ : nullptr, a->grad_betas, a->grad_pose, a->grad_transl, st)))
      return rc;
  }
  return 0;
}

}  // extern "C"
