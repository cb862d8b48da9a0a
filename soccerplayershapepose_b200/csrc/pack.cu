// Host-side model packing (runs once per model, on the CPU, in b200smpl_model_create).
//
// Input: the buffers smplx.SMPL.__init__ registers + the three extra regressors of
// models/smpl_official.py:17-25.  Output (see common.cuh):
//   * the blend operand W: one row per output coordinate (3 per vertex) plus 3 rows per "virtual
//     q-group" (joints), each row = [template | shapedirs | posedirs] coefficients, stored as the
//     bf16x3 split along K for the forward GEMM, transposed hi/lo for the backward GEMM, and as
//     plain fp32 for the SIMT verification mode;
//   * the 4-sparse skinning plan (per 32-vertex tile: processing order, 4 joint slots, reload mask);
//   * joint terms: every non-chain output joint as a short list of (skin joint, q rows, coefficient);
//   * J_template / J_shapedirs (rest joints as an affine function of betas) and the chain tables.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include <map>
#include <numeric>

#include "common.cuh"

namespace b200smpl {

static inline __nv_bfloat16 h_bf16(float x) { return __float2bfloat16_rn(x); }
static inline float h_f32(__nv_bfloat16 x) { return __bfloat162float(x); }

int pack_model(const b200smpl_model_desc* d, HostArrays& h, DevModel& dm, std::string& err) {
  const int V = d->num_verts, nb = d->num_betas, nvj = d->num_vertex_joints, nreg = d->num_regressed_joints;
  if (d->num_joints != NJ) { err = "num_joints must be 24"; return B200SMPL_ERR_INVALID; }
  if (V < 1 || V > (1 << 20)) { err = "bad num_verts"; return B200SMPL_ERR_INVALID; }
  if (nb < 1 || nb > MAX_BETAS) { err = "num_betas must be in [1,16]"; return B200SMPL_ERR_INVALID; }
  if (!d->v_template || !d->shapedirs || !d->posedirs || !d->J_regressor || !d->lbs_weights || !d->parents ||
      (nvj > 0 && !d->vertex_joint_ids) || (nreg > 0 && !d->joint_regressors)) {
    err = "null model array";
    return B200SMPL_ERR_INVALID;
  }
  const FeatLayout fl = make_feat_layout(nb);
  const int nf = fl.nf;

  // ---- chain tables (kinematic tree must be parent-before-child; bit-exact integer work) ----
  ChainTables ch;
  memset(&ch, 0, sizeof(ch));
  ch.maxdepth = 0;
  for (int j = 0; j < NJ; ++j) {
    const long long p = d->parents[j];
    if ((j == 0 && p != -1) || (j > 0 && (p < 0 || p >= j))) { err = "parents must satisfy parents[0]=-1, 0<=parents[i]<i"; return B200SMPL_ERR_INVALID; }
    ch.parent[j] = (int8_t)p;
    ch.depth[j] = j == 0 ? 0 : (int8_t)(ch.depth[p] + 1);
    ch.maxdepth = std::max<int>(ch.maxdepth, ch.depth[j]);
    for (int k = 0; k < MAX_CHILD; ++k) ch.child[j][k] = -1;
  }
  for (int j = 1; j < NJ; ++j) {
    const int p = ch.parent[j];
    if (ch.nchild[p] >= MAX_CHILD) { err = "a joint has more than 4 children"; return B200SMPL_ERR_INVALID; }
    ch.child[p][ch.nchild[p]++] = (int8_t)j;
  }
  for (int j = 0; j < NJ; ++j)
    if (ch.depth[j] + 1 < NJ) ch.maxchild_at[ch.depth[j] + 1] = std::max(ch.maxchild_at[ch.depth[j] + 1], ch.nchild[j]);

  {  // joints by level (the lane = body pose kernels walk the tree one level at a time, one warp per joint of the level)
    int n = 0;
    for (int dpt = 0; dpt <= ch.maxdepth; ++dpt) {
      ch.level_ptr[dpt] = (int8_t)n;
      for (int j = 0; j < NJ; ++j)
        if (ch.depth[j] == dpt) ch.order[n++] = (int8_t)j;
    }
    for (int dpt = ch.maxdepth + 1; dpt <= NJ; ++dpt) ch.level_ptr[dpt] = (int8_t)n;
  }

  // ---- skinning influences per vertex (<= 4 non-zeros) ----
  struct Infl { int n; int j[4]; float w[4]; };
  std::vector<Infl> infl(V);
  for (int v = 0; v < V; ++v) {
    Infl I{};
    for (int j = 0; j < NJ; ++j) {
      const float w = d->lbs_weights[(size_t)v * NJ + j];
      if (w != 0.f) {
        if (I.n == 4) { err = "lbs_weights row " + std::to_string(v) + " has more than 4 non-zeros"; return B200SMPL_ERR_INVALID; }
        I.j[I.n] = j;
        I.w[I.n] = w;
        ++I.n;
      }
    }
    infl[v] = I;
  }

  // ---- virtual q-groups: picked joints (copy of a vertex) and regressed joints ----
  // group g -> rows n_virt0 + 3g + k ; coefficient vector over [template | nf features] per row
  const int ntiles = round_up((V + TILE_V - 1) / TILE_V, 4);
  const int n_virt0 = ntiles * TILE_V * 3;
  struct Term { int joint; int group; float c; };
  std::vector<std::vector<Term>> joint_terms(nvj + nreg);
  // each group: sparse list of (vertex, coefficient) -> row = sum coef * Wrow(vertex)
  std::vector<std::vector<std::pair<int, double>>> group_src;
  for (int s = 0; s < nvj; ++s) {
    // a picked joint is a regressor row with a single unit entry: one q-group per influence,
    // q = w_vi * p_v, c = w_vi
    const long long v = d->vertex_joint_ids[s];
    if (v < 0 || v >= V) { err = "vertex_joint_ids out of range"; return B200SMPL_ERR_INVALID; }
    for (int i = 0; i < infl[v].n; ++i) {
      const int g = (int)group_src.size();
      group_src.push_back({{(int)v, (double)infl[v].w[i]}});
      joint_terms[s].push_back({infl[v].j[i], g, infl[v].w[i]});
    }
  }
  for (int r = 0; r < nreg; ++r) {
    const float* row = d->joint_regressors + (size_t)r * V;
    std::map<int, int> group_of_joint;   // skin joint -> group index (ordered by joint id)
    std::map<int, double> csum;
    for (int v = 0; v < V; ++v) {
      if (row[v] == 0.f) continue;
      for (int i = 0; i < infl[v].n; ++i) {
        const int j = infl[v].j[i];
        if (!group_of_joint.count(j)) {
          group_of_joint[j] = (int)group_src.size();
          group_src.emplace_back();
        }
        const double coef = (double)row[v] * (double)infl[v].w[i];
        group_src[group_of_joint[j]].push_back({v, coef});
        csum[j] += coef;
      }
    }
    for (auto& kv : group_of_joint) joint_terms[nvj + r].push_back({kv.first, kv.second, (float)csum[kv.first]});
  }
  // ---- lay the q-groups out in 32-group "virtual tiles" (96 blend rows each): the groups of one
  // output joint are consecutive and never straddle a tile (dummy groups pad the gap), so a warp
  // that owns a tile can finish whole joints.
  for (int J = 0; J < nvj + nreg; ++J)
    if (joint_terms[J].empty()) {                          // all-zero regressor row: one null term keeps the
      joint_terms[J].push_back({0, (int)group_src.size(), 0.f});   // joint on the common path (value = transl)
      group_src.emplace_back();
    }
  std::vector<int> group_slot(group_src.size(), -1);     // group -> slot (position) in the padded layout
  std::vector<uint32_t> qmeta;                            // per slot: joint | reload<<5 | jl<<8 | valid<<14
  std::vector<float> qcoef;
  std::vector<int32_t> vt_j0, vt_nj;
  {
    // a tile = up to 32 q-groups covering whole, consecutive output joints; inside the tile the groups are
    // ordered by SKINNING joint, so that the kernels keep one transform (and, backward, one gradient
    // accumulator) in registers across all the output joints of the tile that share it
    struct Entry { int joint, jl, group; float c; };
    std::vector<Entry> cur;
    int cur_j0 = -1, cur_nj = 0;
    auto flush_tile = [&]() {
      if (cur_j0 < 0) return;
      std::stable_sort(cur.begin(), cur.end(), [](const Entry& a, const Entry& b) {
        return a.joint != b.joint ? a.joint < b.joint : a.jl < b.jl;
      });
      int prev_joint = -1;
      for (const Entry& e : cur) {
        const uint32_t mword = (uint32_t)e.joint | ((e.joint != prev_joint ? 1u : 0u) << 5) | ((uint32_t)e.jl << 8) |
                               (1u << 14);
        prev_joint = e.joint;
        group_slot[e.group] = (int)qmeta.size();
        qmeta.push_back(mword);
        qcoef.push_back(e.c);
      }
      while (qmeta.size() % 32) { qmeta.push_back(0u); qcoef.push_back(0.f); }
      vt_j0.push_back(cur_j0);
      vt_nj.push_back(cur_nj);
      cur.clear();
      cur_j0 = -1;
      cur_nj = 0;
    };
    for (int J = 0; J < nvj + nreg; ++J) {
      auto& tv = joint_terms[J];
      const int k = (int)tv.size();
      if (k == 0) continue;
      if (k > 32) { err = "a joint depends on more than 32 skinning joints"; return B200SMPL_ERR_INVALID; }
      if (cur_j0 >= 0 && ((int)cur.size() + k > 32 || J - cur_j0 >= 32)) flush_tile();
      if (cur_j0 < 0) cur_j0 = J;
      const int jl = J - cur_j0;                          // joints of a tile are consecutive (gaps stay at transl)
      for (int t = 0; t < k; ++t) cur.push_back({tv[t].joint, jl, tv[t].group, tv[t].c});
      cur_nj = jl + 1;
    }
    flush_tile();
  }
  const int ntv = (int)qmeta.size() / 32;
  // re-index groups by slot: slot s owns blend rows n_virt0 + 3 s + k
  {
    std::vector<std::vector<std::pair<int, double>>> by_slot(qmeta.size());
    for (size_t gi = 0; gi < group_src.size(); ++gi)
      if (group_slot[gi] >= 0) by_slot[group_slot[gi]] = group_src[gi];
    for (auto& jt : joint_terms)
      for (auto& tm : jt) tm.group = group_slot[tm.group];
    group_src.swap(by_slot);
  }
  const int nq = (int)group_src.size();                   // = 32 * ntv slots (dummy slots have zero rows)
  const int n_rows = n_virt0 + 3 * nq;
  const int n_pad = round_up(std::max(n_rows, 1), 384);   // whole 128-row GEMM tiles and whole 96-row chunks

  // ---- fp32 rows W32[1+nf][n_pad]: row 0 template, 1..nb shapedirs, nb+1.. posedirs ----
  h.W32.assign((size_t)(1 + nf) * n_pad, 0.f);
  for (int v = 0; v < V; ++v)
    for (int k = 0; k < 3; ++k) {
      const size_t n = (size_t)v * 3 + k;
      h.W32[n] = d->v_template[n];
      for (int l = 0; l < nb; ++l) h.W32[(size_t)(1 + l) * n_pad + n] = d->shapedirs[n * nb + l];
      for (int p = 0; p < NPOSE; ++p) h.W32[(size_t)(1 + nb + p) * n_pad + n] = d->posedirs[(size_t)p * V * 3 + n];
    }
  {
    std::vector<double> acc(1 + nf);
    for (int g = 0; g < nq; ++g)
      for (int k = 0; k < 3; ++k) {
        std::fill(acc.begin(), acc.end(), 0.0);
        for (auto& sc : group_src[g]) {
          const size_t n = (size_t)sc.first * 3 + k;
          for (int f = 0; f <= nf; ++f) acc[f] += sc.second * (double)h.W32[(size_t)f * n_pad + n];
        }
        const size_t nr = (size_t)n_virt0 + 3 * g + k;
        for (int f = 0; f <= nf; ++f) h.W32[(size_t)f * n_pad + nr] = (float)acc[f];
      }
  }

  // ---- bf16 split operands ----
  h.Wf.assign((size_t)n_pad * fl.pitch, h_bf16(0.f));
  h.Wb_hi.assign((size_t)fl.nf_pad * n_pad, h_bf16(0.f));
  h.Wb_lo.assign((size_t)fl.nf_pad * n_pad, h_bf16(0.f));
  for (int n = 0; n < n_rows; ++n) {
    __nv_bfloat16* wr = h.Wf.data() + (size_t)n * fl.pitch;
    {  // template: exact 3-way split against the constant features [1,1,1]
      const float t = h.W32[n];
      const __nv_bfloat16 t0 = h_bf16(t);
      const __nv_bfloat16 t1 = h_bf16(t - h_f32(t0));
      const __nv_bfloat16 t2 = h_bf16(t - h_f32(t0) - h_f32(t1));
      wr[0] = t0; wr[1] = t1; wr[2] = t2;
    }
    for (int f = 0; f < nf; ++f) {
      const float x = h.W32[(size_t)(1 + f) * n_pad + n];
      const __nv_bfloat16 hi = h_bf16(x), lo = h_bf16(x - h_f32(hi));
      if (f < nb) {   // features: [b_hi | b_lo | b_hi]  x  rows: [S_hi | S_hi | S_lo]
        wr[fl.off_s0 + f] = hi; wr[fl.off_s1 + f] = hi; wr[fl.off_s2 + f] = lo;
      } else {        // pose segments [P_hi | P_lo]; the kernel forms pf_hi.P_hi + pf_lo.P_hi + pf_hi.P_lo
        const int p = f - nb;
        wr[fl.off_p0 + p] = hi; wr[fl.off_p1 + p] = lo;
      }
      h.Wb_hi[(size_t)f * n_pad + n] = hi;
      h.Wb_lo[(size_t)f * n_pad + n] = lo;
    }
  }

  // ---- rest joints as an affine function of betas (fp64 fold of J_regressor) ----
  h.Jt.assign(NJ * 3, 0.f);
  h.Jsd.assign((size_t)NJ * 3 * nb, 0.f);
  for (int j = 0; j < NJ; ++j) {
    std::vector<double> acc(3 * (1 + nb), 0.0);
    for (int v = 0; v < V; ++v) {
      const double r = d->J_regressor[(size_t)j * V + v];
      if (r == 0.0) continue;
      for (int k = 0; k < 3; ++k) {
        acc[k * (1 + nb)] += r * (double)d->v_template[v * 3 + k];
        for (int l = 0; l < nb; ++l) acc[k * (1 + nb) + 1 + l] += r * (double)d->shapedirs[((size_t)v * 3 + k) * nb + l];
      }
    }
    for (int k = 0; k < 3; ++k) {
      h.Jt[j * 3 + k] = (float)acc[k * (1 + nb)];
      for (int l = 0; l < nb; ++l) h.Jsd[((size_t)j * 3 + k) * nb + l] = (float)acc[k * (1 + nb) + 1 + l];
    }
  }

  // ---- skinning plan: vertices in their original order; four joint "slots" persist along the whole
  // vertex sequence (a warp walks a contiguous run of tiles and forces a reload of all four slots at
  // its first vertex), so a slot is (re)loaded only where a vertex needs a joint that is not resident
  h.vmeta.assign((size_t)ntiles * TILE_V, 0u);
  h.vwts.assign((size_t)ntiles * TILE_V * 4, 0.f);
  {
    int slot_joint[4] = {0, 0, 0, 0};
    for (int v = 0; v < ntiles * TILE_V; ++v) {
      uint32_t meta = 0;
      float w4[4] = {0.f, 0.f, 0.f, 0.f};
      uint32_t reload = 0;
      if (v < V) {
        const Infl& I = infl[v];
        bool placed[4] = {false, false, false, false};
        bool slot_used[4] = {false, false, false, false};
        for (int a = 0; a < I.n; ++a)            // joints already resident keep their slot
          for (int s = 0; s < 4; ++s)
            if (!slot_used[s] && !placed[a] && slot_joint[s] == I.j[a]) {
              placed[a] = true; slot_used[s] = true; w4[s] = I.w[a];
            }
        for (int a = 0; a < I.n; ++a) {
          if (placed[a]) continue;
          // evict the resident joint whose next use is farthest away
          int pick = -1, pick_dist = -1;
          for (int s = 0; s < 4; ++s) {
            if (slot_used[s]) continue;
            int dist = 1 << 30;
            for (int u = v + 1; u < V && u < v + 256; ++u) {
              bool uses = false;
              for (int b = 0; b < infl[u].n; ++b) uses |= (infl[u].j[b] == slot_joint[s]);
              if (uses) { dist = u - v; break; }
            }
            if (dist > pick_dist) { pick_dist = dist; pick = s; }
          }
          slot_used[pick] = true; placed[a] = true;
          slot_joint[pick] = I.j[a]; w4[pick] = I.w[a]; reload |= 1u << pick;
        }
        meta |= VMETA_VALID;
      }
      for (int s = 0; s < 4; ++s) meta |= (uint32_t)slot_joint[s] << (5 * s);
      meta |= reload << 20;
      meta |= (uint32_t)(v % TILE_V) << 24;
      h.vmeta[v] = meta;
      for (int s = 0; s < 4; ++s) h.vwts[(size_t)v * 4 + s] = w4[s];
    }
  }

  // the same plan as 160-byte records of 8 vertices (8 float4 weights, then 8 plan words): what the skinning
  // kernels pull with one bulk copy per item
  h.vplan.assign((size_t)ntiles * (TILE_V / 8) * 40, 0u);
  for (int v = 0; v < ntiles * TILE_V; ++v) {
    uint32_t* rec = h.vplan.data() + (size_t)(v / 8) * 40;
    memcpy(rec + (v % 8) * 4, &h.vwts[(size_t)v * 4], 16);
    rec[32 + v % 8] = h.vmeta[v];
  }

  // ---- joint terms, flattened ----
  h.term_ptr.assign(nvj + nreg + 1, 0);
  h.term_joint.clear(); h.term_qrow.clear(); h.term_c.clear();
  for (int J = 0; J < nvj + nreg; ++J) {
    // terms sharing a q-group must be consecutive (joints_bwd relies on it): sort by group
    std::stable_sort(joint_terms[J].begin(), joint_terms[J].end(),
                     [](const Term& a, const Term& b) { return a.group < b.group; });
    for (auto& tm : joint_terms[J]) {
      h.term_joint.push_back((uint8_t)tm.joint);
      h.term_qrow.push_back(n_virt0 + 3 * tm.group);
      h.term_c.push_back(tm.c);
    }
    h.term_ptr[J + 1] = (int32_t)h.term_joint.size();
  }
  if (h.term_joint.empty()) { h.term_joint.push_back(0); h.term_qrow.push_back(0); h.term_c.push_back(0.f); }

  memset(&dm, 0, sizeof(dm));
  h.qmeta = qmeta; h.qcoef = qcoef; h.vt_j0 = vt_j0; h.vt_nj = vt_nj;
  dm.ntv = ntv;
  dm.vt_maxcols = 3;
  for (int x : vt_nj) dm.vt_maxcols = std::max(dm.vt_maxcols, 3 * x);
  dm.V = V; dm.ntiles = ntiles; dm.n_real = 3 * V; dm.nq = nq; dm.n_virt0 = n_virt0; dm.n_rows = n_rows;
  dm.n_pad = n_pad; dm.njout = NJ + nvj + nreg; dm.nterms = h.term_ptr.back();
  dm.fl = fl; dm.chain = ch;
  h.chain_order.assign(ch.order, ch.order + NJ);
  h.chain_level_ptr.assign(ch.level_ptr, ch.level_ptr + NJ + 1);
  return 0;
}

}  // namespace b200smpl
