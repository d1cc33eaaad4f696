// Forward simulation of trait data down the network (pgbp_simulate): every batch element draws one replicate of
// every node from the model's node-family factors -- the same factors K1 assigns -- in preorder, and writes the tip
// records in the layout pgbp_assign_factors[_device] reads.  Contract: include/pgbp_b200.h.
//
// Host preparation (once per batch and mem_parent table): each internal node gets its depth level (root 0, else 1 +
// the deepest parent) and one descriptor (SimNode); descriptors are sorted by level, and an internal node's row in
// the value scratch is its position in that order.  Tips are leaves: one descriptor per data row, one final pass.
// Device: k_sim_prep (one thread per parameter record: Cholesky factors of the rates and of V, status word),
// k_sim_level (one launch per level, one thread per (element, node); values in SoA scratch [rows * p][ldc], batch
// innermost, so parent reads and node writes are coalesced over elements), k_sim_tips (tiles of 32 elements x R data
// rows staged in shared memory: parent reads coalesced over elements, tipdata written as runs of R * p doubles per
// element, each tip value crossing HBM once).  The scratch is bounded by PGBP_SIM_SCRATCH_BYTES: elements are
// processed in chunks, which changes no value since every draw depends on (seed, replicate, node, trait pair) only.
#include <algorithm>
#include <memory>
#include <vector>

#include "pgbp_factors.cuh"
#include "pgbp_launch.h"
#include "pgbp_philox.h"

using namespace pgbp;

#define PGBP_SIM_SCRATCH_BYTES (4ull << 30)  // bound of the internal-node value scratch of one chunk

namespace pgbp {

// One node: parents in the per-parent arrays [k0, k0 + np).  color = the shared colour of the parent edges (-1: a
// hybrid whose edges differ in colour), t0 = the edge length (one parent) or sum gamma_k^2 t_k (K1's t0).
struct SimNode {
  int32_t v, row;  // preorder index; internal row (internal nodes) or data row (tips)
  int32_t k0, np;
  int32_t color, pad;
  double t0;
};

// Rows of the per-record table prep (SoA [rows][ldp]).  BM: lower Cholesky factor of every rate (column-major),
// mu, lower factor of V, root kind (0 fixed, 1 proper), status word.  OU: gamma2 = sigma2 / (2 alpha), alpha, theta,
// mu, sqrt(v), root kind, status word.
struct SimRows {
  int p, nc, model;
  PGBP_HD int L(int c) const { return c * p * p; }
  PGBP_HD int mu() const { return model == PGBP_MODEL_OU ? 3 : nc * p * p; }
  PGBP_HD int LV() const { return model == PGBP_MODEL_OU ? 4 : mu() + p; }
  PGBP_HD int kind() const { return model == PGBP_MODEL_OU ? 5 : LV() + p * p; }
  PGBP_HD int fail() const { return kind() + 1; }
  PGBP_HD int nrows() const { return fail() + 1; }
};

// upper Cholesky factor U'U = A in place (column-major p x p, upper triangle read; the loop of spd_inverse_logdet),
// 0 or the 1-based failing pivot
PGBP_HD int chol_upper(double* w, int p) {
  for (int k = 0; k < p; k++) {
    const double d = w[k * p + k];
    if (!(d > 0.0)) return k + 1;
    const double r = sqrt(d);
    w[k * p + k] = r;
    for (int c = k + 1; c < p; c++) w[c * p + k] /= r;
    for (int c = k + 1; c < p; c++)
      for (int rr = k + 1; rr <= c; rr++) w[c * p + rr] -= w[rr * p + k] * w[c * p + k];
  }
  return 0;
}

struct SimPrep {
  const double* params;
  double* prep;
  int64_t ldp;
  SimRows sr;
  PGBP_HD void operator()(int64_t ip) const {
    double* o = prep + ip;
    int32_t fail = 0;
    if (sr.model == PGBP_MODEL_OU) {
      const double* s = params + 5 * ip;
      const double sigma2 = s[0], alpha = s[1], theta = s[2], mu = s[3], v = s[4];
      if (!(sigma2 > 0.0) || !(alpha > 0.0)) fail = PGBP_STATUS(0x7ffffd, 1);
      else if (v == INFINITY) fail = PGBP_STATUS(0x7ffff7, 1);
      else if (!(v >= 0.0)) fail = PGBP_STATUS(0x7ffffd, 1);
      o[0] = sigma2 / (2.0 * alpha);
      o[ldp] = alpha;
      o[2 * ldp] = theta;
      o[3 * ldp] = mu;
      o[4 * ldp] = v > 0.0 ? sqrt(v) : 0.0;
      o[5 * ldp] = v > 0.0 ? 1.0 : 0.0;
      o[6 * ldp] = (double)fail;
      return;
    }
    const int p = sr.p, nc = sr.nc, pp = p * p;
    const double* src = params + ip * (int64_t)(nc * pp + p + pp);
    double w[PGBP_MAX_TRAITS * PGBP_MAX_TRAITS];
    for (int c = 0; c < nc; c++) {  // like ThetaPrep: the last failing colour names the pivot
      for (int k = 0; k < pp; k++) w[k] = src[c * pp + k];
      const int info = chol_upper(w, p);
      if (info) fail = PGBP_STATUS(0x7ffffd, info);
      for (int s = 0; s < p; s++)
        for (int t = 0; t < p; t++) o[(int64_t)(sr.L(c) + s * p + t) * ldp] = t >= s ? w[t * p + s] : 0.0;
    }
    const double* mu = src + nc * pp;
    const double* v = mu + p;
    for (int t = 0; t < p; t++) o[(int64_t)(sr.mu() + t) * ldp] = mu[t];
    bool allzero = true, anyinf = false;
    for (int k = 0; k < pp; k++) if (v[k] != 0.0) allzero = false;
    for (int t = 0; t < p; t++) if (v[t * p + t] == INFINITY) anyinf = true;
    for (int k = 0; k < pp; k++) w[k] = allzero ? 0.0 : v[k];
    if (!allzero && !fail) {
      if (anyinf) fail = PGBP_STATUS(0x7ffff7, 1);  // improper root: nothing to draw from
      else {
        const int info = chol_upper(w, p);
        if (info) fail = PGBP_STATUS(0x7ffffd, info);
      }
    }
    for (int s = 0; s < p; s++)
      for (int t = 0; t < p; t++) o[(int64_t)(sr.LV() + s * p + t) * ldp] = (t >= s && !allzero) ? w[t * p + s] : 0.0;
    o[(int64_t)sr.kind() * ldp] = allzero ? 0.0 : 1.0;
    o[(int64_t)sr.fail() * ldp] = (double)fail;
  }
};

struct SimArgs {
  const SimNode* nodes;  // internal nodes, level order
  const SimNode* tips;   // one per data row (v < 0: no node has this row)
  const int32_t* prow;   // per parent entry: internal row of the parent
  const double* pgam;    // gamma_k
  const double* plen;    // t_k
  const int32_t* pcol;   // colour of the edge
  const double* prep;    // SimRows table
  int64_t ldp;
  const double* params;  // BM records (mixed-colour hybrids read the rates)
  const uint8_t* tip_missing;  // [ntips * p] or null
  double* soa;           // internal values of the chunk [ninternal * p][ldc]
  int64_t ldc;
  double* tipdata;       // [B][ntips][p] or null
  double* nodes_out;     // [B][nnodes][p] or null
  int32_t* status;
  int64_t e0, nparamsets, first;
  uint64_t seed;
  int32_t nnodes, ntips;
  SimRows sr;
};

// Value of node nd for element e0 + el: x = mean + L z (module comment of include/pgbp_b200.h, section simulate).
template <int MAXP>
PGBP_HD void sim_value(const SimArgs& a, const SimNode& nd, int64_t el, double* x) {
  const int p = a.sr.p;
  const int64_t eg = a.e0 + el;
  const double* th = a.prep + (a.nparamsets == 1 ? 0 : eg);
  const int64_t ldp = a.ldp;
  if (th[(int64_t)a.sr.fail() * ldp] != 0.0) {
#pragma unroll
    for (int t = 0; t < MAXP; t++) x[t] = NAN;
    return;
  }
  const uint64_t r = (uint64_t)(a.first + eg);
  double z[MAXP];
  const bool draw = nd.np == 0 ? th[(int64_t)a.sr.kind() * ldp] != 0.0 : nd.t0 != 0.0 || nd.color < 0;
#pragma unroll
  for (int k = 0; k < MAXP / 2; k++) {
    z[2 * k] = z[2 * k + 1] = 0.0;
    if (draw && 2 * k < p) normal_pair(a.seed, (uint32_t)nd.v, (uint32_t)k, (uint32_t)r, (uint32_t)(r >> 32), &z[2 * k], &z[2 * k + 1]);
  }
  if (a.sr.model == PGBP_MODEL_OU) {
    if (nd.np == 0) {
      x[0] = th[3 * ldp] + th[4 * ldp] * z[0];
      return;
    }
    const double g2 = th[0], alpha = th[ldp], theta = th[2 * ldp];
    double m = 0.0, var = 0.0;
    for (int k = 0; k < nd.np; k++) {
      const int j = nd.k0 + k;
      const double t = a.plen[j], gam = nd.np == 1 ? 1.0 : a.pgam[j];
      const double xp = a.soa[(int64_t)a.prow[j] * a.ldc + el];
      const double q = exp(-alpha * t), omq = -expm1(-alpha * t), omq2 = -expm1(-2.0 * alpha * t);
      m += gam * (q * xp + omq * theta);
      var += gam * gam * (g2 * omq2);
    }
    x[0] = m + sqrt(var) * z[0];
    return;
  }
  if (nd.np == 0) {  // root: mu (+ chol_lower(V) z for a proper prior)
#pragma unroll
    for (int t = 0; t < MAXP; t++) {
      if (t >= p) break;
      double s = 0.0;
      for (int u = 0; u <= t; u++) s += th[(int64_t)(a.sr.LV() + u * p + t) * ldp] * z[u];
      x[t] = th[(int64_t)(a.sr.mu() + t) * ldp] + s;
    }
    return;
  }
  double m[MAXP];
#pragma unroll
  for (int t = 0; t < MAXP; t++) m[t] = 0.0;
  for (int k = 0; k < nd.np; k++) {
    const int j = nd.k0 + k;
    const double c = nd.np == 1 ? 1.0 : a.pgam[j];
    const double* xp = a.soa + (int64_t)a.prow[j] * p * a.ldc + el;
#pragma unroll
    for (int t = 0; t < MAXP; t++)
      if (t < p) m[t] += c * xp[(int64_t)t * a.ldc];
  }
  if (nd.color >= 0) {  // L = sqrt(t0) chol_lower(R_c)
    const double st = sqrt(nd.t0);
    const int L0 = a.sr.L(nd.color);
#pragma unroll
    for (int t = 0; t < MAXP; t++) {
      if (t >= p) break;
      double s = 0.0;
      if (draw)
        for (int u = 0; u <= t; u++) s += th[(int64_t)(L0 + u * p + t) * ldp] * z[u];
      x[t] = draw ? m[t] + st * s : m[t];
    }
    return;
  }
  // hybrid whose parent edges differ in colour: L = chol_lower(sum_k gamma_k^2 t_k R_{c_k}), per thread (rare)
  const int pp = p * p;
  const double* R = a.params + (a.nparamsets == 1 ? 0 : eg) * (int64_t)(a.sr.nc * pp + p + pp);
  double w[MAXP * MAXP];
  for (int q = 0; q < pp; q++) w[q] = 0.0;
  for (int k = 0; k < nd.np; k++) {
    const int j = nd.k0 + k;
    const double f = a.pgam[j] * a.pgam[j] * a.plen[j];
    for (int q = 0; q < pp; q++) w[q] += f * R[a.pcol[j] * pp + q];
  }
  const int info = chol_upper(w, p);
  if (info) {
    status_fail(a.status, eg, PGBP_STATUS(0x7ffffc, info));
#pragma unroll
    for (int t = 0; t < MAXP; t++) x[t] = NAN;
    return;
  }
#pragma unroll
  for (int t = 0; t < MAXP; t++) {
    if (t >= p) break;
    double s = 0.0;
    for (int u = 0; u <= t; u++) s += w[t * p + u] * z[u];
    x[t] = m[t] + s;
  }
}

// the element's status word, recorded once (by the root's thread)
PGBP_HD void sim_root_status(const SimArgs& a, int64_t el) {
  const int64_t eg = a.e0 + el;
  const double f = a.prep[(a.nparamsets == 1 ? 0 : eg) + (int64_t)a.sr.fail() * a.ldp];
  if (f != 0.0) status_fail(a.status, eg, (int32_t)f);
}

template <int MAXP>
PGBP_HD void sim_level_thread(const SimArgs& a, int32_t n0, int64_t C, int64_t idx) {
  const int64_t i = idx / C, el = idx % C;
  const SimNode nd = a.nodes[n0 + i];
  const int p = a.sr.p;
  double x[MAXP];
  sim_value<MAXP>(a, nd, el, x);
  if (nd.np == 0) sim_root_status(a, el);
  double* o = a.soa + (int64_t)nd.row * p * a.ldc + el;
#pragma unroll
  for (int t = 0; t < MAXP; t++)
    if (t < p) o[(int64_t)t * a.ldc] = x[t];
  if (a.nodes_out) {
    double* no = a.nodes_out + ((a.e0 + el) * a.nnodes + nd.v) * p;
    for (int t = 0; t < p; t++) no[t] = x[t];
  }
}

// value of data row `row` for element el: the tip's value, NaN where the plan marks the trait missing (nodes_out
// keeps the true value)
template <int MAXP>
PGBP_HD void sim_tip_value(const SimArgs& a, int32_t row, int64_t el, double* x) {
  const SimNode nd = a.tips[row];
  const int p = a.sr.p;
  if (nd.v < 0) {
#pragma unroll
    for (int t = 0; t < MAXP; t++) x[t] = NAN;
    return;
  }
  sim_value<MAXP>(a, nd, el, x);
  if (a.nodes_out) {
    double* no = a.nodes_out + ((a.e0 + el) * a.nnodes + nd.v) * p;
    for (int t = 0; t < p; t++) no[t] = x[t];
  }
  if (a.tip_missing)
#pragma unroll
    for (int t = 0; t < MAXP; t++)
      if (t < p && a.tip_missing[(int64_t)row * p + t]) x[t] = NAN;
}

#ifndef PGBP_HOST_EMUL
__global__ void __launch_bounds__(128) k_sim_prep(SimPrep f, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) f(i);
}

template <int MAXP>
__global__ void __launch_bounds__(128) k_sim_level(SimArgs a, int32_t n0, int64_t C, int64_t total) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < total) sim_level_thread<MAXP>(a, n0, C, idx);
}

#define PGBP_SIM_TILE_E 32
#define PGBP_SIM_TILE_RP 128  // R * p <= 128 doubles per element and tile
// blockIdx.x: 32 elements of the chunk; blockIdx.y: R = max(1, 128 / p) consecutive data rows
template <int MAXP>
__global__ void __launch_bounds__(256) k_sim_tips(SimArgs a, int64_t C, int R, int32_t row0) {
  __shared__ double tile[PGBP_SIM_TILE_E][PGBP_SIM_TILE_RP + 1];
  const int p = a.sr.p;
  const int64_t e0 = (int64_t)blockIdx.x * PGBP_SIM_TILE_E;
  const int32_t r0 = row0 + (int32_t)blockIdx.y * R;
  const int nrow = min(R, a.ntips - r0);
  const int ne = C - e0 < PGBP_SIM_TILE_E ? (int)(C - e0) : PGBP_SIM_TILE_E;
  // 1. values: consecutive threads = consecutive elements of one row (parent reads coalesced)
  for (int w = threadIdx.x; w < PGBP_SIM_TILE_E * nrow; w += blockDim.x) {
    const int le = w % PGBP_SIM_TILE_E, rr = w / PGBP_SIM_TILE_E;
    if (le >= ne) continue;
    double x[MAXP];
    sim_tip_value<MAXP>(a, r0 + rr, e0 + le, x);
#pragma unroll
    for (int t = 0; t < MAXP; t++)
      if (t < p) tile[le][rr * p + t] = x[t];
  }
  __syncthreads();
  if (!a.tipdata) return;  // nodes only
  // 2. tipdata: element le's rows r0 .. r0 + nrow are one contiguous run of nrow * p doubles
  const int run = nrow * p;
  for (int w = threadIdx.x; w < ne * run; w += blockDim.x) {
    const int le = w / run, q = w % run;
    a.tipdata[((a.e0 + e0 + le) * a.ntips + r0) * p + q] = tile[le][q];
  }
}
#endif

namespace {

// Host-side form of one mem_parent table on one plan (cached on the batch), and its device copy.
struct SimPlan {
  std::vector<int32_t> mem_parent;  // the key
  std::vector<SimNode> nodes, tips;
  std::vector<int32_t> level_off;   // [nlevels + 1] ranges of `nodes`
  std::vector<int32_t> prow, pcol;
  std::vector<double> pgam, plen;
  int32_t ninternal = 0;
  // device
  std::vector<void*> owned;
  SimNode *d_nodes = nullptr, *d_tips = nullptr;
  int32_t *d_prow = nullptr, *d_pcol = nullptr;
  double *d_pgam = nullptr, *d_plen = nullptr;
  uint8_t* d_missing = nullptr;
  ~SimPlan() { for (void* v : owned) dev_free(v); }
};

template <class T>
int upload_vec(pgbp_batch* b, SimPlan* sp, T** dst, const T* src, size_t n) {
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, std::max<size_t>(1, n) * sizeof(T)));
  sp->owned.push_back(v);
  *dst = (T*)v;
  b->device_bytes += (int64_t)(n * sizeof(T));
  return h2d(v, src, n * sizeof(T), b->stream);
}

int build_plan(pgbp_batch* b, const int32_t* mem_parent, SimPlan* sp) {
  const FamilyTable& F = b->plan->fam;
  const int n = F.nnodes, nm = F.mem_off[n];
  sp->mem_parent.assign(mem_parent, mem_parent + nm);
  std::vector<int32_t> level(n, 0), nchild(n, 0);
  for (int v = 0; v < n; v++) {
    const int o0 = F.mem_off[v], o1 = F.mem_off[v + 1];
    if (mem_parent[o0] != -1) PGBP_FAIL(PGBP_EINVAL, "simulate: mem_parent of node %d's own entry must be -1", v);
    if (v > 0 && o1 - o0 < 2) PGBP_FAIL(PGBP_EINVAL, "simulate: node %d is not the root and has no parent", v);
    for (int k = o0 + 1; k < o1; k++) {
      const int q = mem_parent[k];
      if (q < 0 || q >= n) PGBP_FAIL(PGBP_EINVAL, "simulate: node %d: parent index %d out of range", v, q);
      if (q >= v) PGBP_FAIL(PGBP_EINVAL, "simulate: node %d: parent %d is not before it in preorder", v, q);
      level[v] = std::max(level[v], level[q] + 1);
      nchild[q]++;
    }
  }
  // internal nodes by level (stable: preorder inside a level); tips by data row
  std::vector<int32_t> order;
  for (int v = 0; v < n; v++) {
    if (F.node_datarow[v] < 0) order.push_back(v);
    else if (nchild[v]) PGBP_FAIL(PGBP_EINVAL, "simulate: node %d has a data row and children (tips must be leaves)", v);
  }
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return level[x] < level[y]; });
  std::vector<int32_t> row(n, -1);
  for (size_t i = 0; i < order.size(); i++) row[order[i]] = (int32_t)i;
  sp->ninternal = (int32_t)order.size();
  auto make = [&](int v, int32_t r) {
    const int o0 = F.mem_off[v], o1 = F.mem_off[v + 1];
    SimNode d{};
    d.v = v; d.row = r; d.k0 = (int32_t)sp->prow.size(); d.np = o1 - o0 - 1; d.color = 0; d.t0 = 0.0;
    for (int k = o0 + 1; k < o1; k++) {
      sp->prow.push_back(row[mem_parent[k]]);
      sp->pcol.push_back(F.mem_color[k]);
      sp->pgam.push_back(F.mem_gamma[k]);
      sp->plen.push_back(F.mem_length[k]);
      if (F.mem_color[k] != F.mem_color[o0 + 1]) d.color = -1;
    }
    if (d.np > 0 && d.color == 0) d.color = F.mem_color[o0 + 1];
    if (d.np == 1) d.t0 = F.mem_length[o0 + 1];
    else for (int k = o0 + 1; k < o1; k++) d.t0 += F.mem_gamma[k] * F.mem_gamma[k] * F.mem_length[k];
    return d;
  };
  sp->level_off.assign(1, 0);
  for (size_t i = 0; i < order.size(); i++) {
    const int v = order[i];
    if (i > 0 && level[v] != level[order[i - 1]]) sp->level_off.push_back((int32_t)i);
    sp->nodes.push_back(make(v, (int32_t)i));
  }
  sp->level_off.push_back((int32_t)order.size());
  SimNode none{};
  none.v = -1;
  sp->tips.assign(F.ntips, none);
  for (int v = 0; v < n; v++)
    if (F.node_datarow[v] >= 0) {
      if (sp->tips[F.node_datarow[v]].v >= 0) PGBP_FAIL(PGBP_EINVAL, "simulate: two nodes share data row %d", F.node_datarow[v]);
      sp->tips[F.node_datarow[v]] = make(v, F.node_datarow[v]);
    }
  PGBP_TRY(upload_vec(b, sp, &sp->d_nodes, sp->nodes.data(), sp->nodes.size()));
  PGBP_TRY(upload_vec(b, sp, &sp->d_tips, sp->tips.data(), sp->tips.size()));
  PGBP_TRY(upload_vec(b, sp, &sp->d_prow, sp->prow.data(), sp->prow.size()));
  PGBP_TRY(upload_vec(b, sp, &sp->d_pcol, sp->pcol.data(), sp->pcol.size()));
  PGBP_TRY(upload_vec(b, sp, &sp->d_pgam, sp->pgam.data(), sp->pgam.size()));
  PGBP_TRY(upload_vec(b, sp, &sp->d_plen, sp->plen.data(), sp->plen.size()));
  if (F.scoped) PGBP_TRY(upload_vec(b, sp, &sp->d_missing, F.tip_missing.data(), F.tip_missing.size()));
  return stream_sync(b->stream);  // the host vectors stay, but keep the upload out of later timings
}

int sim_check(pgbp_batch* b, int32_t model, int32_t ncolors, const int32_t* mem_parent, const void* params,
              int64_t nparamsets, int64_t first_replicate, const void* tipdata, const void* nodes) {
  if (!b || !params || !mem_parent) PGBP_FAIL(PGBP_EINVAL, "null argument");
  const pgbp_plan* p = b->plan;
  if (!p->has_families) PGBP_FAIL(PGBP_ESTATE, "simulate: the plan has no node-family table");
  if (model != PGBP_MODEL_BM && model != PGBP_MODEL_OU) PGBP_FAIL(PGBP_EINVAL, "simulate: unknown model %d", model);
  if (p->ntraits > PGBP_MAX_TRAITS) PGBP_FAIL(PGBP_EINVAL, "simulate: ntraits %d > %d", p->ntraits, PGBP_MAX_TRAITS);
  if (model == PGBP_MODEL_OU && (p->ntraits != 1 || ncolors != 1))
    PGBP_FAIL(PGBP_EINVAL, "simulate: the Ornstein-Uhlenbeck model needs ntraits == 1 and ncolors == 1");
  if (ncolors < p->fam.ncolors_min)
    PGBP_FAIL(PGBP_EINVAL, "simulate: ncolors %d but the family table uses colour %d", ncolors, p->fam.ncolors_min - 1);
  if (nparamsets != 1 && nparamsets != b->B) PGBP_FAIL(PGBP_EINVAL, "simulate: nparamsets must be 1 or B");
  if (nparamsets > 1 && b->group_size > 1)
    PGBP_FAIL(PGBP_EINVAL, "simulate: a shared-precision batch takes a single parameter record");
  if (first_replicate < 0) PGBP_FAIL(PGBP_EINVAL, "simulate: first_replicate < 0");
  if (!tipdata && !nodes) PGBP_FAIL(PGBP_EINVAL, "simulate: both outputs are null");
  return 0;
}

int get_plan(pgbp_batch* b, const int32_t* mem_parent, SimPlan** out) {
  SimPlan* sp = (SimPlan*)b->d_sim;
  if (!sp || !std::equal(sp->mem_parent.begin(), sp->mem_parent.end(), mem_parent)) {
    sim_free(b);
    std::unique_ptr<SimPlan> fresh(new SimPlan);
    PGBP_TRY(build_plan(b, mem_parent, fresh.get()));
    sp = fresh.release();
    b->d_sim = sp;
  }
  *out = sp;
  return 0;
}

struct SimLayout {
  int64_t ldp, C, ldc;
  size_t prep, soa;  // doubles
};

SimLayout layout(const pgbp_batch* b, const SimPlan* sp, const SimRows& sr, int64_t nparamsets) {
  SimLayout L;
  L.ldp = (nparamsets + 31) / 32 * 32;
  const int64_t per = std::max<int64_t>(1, (int64_t)sp->ninternal * sr.p) * 8;
  int64_t C = (int64_t)(PGBP_SIM_SCRATCH_BYTES / (uint64_t)per) / 32 * 32;
  C = std::max<int64_t>(32, C);
  L.C = std::min<int64_t>(b->B, C);
  L.ldc = (L.C + 31) / 32 * 32;
  L.prep = (size_t)sr.nrows() * (size_t)L.ldp;
  L.soa = (size_t)std::max(1, sp->ninternal * sr.p) * (size_t)L.ldc;
  return L;
}

template <int MAXP>
int launch_chunk(pgbp_batch* b, const SimPlan& sp, const SimArgs& a, int64_t C) {
  for (size_t l = 0; l + 1 < sp.level_off.size(); l++) {
    const int32_t n0 = sp.level_off[l];
    const int64_t total = (int64_t)(sp.level_off[l + 1] - n0) * C;
#ifdef PGBP_HOST_EMUL
    for (int64_t i = 0; i < total; i++) sim_level_thread<MAXP>(a, n0, C, i);
#else
    k_sim_level<MAXP><<<(unsigned)((total + 127) / 128), 128, 0, b->stream>>>(a, n0, C, total);
    PGBP_TRY(check_launch("k_sim_level"));
#endif
    b->launches++;
  }
  if (!a.tipdata && !a.nodes_out) return 0;
  const int p = a.sr.p, ntips = a.ntips;
  if (ntips == 0) return 0;
#ifdef PGBP_HOST_EMUL
  double x[MAXP];
  for (int64_t el = 0; el < C; el++)
    for (int32_t row = 0; row < ntips; row++) {
      sim_tip_value<MAXP>(a, row, el, x);
      if (a.tipdata)
        for (int t = 0; t < p; t++) a.tipdata[((a.e0 + el) * ntips + row) * p + t] = x[t];
    }
  b->launches++;
#else
  const int R = std::max(1, PGBP_SIM_TILE_RP / p);
  const int64_t nty = (ntips + R - 1) / R;
  for (int64_t y0 = 0; y0 < nty; y0 += 65535) {
    const unsigned gy = (unsigned)std::min<int64_t>(65535, nty - y0);
    dim3 grid((unsigned)((C + PGBP_SIM_TILE_E - 1) / PGBP_SIM_TILE_E), gy);
    k_sim_tips<MAXP><<<grid, 256, 0, b->stream>>>(a, C, R, (int32_t)(y0 * R));
    PGBP_TRY(check_launch("k_sim_tips"));
    b->launches++;
  }
#endif
  return 0;
}

// Enqueue the whole simulation: d_params on the device, outputs on the device ([B][ntips][p], [B][nnodes][p]).
int sim_enqueue(pgbp_batch* b, int32_t model, int32_t ncolors, const int32_t* mem_parent, const double* d_params,
                int64_t nparamsets, int64_t seed, int64_t first_replicate, double* d_tip, double* d_nodes,
                size_t extra_doubles, double** extra) {
  PGBP_TRY(set_device(b->device));
  SimPlan* sp;
  PGBP_TRY(get_plan(b, mem_parent, &sp));
  const pgbp_plan* p = b->plan;
  const SimRows sr{p->ntraits, ncolors, model};
  const SimLayout L = layout(b, sp, sr, nparamsets);
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (L.prep + L.soa + extra_doubles)));
  double* d_prep = b->scratch;
  double* d_soa = d_prep + L.prep;
  if (extra) {  // the host entry point stages its records here and then calls again with extra == nullptr
    *extra = d_soa + L.soa;
    return 0;
  }
  SimPrep prep{d_params, d_prep, L.ldp, sr};
#ifdef PGBP_HOST_EMUL
  for (int64_t i = 0; i < nparamsets; i++) prep(i);
#else
  k_sim_prep<<<(unsigned)((nparamsets + 127) / 128), 128, 0, b->stream>>>(prep, nparamsets);
  PGBP_TRY(check_launch("k_sim_prep"));
#endif
  b->launches++;
  SimArgs a{};
  a.nodes = sp->d_nodes; a.tips = sp->d_tips;
  a.prow = sp->d_prow; a.pgam = sp->d_pgam; a.plen = sp->d_plen; a.pcol = sp->d_pcol;
  a.prep = d_prep; a.ldp = L.ldp; a.params = d_params; a.tip_missing = sp->d_missing;
  a.soa = d_soa; a.ldc = L.ldc; a.tipdata = d_tip; a.nodes_out = d_nodes; a.status = b->status;
  a.nparamsets = nparamsets; a.first = first_replicate; a.seed = (uint64_t)seed;
  a.nnodes = p->fam.nnodes; a.ntips = p->fam.ntips; a.sr = sr;
  for (int64_t e0 = 0; e0 < b->B; e0 += L.C) {
    a.e0 = e0;
    const int64_t C = std::min(L.C, b->B - e0);
    if (sr.p <= 4) PGBP_TRY(launch_chunk<4>(b, *sp, a, C));
    else if (sr.p <= 8) PGBP_TRY(launch_chunk<8>(b, *sp, a, C));
    else PGBP_TRY(launch_chunk<PGBP_MAX_TRAITS>(b, *sp, a, C));
  }
  return 0;
}

}  // namespace

void sim_free(pgbp_batch* b) {
  delete (SimPlan*)b->d_sim;
  b->d_sim = nullptr;
}

}  // namespace pgbp

extern "C" {

int32_t pgbp_simulate_device(pgbp_batch* b, int32_t model, int32_t ncolors, const int32_t* mem_parent,
                             const double* d_params, int64_t nparamsets, int64_t seed, int64_t first_replicate,
                             double* d_tipdata, double* d_nodes) {
  PGBP_TRY(sim_check(b, model, ncolors, mem_parent, d_params, nparamsets, first_replicate, d_tipdata, d_nodes));
  return sim_enqueue(b, model, ncolors, mem_parent, d_params, nparamsets, seed, first_replicate, d_tipdata, d_nodes, 0,
                     nullptr);
}

int32_t pgbp_simulate(pgbp_batch* b, int32_t model, int32_t ncolors, const int32_t* mem_parent, const double* params,
                      int64_t nparamsets, int64_t seed, int64_t first_replicate, double* tipdata, double* nodes) {
  PGBP_TRY(sim_check(b, model, ncolors, mem_parent, params, nparamsets, first_replicate, tipdata, nodes));
  const pgbp_plan* p = b->plan;
  const int pt = p->ntraits;
  const size_t plen = model == PGBP_MODEL_OU ? 5 : (size_t)ncolors * pt * pt + pt + (size_t)pt * pt;
  const size_t np = plen * (size_t)nparamsets;
  const size_t nt = tipdata ? (size_t)b->B * p->fam.ntips * pt : 0;
  const size_t nn = nodes ? (size_t)b->B * p->fam.nnodes * pt : 0;
  double* d_extra = nullptr;
  PGBP_TRY(sim_enqueue(b, model, ncolors, mem_parent, nullptr, nparamsets, seed, first_replicate, nullptr, nullptr,
                       np + nt + nn, &d_extra));
  PGBP_TRY(h2d(d_extra, params, sizeof(double) * np, b->stream));
  double* d_tip = tipdata ? d_extra + np : nullptr;
  double* d_nodes = nodes ? d_extra + np + nt : nullptr;
  PGBP_TRY(sim_enqueue(b, model, ncolors, mem_parent, d_extra, nparamsets, seed, first_replicate, d_tip, d_nodes, 0,
                       nullptr));
  if (tipdata) PGBP_TRY(d2h(tipdata, d_tip, sizeof(double) * nt, b->stream));
  if (nodes) PGBP_TRY(d2h(nodes, d_nodes, sizeof(double) * nn, b->stream));
  return stream_sync(b->stream);
}

}  // extern "C"
