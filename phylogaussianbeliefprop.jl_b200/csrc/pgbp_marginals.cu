// Posterior moments of variable subsets of beliefs (pgbp_marginal_moments): the marginal Gaussian of positions
// `pos` of belief i, mu = (J^-1 h)[pos] and cov = (J^-1)[pos, pos] (integratebelief!, src/beliefupdates.jl:168-200,
// and inv(J) restricted to the subset), for many (belief, positions) queries and every element in one call.
//
// The host groups the queries by belief and uploads one descriptor per queried belief (MargDesc) plus the query
// table; one launch per shape class (as integrate_launch), blockIdx.y over the beliefs of the class.  A thread =
// one (element, belief): it reads and factorises the belief once and writes only the requested rows, so ancestral
// reconstruction of a large network moves p + p(p+1)/2 doubles per node instead of a whole cluster covariance.
#include <algorithm>
#include <climits>
#include <vector>

#include "pgbp_kernels.cuh"
#include "pgbp_launch.h"
#include "pgbp_shapes.h"

using namespace pgbp;

namespace pgbp {

#ifndef PGBP_HOST_EMUL
template <int MAXM>
__global__ void __launch_bounds__(128) k_marginals(const double* state, int32_t* status, int64_t B, int64_t ld,
                                                   const MargDesc* descs, const int32_t* qtab, const int32_t* qpos,
                                                   double* mu_soa, double* cov_soa, int64_t ld_out, JSide js) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  marginal_thread<MAXM>(state, status, ld, e, descs[blockIdx.y], qtab, qpos, mu_soa, cov_soa, ld_out, jcolumn(js, e), js.ld);
}
#endif

namespace {

// shape classes of integrate_launch: M <= 4 / 12 / 32 / PGBP_MAX_DIM
int shape_class_of(int m) { return m <= 4 ? 0 : m <= 12 ? 1 : m <= 32 ? 2 : 3; }

template <int MAXM>
int launch_class(pgbp_batch* b, const MargDesc* d_descs, int n, const int32_t* d_qtab, const int32_t* d_qpos,
                 double* d_mu, double* d_cov, const JSide& js) {
#ifdef PGBP_HOST_EMUL
  for (int i = 0; i < n; i++)
    for (int64_t e = 0; e < b->B; e++)
      marginal_thread<MAXM>(b->state, b->status, b->ld, e, d_descs[i], d_qtab, d_qpos, d_mu, d_cov, b->ld,
                            jcolumn(js, e), js.ld);
  b->launches++;
  return 0;
#else
  const unsigned gx = (unsigned)((b->B + 127) / 128);
  for (int i0 = 0; i0 < n; i0 += 65535) {  // gridDim.y limit
    const unsigned gy = (unsigned)std::min(n - i0, 65535);
    k_marginals<MAXM><<<dim3(gx, gy), 128, 0, b->stream>>>(b->state, b->status, b->B, b->ld, d_descs + i0, d_qtab,
                                                           d_qpos, d_mu, d_cov, b->ld, js);
    b->launches++;
    PGBP_TRY(check_launch("k_marginals"));
  }
  return 0;
#endif
}

// Validated, grouped form of one call's queries.
struct MargPlan {
  std::vector<MargDesc> descs;  // sorted by shape class, then belief
  int ncls[4] = {0, 0, 0, 0};   // beliefs per class
  std::vector<int32_t> qtab;    // [4 * nq] in grouped order: (k, position offset, mu row, cov row)
  std::vector<int32_t> qpos;    // positions in grouped order
  std::vector<int64_t> mu_row, cov_row;  // per query in the caller's order
  int64_t nmu = 0, ncov = 0, ncov_full = 0;  // sum k, sum k(k+1)/2, sum k^2
  bool any_sepset = false;
};

int plan_queries(const pgbp_batch* b, int32_t nq, const int32_t* qb, const int32_t* qoff, const int32_t* qpos,
                 MargPlan* mp) {
  const pgbp_plan* p = b->plan;
  if (nq < 1) PGBP_FAIL(PGBP_EINVAL, "marginal moments: nq must be >= 1");
  if (!qb || !qoff || !qpos) PGBP_FAIL(PGBP_EINVAL, "marginal moments: null query array");
  if (qoff[0] < 0) PGBP_FAIL(PGBP_EINVAL, "marginal moments: q_off[0] < 0");
  std::vector<int32_t> seen((size_t)p->max_dim + 1, -1);
  mp->mu_row.resize(nq);
  mp->cov_row.resize(nq);
  for (int32_t q = 0; q < nq; q++) {
    const int32_t i = qb[q];
    if (i < 0 || i >= p->nbeliefs) PGBP_FAIL(PGBP_EINVAL, "marginal moments: query %d names belief %d (out of range)", q, i);
    if (qoff[q + 1] < qoff[q]) PGBP_FAIL(PGBP_EINVAL, "marginal moments: q_off decreases at query %d", q);
    const int m = p->dim[i];
    const int64_t k = (int64_t)qoff[q + 1] - qoff[q];
    for (int32_t r = qoff[q]; r < qoff[q + 1]; r++) {
      const int32_t x = qpos[r];
      if (x < 0 || x >= m) PGBP_FAIL(PGBP_EINVAL, "marginal moments: query %d: position %d outside [0, %d)", q, x, m);
      if (seen[x] == q) PGBP_FAIL(PGBP_EINVAL, "marginal moments: query %d: position %d repeated", q, x);
      seen[x] = q;
    }
    mp->mu_row[q] = mp->nmu;
    mp->cov_row[q] = mp->ncov;
    mp->nmu += k;
    mp->ncov += k * (k + 1) / 2;
    mp->ncov_full += k * k;
    if (i >= p->nclusters) mp->any_sepset = true;
  }
  if (mp->ncov_full > INT32_MAX) PGBP_FAIL(PGBP_EINVAL, "marginal moments: too many output rows in one call");
  // group by (shape class, belief); queries of one belief stay in the caller's order
  std::vector<int32_t> order(nq);
  for (int32_t q = 0; q < nq; q++) order[q] = q;
  auto key = [&](int32_t q) { return std::make_pair(shape_class_of(p->dim[qb[q]]), qb[q]); };
  std::stable_sort(order.begin(), order.end(), [&](int32_t x, int32_t y) { return key(x) < key(y); });
  mp->qtab.resize(4 * (size_t)nq);
  for (int32_t t = 0; t < nq; t++) {
    const int32_t q = order[t], i = qb[q];
    if (t == 0 || qb[order[t - 1]] != i) {
      MargDesc d{};
      d.jslot = p->jslot[i];
      d.hrow = batch_hrow(b, i);
      d.m = p->dim[i];
      d.t0 = t;
      mp->descs.push_back(d);
      mp->ncls[shape_class_of(d.m)]++;
    }
    mp->descs.back().t1 = t + 1;
    mp->qtab[4 * (size_t)t] = qoff[q + 1] - qoff[q];
    mp->qtab[4 * (size_t)t + 1] = (int32_t)mp->qpos.size();
    mp->qtab[4 * (size_t)t + 2] = (int32_t)mp->mu_row[q];
    mp->qtab[4 * (size_t)t + 3] = (int32_t)mp->cov_row[q];
    mp->qpos.insert(mp->qpos.end(), qpos + qoff[q], qpos + qoff[q + 1]);
  }
  return 0;
}

size_t index_bytes(const MargPlan& mp) {
  return sizeof(MargDesc) * mp.descs.size() + sizeof(int32_t) * (mp.qtab.size() + mp.qpos.size());
}

// Upload the index data to `d_index` (device, 8-byte aligned, index_bytes(mp) long) and launch every class.
int enqueue(pgbp_batch* b, const MargPlan& mp, char* d_index, double* d_mu, double* d_cov) {
  if (mp.any_sepset) PGBP_TRY(batch_materialize_sepsets(b));
  MargDesc* d_descs = (MargDesc*)d_index;
  int32_t* d_qtab = (int32_t*)(d_descs + mp.descs.size());
  int32_t* d_qpos = d_qtab + mp.qtab.size();
  // pageable sources: cudaMemcpyAsync returns once they are staged, so the vectors may go out of scope
  PGBP_TRY(h2d(d_descs, mp.descs.data(), sizeof(MargDesc) * mp.descs.size(), b->stream));
  PGBP_TRY(h2d(d_qtab, mp.qtab.data(), sizeof(int32_t) * mp.qtab.size(), b->stream));
  PGBP_TRY(h2d(d_qpos, mp.qpos.data(), sizeof(int32_t) * mp.qpos.size(), b->stream));
  const JSide js = batch_jside(b);
  int first = 0;
  for (int c = 0; c < 4; c++) {
    const int n = mp.ncls[c];
    if (!n) continue;
    const MargDesc* dd = d_descs + first;
    switch (c) {
      case 0: PGBP_TRY(launch_class<4>(b, dd, n, d_qtab, d_qpos, d_mu, d_cov, js)); break;
      case 1: PGBP_TRY(launch_class<12>(b, dd, n, d_qtab, d_qpos, d_mu, d_cov, js)); break;
      case 2: PGBP_TRY(launch_class<32>(b, dd, n, d_qtab, d_qpos, d_mu, d_cov, js)); break;
      default: PGBP_TRY(launch_class<PGBP_MAX_DIM>(b, dd, n, d_qtab, d_qpos, d_mu, d_cov, js)); break;
    }
    first += n;
  }
  return 0;
}

}  // namespace
}  // namespace pgbp

extern "C" {

int32_t pgbp_marginal_moments_device(pgbp_batch* b, int32_t nq, const int32_t* q_belief, const int32_t* q_off,
                                     const int32_t* q_pos, double* d_mu, double* d_cov) {
  if (!b || !d_mu) PGBP_FAIL(PGBP_EINVAL, "null argument");
  MargPlan mp;
  PGBP_TRY(plan_queries(b, nq, q_belief, q_off, q_pos, &mp));
  PGBP_TRY(set_device(b->device));
  PGBP_TRY(batch_need_scratch(b, index_bytes(mp)));
  return enqueue(b, mp, (char*)b->scratch, d_mu, d_cov);
}

int32_t pgbp_marginal_moments(pgbp_batch* b, int32_t nq, const int32_t* q_belief, const int32_t* q_off,
                              const int32_t* q_pos, double* mu, double* cov) {
  if (!b || !mu) PGBP_FAIL(PGBP_EINVAL, "null argument");
  MargPlan mp;
  PGBP_TRY(plan_queries(b, nq, q_belief, q_off, q_pos, &mp));
  // the transposes to the host layout take at most 65535 * 32 columns (gridDim.y of k_soa_to_aos)
  if (mp.nmu > 65535 * 32 || (cov && mp.ncov_full > 65535 * 32))
    PGBP_FAIL(PGBP_EINVAL, "marginal moments: too many output columns for one host call (split the queries)");
  PGBP_TRY(set_device(b->device));
  const int64_t ld = b->ld, B = b->B;
  const int64_t ncov = cov ? mp.ncov : 0, nfull = cov ? mp.ncov_full : 0;
  // scratch: mu SoA | packed cov SoA | AoS staging | index data | full-square slot table of the covariances
  const size_t stage = (size_t)B * (size_t)std::max(mp.nmu, nfull);
  const size_t nd_soa = (size_t)ld * (size_t)(mp.nmu + ncov);
  const size_t idx = index_bytes(mp);
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (nd_soa + stage) + (idx + 7) / 8 * 8 + sizeof(int32_t) * (size_t)nfull));
  double* d_mu = b->scratch;
  double* d_cov = cov ? d_mu + ld * mp.nmu : nullptr;
  double* d_aos = b->scratch + nd_soa;
  char* d_index = (char*)(d_aos + stage);
  int32_t* d_slot = (int32_t*)(d_index + (idx + 7) / 8 * 8);
  PGBP_TRY(enqueue(b, mp, d_index, d_mu, d_cov));
  if (mp.nmu > 0) {
    PGBP_TRY(soa_to_aos(b, d_mu, ld, d_aos, (int)mp.nmu, nullptr));
    PGBP_TRY(d2h(mu, d_aos, sizeof(double) * (size_t)B * (size_t)mp.nmu, b->stream));
  }
  if (cov && nfull > 0) {
    // host layout: column-major k x k per query, both triangles, from the packed upper rows
    std::vector<int32_t> sl((size_t)nfull);
    size_t w = 0;
    for (int32_t q = 0; q < nq; q++) {
      const int k = q_off[q + 1] - q_off[q];
      for (int c = 0; c < k; c++)
        for (int r = 0; r < k; r++) sl[w++] = (int32_t)(mp.cov_row[q] + (r <= c ? pk(r, c) : pk(c, r)));
    }
    PGBP_TRY(h2d(d_slot, sl.data(), sizeof(int32_t) * sl.size(), b->stream));
    PGBP_TRY(soa_to_aos(b, d_cov, ld, d_aos, (int)nfull, d_slot));
    PGBP_TRY(d2h(cov, d_aos, sizeof(double) * (size_t)B * (size_t)nfull, b->stream));
  }
  return stream_sync(b->stream);
}

}  // extern "C"
