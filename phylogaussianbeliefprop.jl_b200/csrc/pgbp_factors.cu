// K1 factor assignment, K4 factored energy, K5 regularisation.
#include <algorithm>
#include <set>

#include "pgbp_factors.cuh"
#include "pgbp_kernels.cuh"
#include "pgbp_launch.h"

using namespace pgbp;

namespace pgbp {

// --------------------------------------------------------------------------
// generic launcher: body(e, y) for e < B, y < ny
// --------------------------------------------------------------------------
#ifndef PGBP_HOST_EMUL
template <class F>
__global__ void __launch_bounds__(128) k_generic(F f, int64_t B) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  f(e, (int)blockIdx.y);
}
// same, at least MINB blocks of 128 threads per SM (caps registers; for K1)
template <class F, int MINB>
__global__ void __launch_bounds__(128, MINB) k_generic_occ(F f, int64_t B) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  f(e, (int)blockIdx.y);
}

// Few elements, many rows (the group batch of a shared-precision batch: one element per parameter vector, 10^5
// clusters): one thread per ROW y instead of one block per row with a single live thread.
template <class F>
__global__ void __launch_bounds__(128) k_generic_rows(F f, int64_t n, int ny) {
  const int y = blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= ny) return;
  for (int64_t e = 0; e < n; e++) f(e, y);
}
#endif

template <class F, int MINB = 0>
static int launch_generic(pgbp_batch* b, const char* name, int64_t n, int ny, F f) {
  if (ny <= 0 || n <= 0) return 0;
#ifdef PGBP_HOST_EMUL
  for (int y = 0; y < ny; y++)
    for (int64_t e = 0; e < n; e++) f(e, y);
  b->launches++;
#else
  if (n <= 4 && ny >= 1024) {
    F g = f;
    g.y0 = 0;
    k_generic_rows<<<(unsigned)((ny + 127) / 128), 128, 0, b->stream>>>(g, n, ny);
    b->launches++;
    return check_launch(name);
  }
  for (int y0 = 0; y0 < ny; y0 += 65535) {
    const int cnt = std::min(65535, ny - y0);
    F g = f;
    g.y0 = y0;
    dim3 grid((unsigned)((n + 127) / 128), (unsigned)cnt);
    if constexpr (MINB > 0) k_generic_occ<F, MINB><<<grid, 128, 0, b->stream>>>(g, n);
    else k_generic<<<grid, 128, 0, b->stream>>>(g, n);
    b->launches++;
  }
#endif
  return check_launch(name);
}

// --------------------------------------------------------------------------
// K1: per-parameter-set preparation
// --------------------------------------------------------------------------
struct ThetaPrep {
  const double* params;  // AoS [np][nc*p*p + p + p*p]
  double* theta;         // SoA [rows][ldp]
  int64_t ldp;
  ThetaRows tr;
  int y0 = 0;
  PGBP_HD void operator()(int64_t ip, int) const {
    const int p = tr.p, nc = tr.nc, pp = p * p;
    const double* src = params + ip * (int64_t)(nc * pp + p + pp);
    double w[PGBP_MAX_TRAITS * PGBP_MAX_TRAITS], out[PGBP_MAX_TRAITS * PGBP_MAX_TRAITS];
    double* th = theta + ip;
    double kind = 0.0;
    for (int c = 0; c < nc; c++) {
      for (int k = 0; k < pp; k++) {
        w[k] = src[c * pp + k];
        th[(int64_t)(tr.R(c) + k) * ldp] = w[k];
      }
      double ld;
      const int info = spd_inverse_logdet(w, out, p, &ld);
      if (info) kind = -(double)info;
      for (int k = 0; k < pp; k++) th[(int64_t)(tr.P(c) + k) * ldp] = out[k];
      th[(int64_t)tr.g0(c) * ldp] = -0.5 * (p * PGBP_LOG2PI + ld);  // branch_logdet_variance
    }
    const double* mu = src + nc * pp;
    const double* v = mu + p;
    for (int k = 0; k < p; k++) th[(int64_t)(tr.mu() + k) * ldp] = mu[k];
    bool allzero = true, anyinf = false;
    for (int k = 0; k < pp; k++) if (v[k] != 0.0) allzero = false;
    for (int k = 0; k < p; k++) if (v[k * p + k] == INFINITY) anyinf = true;
    double rootg = 0.0;
    for (int k = 0; k < pp; k++) out[k] = 0.0;
    double rh[PGBP_MAX_TRAITS];
    for (int k = 0; k < p; k++) rh[k] = 0.0;
    if (kind >= 0.0) {
      if (allzero) kind = 0.0;
      else if (anyinf) kind = 2.0;
      else {
        kind = 1.0;
        for (int k = 0; k < pp; k++) w[k] = v[k];
        double ld;
        const int info = spd_inverse_logdet(w, out, p, &ld);  // j = inv(v); logdet(j) = -ld
        if (info) kind = -(double)info;
        double quad = 0.0;
        for (int r = 0; r < p; r++) {
          double s = 0.0;
          for (int c = 0; c < p; c++) s += out[c * p + r] * mu[c];
          rh[r] = s;
          quad += mu[r] * s;
        }
        rootg = 0.5 * (-p * PGBP_LOG2PI - ld - quad);  // src/evomodels/evomodels.jl:394
      }
    }
    for (int k = 0; k < pp; k++) th[(int64_t)(tr.rootP() + k) * ldp] = out[k];
    for (int k = 0; k < p; k++) th[(int64_t)(tr.rooth() + k) * ldp] = rh[k];
    th[(int64_t)tr.rootg() * ldp] = rootg;
    th[(int64_t)tr.kind() * ldp] = kind;
  }
};

// K1 main: one thread = (cluster y, element e).  Zeroes the cluster, then adds
// the factor of every node family assigned to it, in node order
// (src/beliefs.jl:798-859), with evidence absorbed in closed form:
//   phi_v = N(sum_a c_a x_a ; 0, j^-1),  c = (1, -gamma_1, ..),  fixed members
//   contribute z = sum c_a y_a:  J_ab += c_a c_b j,  h_b -= c_b j z,
//   g += g_v - z'jz/2   (absorbevidence!, src/beliefupdates.jl:210-231).
struct AssignBody {
  FamDev F;
  const double* theta;
  int64_t ldp;
  const double* tip;  // SoA [ntips*p][ldd]
  int64_t ldd;
  double* state;
  int32_t* status;
  int64_t ld;
  int64_t np, nd;
  int pairing;
  ThetaRows tr;
  int64_t gs = 0;  // != 0: element side of a shared-precision batch -- h and g only (compact rows in cl_hslot / cl_gslot);
                   // the J rows are the group batch's and are assigned there
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const { run(e, y + y0); }
  PGBP_HD void run(int64_t e, int c) const {
    const int p = F.p, pp = p * p;
    int64_t ip, id;
    if (pairing == PGBP_PAIR_PRODUCT) { ip = e / nd; id = e % nd; }
    else { ip = np == 1 ? 0 : e; id = nd == 1 ? 0 : e; }
    const double* th = theta + ip;
    const double* td = tip + id;
    double* st = state + e;
    const bool lead = this->gs == 0;
    const int64_t js = F.cl_jslot[c], hs = F.cl_hslot[c], gs = F.cl_gslot[c];
    const int m = F.cl_dim[c];
    if (lead) for (int q = 0; q < tri(m); q++) st[(js + q) * ld] = 0.0;
    for (int q = 0; q < m; q++) st[(hs + q) * ld] = 0.0;
    double g = 0.0;
    const double kind = th[(int64_t)tr.kind() * ldp];
    if (kind < 0.0) {
      if (c == 0) status_fail(status, e, PGBP_STATUS(0x7ffffd, (int)(-kind)));
      st[gs * ld] = NAN;
      return;
    }
    double j[PGBP_MAX_TRAITS * PGBP_MAX_TRAITS], w[PGBP_MAX_TRAITS * PGBP_MAX_TRAITS];
    double z[PGBP_MAX_TRAITS], jz[PGBP_MAX_TRAITS];
    for (int iv = F.clu_off[c]; iv < F.clu_off[c + 1]; iv++) {
      const int v = F.clu_node[iv];
      const int k0 = F.mem_off[v], nm = F.mem_off[v + 1] - k0;
      if (nm == 1) {  // root family (src/beliefs.jl:803-807)
        const int pos = F.mem_pos[k0];
        if (pos < 0 || kind != 1.0) continue;  // fixed root, or improper prior: factor == 1
        for (int cc = 0; cc < p; cc++) {
          if (lead) for (int r = 0; r <= cc; r++) st[(js + pk(pos + r, pos + cc)) * ld] += th[(int64_t)(tr.rootP() + cc * p + r) * ldp];
          st[(hs + pos + cc) * ld] += th[(int64_t)(tr.rooth() + cc) * ldp];
        }
        g += th[(int64_t)tr.rootg() * ldp];
        continue;
      }
      // precision block j and log-normaliser of the family
      double gv;
      bool samecolor = true;
      for (int k = k0 + 2; k < k0 + nm; k++) if (F.mem_color[k] != F.mem_color[k0 + 1]) samecolor = false;
      if (samecolor) {
        const int col = F.mem_color[k0 + 1];
        double t0 = 0.0;
        if (nm == 2) t0 = F.mem_length[k0 + 1];
        else for (int k = k0 + 1; k < k0 + nm; k++) t0 += F.mem_gamma[k] * F.mem_gamma[k] * F.mem_length[k];
        for (int q = 0; q < pp; q++) j[q] = th[(int64_t)(tr.P(col) + q) * ldp] / t0;
        gv = th[(int64_t)tr.g0(col) * ldp] - 0.5 * p * log(t0);
      } else {  // heterogeneous hybrid: j = (sum gamma^2 t R_c)^-1 (src/evomodels/heterogeneousmodels.jl:135-150)
        for (int q = 0; q < pp; q++) w[q] = 0.0;
        for (int k = k0 + 1; k < k0 + nm; k++) {
          const double f = F.mem_gamma[k] * F.mem_gamma[k] * F.mem_length[k];
          const int col = F.mem_color[k];
          for (int q = 0; q < pp; q++) w[q] += f * th[(int64_t)(tr.R(col) + q) * ldp];
        }
        double ldv;
        const int info = spd_inverse_logdet(w, j, p, &ldv);
        if (info) { status_fail(status, e, PGBP_STATUS(0x7ffffc, info)); st[gs * ld] = NAN; return; }
        gv = -0.5 * (p * PGBP_LOG2PI + ldv);
      }
      // evidence: z = sum over fixed members of c_a * value_a
      bool anyfixed = false;
      for (int t = 0; t < p; t++) z[t] = 0.0;
      for (int a = 0; a < nm; a++) {
        if (F.mem_pos[k0 + a] >= 0) continue;
        anyfixed = true;
        const double ca = a == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + a]);
        if (a == 0) {
          const int row = F.node_datarow[v];
          for (int t = 0; t < p; t++) z[t] += ca * td[(int64_t)(row * p + t) * ldd];
        } else {
          for (int t = 0; t < p; t++) z[t] += ca * th[(int64_t)(tr.mu() + t) * ldp];
        }
      }
      if (anyfixed) {
        // missing tip data (NaN) needs trait-level scopes (src/beliefs.jl:505-559): not handled on the
        // device -- flag the element instead of propagating NaNs silently
        for (int t = 0; t < p; t++) if (z[t] != z[t]) status_fail(status, e, PGBP_STATUS(0x7ffffa, t + 1));
        double quad = 0.0;
        for (int r = 0; r < p; r++) {
          double s = 0.0;
          for (int cc = 0; cc < p; cc++) s += j[cc * p + r] * z[cc];
          jz[r] = s;
          quad += z[r] * s;
        }
        gv -= 0.5 * quad;
      }
      g += gv;
      for (int a = 0; a < nm; a++) {
        const int pa = F.mem_pos[k0 + a];
        if (pa < 0) continue;
        const double ca = a == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + a]);
        if (anyfixed)
          for (int t = 0; t < p; t++) st[(hs + pa + t) * ld] -= ca * jz[t];
        for (int bq = a; lead && bq < nm; bq++) {
          const int pb = F.mem_pos[k0 + bq];
          if (pb < 0) continue;
          const double cb = bq == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + bq]);
          const double cab = ca * cb;
          for (int tb = 0; tb < p; tb++)
            for (int ta = 0; ta < (bq == a ? tb + 1 : p); ta++) {
              const int r = pa + ta, cc = pb + tb;  // pa <= pb: member positions increase along the family
              st[(js + (r <= cc ? pk(r, cc) : pk(cc, r))) * ld] += cab * j[tb * p + ta];
            }
        }
      }
    }
    st[gs * ld] = g;
  }
};

// K1 for plans with trait-level scopes (missing data).  One thread = (cluster, element); it follows the
// reference's own sequence for every node family of the cluster (src/beliefs.jl:798-859):
//   full factor phi_v over (child, parents) x traits  (homogeneousbrownianmotion.jl:222-351,
//   heterogeneousmodels.jl:119-150, evomodels.jl:377-396)
//   -> absorbleaf!: absorb the observed traits of a leaf, marginalise its missing ones (beliefupdates.jl:266-274)
//   -> absorbevidence! of a fixed root among the parents (beliefs.jl:828-831)
//   -> marginalise the child's out-of-scope traits, drop the parents' (beliefs.jl:836-857; see below)
//   -> mult! into the cluster at the scope positions (beliefs.jl:858).
// The working factor is a dense packed-upper matrix over the live variables in thread-local memory
// (<= PGBP_SCOPED_MAXN variables): this path is about coverage, not speed.  marginalize() keeps the
// reference's shortcuts (beliefupdates.jl:56,62-66) and failure rule (status instead of an exception).
struct ScopedFactor {
  double A[PGBP_SCOPED_MAXN * (PGBP_SCOPED_MAXN + 1) / 2];  // packed upper over live variables
  double Bq[PGBP_SCOPED_MAXN * (PGBP_SCOPED_MAXN + 1) / 2];  // scratch (permuted copy)
  double h[PGBP_SCOPED_MAXN], hb[PGBP_SCOPED_MAXN];
  int16_t id[PGBP_SCOPED_MAXN], idb[PGBP_SCOPED_MAXN];  // original variable (member * p + trait) of each live position
  int n;
  double g;
  PGBP_HD double& a(int r, int c) { return r <= c ? A[pk(r, c)] : A[pk(c, r)]; }
  // absorbevidence! (beliefupdates.jl:210-231) of the live positions flagged in `sel` with values val[pos]
  PGBP_HD void absorb(const bool* sel, const double* val) {
    double gl = 0.0, quad = 0.0;
    for (int i = 0; i < n; i++) if (sel[i]) {
      gl += h[i] * val[i];
      double s = 0.0;
      for (int j = 0; j < n; j++) if (sel[j]) s += a(i, j) * val[j];
      quad += s * val[i];
    }
    g += gl - 0.5 * quad;
    for (int k = 0; k < n; k++) if (!sel[k]) {
      double s = 0.0;
      for (int j = 0; j < n; j++) if (sel[j]) s += a(k, j) * val[j];
      h[k] -= s;
    }
    compact_keep(sel);
  }
  // drop the flagged positions (keep the others, order preserved)
  PGBP_HD void compact_keep(const bool* drop) {
    int m = 0;
    for (int c = 0; c < n; c++) {
      if (drop[c]) continue;
      int mr = 0;
      for (int r = 0; r <= c; r++) {
        if (drop[r]) continue;
        Bq[pk(mr, m)] = A[pk(r, c)];
        mr++;
      }
      hb[m] = h[c];
      idb[m] = id[c];
      m++;
    }
    n = m;
    for (int q = 0; q < tri(n); q++) A[q] = Bq[q];
    for (int k = 0; k < n; k++) { h[k] = hb[k]; id[k] = idb[k]; }
  }
  // marginalize(h, J, g, keep, integrate) (beliefupdates.jl:48-83); returns 0 or the failing pivot
  PGBP_HD int marginalize(const bool* integ) {
    int ni = 0;
    for (int i = 0; i < n; i++) ni += integ[i] ? 1 : 0;
    if (ni == 0) return 0;
    bool allzero = true;
    for (int i = 0; i < n && allzero; i++) if (integ[i]) {
      if (!(fabs(h[i]) <= PGBP_EPS)) allzero = false;
      for (int j = 0; j < n; j++) if (!(fabs(a(i, j)) <= PGBP_EPS)) allzero = false;
    }
    if (allzero) { compact_keep(integ); return 0; }
    // permute to [I; K], then right-looking U'U over the first ni pivots (same update order as K2)
    int perm[PGBP_SCOPED_MAXN];
    int m = 0;
    for (int i = 0; i < n; i++) if (integ[i]) perm[m++] = i;
    for (int i = 0; i < n; i++) if (!integ[i]) perm[m++] = i;
    for (int c = 0; c < n; c++) {
      for (int r = 0; r <= c; r++) Bq[pk(r, c)] = a(perm[r], perm[c]);
      hb[c] = h[perm[c]];
      idb[c] = id[perm[c]];
    }
    double logdet = 0.0, ww = 0.0;
    for (int k = 0; k < ni; k++) {
      const double d = Bq[pk(k, k)];
      if (!(d > 0.0)) return k + 1;
      logdet += log(d);
      const double rinv = 1.0 / sqrt(d);
      for (int c = k + 1; c < n; c++) Bq[pk(k, c)] *= rinv;
      const double wk = hb[k] * rinv;
      ww = fma(wk, wk, ww);
      for (int c = k + 1; c < n; c++) {
        const double akc = Bq[pk(k, c)];
        for (int r = k + 1; r <= c; r++) Bq[pk(r, c)] = fma(-Bq[pk(k, r)], akc, Bq[pk(r, c)]);
        hb[c] = fma(-akc, wk, hb[c]);
      }
    }
    g += 0.5 * ((double)ni * PGBP_LOG2PI - logdet + ww);
    const int nk = n - ni;
    for (int c = 0; c < nk; c++) {
      for (int r = 0; r <= c; r++) A[pk(r, c)] = Bq[pk(ni + r, ni + c)];
      h[c] = hb[ni + c];
      id[c] = idb[ni + c];
    }
    n = nk;
    return 0;
  }
};

struct AssignScoped {
  AssignBody gen;
  const int32_t* mem_tpos;     // [#members * p]
  const uint8_t* tip_missing;  // [ntips * p]
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const { run(e, y + y0); }
  PGBP_HD void run(int64_t e, int c) const {
    const FamDev& F = gen.F;
    const ThetaRows& tr = gen.tr;
    const int p = F.p, pp = p * p;
    const int64_t ld = gen.ld, ldp = gen.ldp, ldd = gen.ldd;
    int64_t ip, idd;
    if (gen.pairing == PGBP_PAIR_PRODUCT) { ip = e / gen.nd; idd = e % gen.nd; }
    else { ip = gen.np == 1 ? 0 : e; idd = gen.nd == 1 ? 0 : e; }
    const double* th = gen.theta + ip;
    const double* td = gen.tip + idd;
    double* st = gen.state + e;
    const bool lead = gen.gs == 0;
    const int64_t js = F.cl_jslot[c], hs = F.cl_hslot[c], gsl = F.cl_gslot[c];
    const int m = F.cl_dim[c];
    if (lead) for (int q = 0; q < tri(m); q++) st[(js + q) * ld] = 0.0;
    for (int q = 0; q < m; q++) st[(hs + q) * ld] = 0.0;
    double g = 0.0;
    const double kind = th[(int64_t)tr.kind() * ldp];
    if (kind < 0.0) {
      if (c == 0) status_fail(gen.status, e, PGBP_STATUS(0x7ffffd, (int)(-kind)));
      st[gsl * ld] = NAN;
      return;
    }
    double j[PGBP_MAX_TRAITS * PGBP_MAX_TRAITS], w[PGBP_MAX_TRAITS * PGBP_MAX_TRAITS];
    ScopedFactor f;
    bool sel[PGBP_SCOPED_MAXN];
    double val[PGBP_SCOPED_MAXN];
    for (int iv = F.clu_off[c]; iv < F.clu_off[c + 1]; iv++) {
      const int v = F.clu_node[iv];
      const int k0 = F.mem_off[v], nm = F.mem_off[v + 1] - k0;
      f.n = nm * p;
      for (int i = 0; i < f.n; i++) { f.h[i] = 0.0; f.id[i] = (int16_t)i; }
      if (nm == 1) {  // root family (src/beliefs.jl:803-807)
        if (F.mem_pos[k0] < 0 || kind != 1.0) continue;  // fixed root, or improper prior: factor == 1
        for (int cc = 0; cc < p; cc++) {
          for (int r = 0; r <= cc; r++) f.A[pk(r, cc)] = th[(int64_t)(tr.rootP() + cc * p + r) * ldp];
          f.h[cc] = th[(int64_t)(tr.rooth() + cc) * ldp];
        }
        f.g = th[(int64_t)tr.rootg() * ldp];
      } else {
        bool samecolor = true;
        for (int k = k0 + 2; k < k0 + nm; k++) if (F.mem_color[k] != F.mem_color[k0 + 1]) samecolor = false;
        if (samecolor) {
          const int col = F.mem_color[k0 + 1];
          double t0 = 0.0;
          if (nm == 2) t0 = F.mem_length[k0 + 1];
          else for (int k = k0 + 1; k < k0 + nm; k++) t0 += F.mem_gamma[k] * F.mem_gamma[k] * F.mem_length[k];
          for (int q = 0; q < pp; q++) j[q] = th[(int64_t)(tr.P(col) + q) * ldp] / t0;
          f.g = th[(int64_t)tr.g0(col) * ldp] - 0.5 * p * log(t0);
        } else {
          for (int q = 0; q < pp; q++) w[q] = 0.0;
          for (int k = k0 + 1; k < k0 + nm; k++) {
            const double fk = F.mem_gamma[k] * F.mem_gamma[k] * F.mem_length[k];
            const int col = F.mem_color[k];
            for (int q = 0; q < pp; q++) w[q] += fk * th[(int64_t)(tr.R(col) + q) * ldp];
          }
          double ldv;
          const int info = spd_inverse_logdet(w, j, p, &ldv);
          if (info) { status_fail(gen.status, e, PGBP_STATUS(0x7ffffc, info)); st[gsl * ld] = NAN; return; }
          f.g = -0.5 * (p * PGBP_LOG2PI + ldv);
        }
        for (int b2 = 0; b2 < nm; b2++) {
          const double cb = b2 == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + b2]);
          for (int a2 = 0; a2 <= b2; a2++) {
            const double ca = a2 == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + a2]);
            const double cab = ca * cb;
            for (int tb = 0; tb < p; tb++)
              for (int ta = 0; ta < (a2 == b2 ? tb + 1 : p); ta++) f.A[pk(a2 * p + ta, b2 * p + tb)] = cab * j[tb * p + ta];
          }
        }
        // absorbleaf!: observed traits of the leaf, then its missing traits
        const int row = F.node_datarow[v];
        const bool child_fixed = F.mem_pos[k0] < 0;
        if (child_fixed && row >= 0) {
          bool anymiss = false;
          for (int i = 0; i < f.n; i++) { sel[i] = false; val[i] = 0.0; }
          for (int t = 0; t < p; t++) {
            if (tip_missing[row * p + t]) { anymiss = true; continue; }
            sel[t] = true;
            val[t] = td[(int64_t)(row * p + t) * ldd];
            if (val[t] != val[t]) status_fail(gen.status, e, PGBP_STATUS(0x7ffffa, t + 1));
          }
          f.absorb(sel, val);
          if (anymiss) {
            for (int i = 0; i < f.n; i++) sel[i] = f.id[i] < p;
            const int info = f.marginalize(sel);
            if (info) { status_fail(gen.status, e, PGBP_STATUS(0x7ffff9, info)); st[gsl * ld] = NAN; return; }
          }
        }
        // a fixed root among the parents: clamp it to the prior mean (src/beliefs.jl:828-831)
        bool anyroot = false;
        for (int i = 0; i < f.n; i++) {
          const int a2 = f.id[i] / p, t = f.id[i] % p;
          sel[i] = a2 >= 1 && F.mem_pos[k0 + a2] < 0;
          val[i] = sel[i] ? th[(int64_t)(tr.mu() + t) * ldp] : 0.0;
          anyroot = anyroot || sel[i];
        }
        if (anyroot) f.absorb(sel, val);
      }
      // out-of-scope traits (src/beliefs.jl:836-857): child first, then parents.  A parent's out-of-scope
      // trait t is observed below none of its children, so the child's trait t is gone by stage 1 (stage 0 or
      // absorbleaf!); under Brownian motion the child's other traits do not depend on the parents' trait t, and
      // its rows of (h, J) are zero in exact arithmetic.  Stage 1 drops them: the reference marginalises them,
      // which factorises their roundoff (~1e-14 on short edges) and adds ~ -log(1e-14)/2 per trait to g, or
      // fails on a negative pivot.
      for (int stage = 0; stage < 2; stage++) {
        bool any = false;
        for (int i = 0; i < f.n; i++) {
          const int a2 = f.id[i] / p, t = f.id[i] % p;
          sel[i] = ((stage == 0) == (a2 == 0)) && mem_tpos[(k0 + a2) * p + t] < 0;
          any = any || sel[i];
        }
        if (!any) continue;
        if (stage == 1) { f.compact_keep(sel); continue; }
        const int info = f.marginalize(sel);
        if (info) { status_fail(gen.status, e, PGBP_STATUS(0x7ffff9, info)); st[gsl * ld] = NAN; return; }
      }
      // mult! (src/beliefs.jl:858)
      g += f.g;
      for (int cc = 0; cc < f.n; cc++) {
        const int pc = mem_tpos[(k0 + f.id[cc] / p) * p + f.id[cc] % p];
        st[(hs + pc) * ld] += f.h[cc];
        if (lead) for (int r = 0; r <= cc; r++) {
          const int pr = mem_tpos[(k0 + f.id[r] / p) * p + f.id[r] % p];
          st[(js + (pr <= pc ? pk(pr, pc) : pk(pc, pr))) * ld] += f.A[pk(r, cc)];
        }
      }
    }
    st[gsl * ld] = g;
  }
};

// K1 write-once path, compile-time trait count P.  The precision j of one family lives in
// registers (P*P doubles).  Families of the cluster are applied in node order, like the loop at
// src/beliefs.jl:798-859; the host has marked, for every family, which of its (member, member)
// blocks and h segments it is the FIRST to touch inside its cluster (first_J / first_h): those are
// written with a plain store (0 + x, the value the reference's zero-then-add produces), later
// families add into them.  Only clusters with scope entries that no family covers are zero-filled
// first (flag bit 0).  No thread-local arrays except for heterogeneous hybrids whose parent edges
// differ in colour (a p x p inverse per element, src/evomodels/heterogeneousmodels.jl:135-150).
// K1 for the univariate Ornstein-Uhlenbeck model (src/evomodels/homogeneousornsteinuhlenbeck.jl:51-66) -- and,
// through it, the generic linear-Gaussian factor X_v ~ N(sum_k gamma_k (q_k x_k + omega_k), sum_k gamma_k^2 v_k)
// of src/evomodels/evomodels.jl:208-245, 314-330 for one trait:
//   q_k = exp(-alpha t_k), v_k = gamma2 (1 - q_k^2), omega_k = (1 - q_k) theta,  gamma2 = sigma2 / (2 alpha).
// With c = (1, -gamma_1 q_1, ..), z = sum over fixed members c_a y_a - omega:  J_ab += c_a c_b j,
// h_b -= c_b j z, g += g0 - j z^2 / 2, g0 = -(log 2pi + log v)/2  (the same absorbed form as the BM path).
// params: AoS records (sigma2, alpha, theta, mu, v);  v == 0 fixed root, v == Inf improper, else proper.
struct AssignOU {
  FamDev F;
  const double* params;  // [np][5]
  const double* tip;     // SoA [ntips][ldd]
  int64_t ldd;
  double* state;
  int32_t* status;
  int64_t ld, np, nd;
  int pairing;
  int64_t gs = 0;
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const {
    const int c = y + y0;
    int64_t ip, id;
    if (pairing == PGBP_PAIR_PRODUCT) { ip = e / nd; id = e % nd; }
    else { ip = np == 1 ? 0 : e; id = nd == 1 ? 0 : e; }
    const double* th = params + 5 * ip;
    const double sigma2 = th[0], alpha = th[1], theta = th[2], mu = th[3], v = th[4];
    const double* td = tip + id;
    double* st = state + e;
    const bool lead = gs == 0;
    const int64_t js = F.cl_jslot[c], hs = F.cl_hslot[c], gsl = F.cl_gslot[c];
    const int m = F.cl_dim[c];
    if (lead) for (int q = 0; q < tri(m); q++) st[(js + q) * ld] = 0.0;
    for (int q = 0; q < m; q++) st[(hs + q) * ld] = 0.0;
    if (!(sigma2 > 0.0) || !(alpha > 0.0)) {  // the reference's constructor rejects these
      if (c == 0) status_fail(status, e, PGBP_STATUS(0x7ffffd, 1));
      st[gsl * ld] = NAN;
      return;
    }
    const double gamma2 = sigma2 / (2.0 * alpha);
    double g = 0.0;
    for (int iv = F.clu_off[c]; iv < F.clu_off[c + 1]; iv++) {
      const int vtx = F.clu_node[iv];
      const int k0 = F.mem_off[vtx], nm = F.mem_off[vtx + 1] - k0;
      if (nm == 1) {  // root prior, as for UnivariateBrownianMotion (src/evomodels/evomodels.jl:377-396)
        const int pos = F.mem_pos[k0];
        if (pos < 0 || v == 0.0 || v == INFINITY) continue;
        const double jr = 1.0 / v;
        if (lead) st[(js + pk(pos, pos)) * ld] += jr;
        st[(hs + pos) * ld] += jr * mu;
        g += 0.5 * (-PGBP_LOG2PI + log(jr) - mu * (jr * mu));
        continue;
      }
      double cf[PGBP_MAX_FAMILY];
      double var = 0.0, omega = 0.0;
      cf[0] = 1.0;
      for (int a = 1; a < nm; a++) {
        const double t = F.mem_length[k0 + a], gam = nm == 2 ? 1.0 : F.mem_gamma[k0 + a];
        const double q = exp(-alpha * t);
        var += gam * gam * (gamma2 * (1.0 - q * q));
        omega += gam * ((1.0 - q) * theta);
        cf[a] = -(gam * q);
      }
      const double j = 1.0 / var;
      double z = -omega;
      for (int a = 0; a < nm; a++) {
        if (F.mem_pos[k0 + a] >= 0) continue;
        z += cf[a] * (a == 0 ? td[(int64_t)F.node_datarow[vtx] * ldd] : mu);
      }
      if (z != z) status_fail(status, e, PGBP_STATUS(0x7ffffa, 1));  // missing tip value
      g += -0.5 * (PGBP_LOG2PI + log(var)) - 0.5 * (z * (j * z));
      for (int a = 0; a < nm; a++) {
        const int pa = F.mem_pos[k0 + a];
        if (pa < 0) continue;
        st[(hs + pa) * ld] -= cf[a] * (j * z);
        for (int bq = a; lead && bq < nm; bq++) {
          const int pb = F.mem_pos[k0 + bq];
          if (pb < 0) continue;
          st[(js + pk(pa, pb)) * ld] += (cf[a] * cf[bq]) * j;
        }
      }
    }
    st[gsl * ld] = g;
  }
};

PGBP_HD double* kaddr(char* base, uint32_t slot, uint32_t ld8) {
  return (double*)(base + (uint64_t)slot * (uint64_t)ld8);  // one IMAD.WIDE.U32
}

template <int P, bool SH = false>
struct AssignFast {
  AssignBody gen;
  const uint8_t* cflag;       // [nclusters] bit 0: zero-fill first
  const uint64_t* first_J;    // [nnodes] bit a*8+b: family v is the first writer of block (a, b), a <= b
  const uint8_t* first_h;     // [nnodes] bit a: first writer of member a's h segment
  // Shared-precision batches: the family precision block j, its log-normaliser and the failure code depend on the
  // group's parameters only.  The group pass (SH = false on the group batch, jucache != null) STORES them per
  // (family, group): [v][P(P+1)/2 + 2][G]; the element pass (SH = true) READS them instead of recomputing a
  // P x P block per element (at P = 16 that block lived in thread-local memory).
  double* jucache = nullptr;
  int64_t juG = 0;
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const {
    const int c = y + y0;
    const FamDev& F = gen.F;
    const ThetaRows& tr = gen.tr;
    const int64_t ldp = gen.ldp, ld = gen.ld, ldd = gen.ldd;
    int64_t ip, id;
    if (gen.pairing == PGBP_PAIR_PRODUCT) { ip = e / gen.nd; id = e % gen.nd; }
    else { ip = gen.np == 1 ? 0 : e; id = gen.nd == 1 ? 0 : e; }
    const double* th = gen.theta + ip;
    const double* td = gen.tip + id;
    double* st = gen.state + e;
    const bool lead = !SH;  // SH: element side of a shared-precision batch (h and g only)
    const int64_t js = F.cl_jslot[c], hs = F.cl_hslot[c], gs = F.cl_gslot[c];
    const double kind = th[(int64_t)tr.kind() * ldp];
    if (kind < 0.0) { gen.run(e, c); return; }  // invalid parameters: generic path records the status
    if (cflag[c] & 1) {
      const int m = F.cl_dim[c];
      if (lead) for (int q = 0; q < tri(m); q++) st[(js + q) * ld] = 0.0;
      for (int q = 0; q < m; q++) st[(hs + q) * ld] = 0.0;
    }
    double g = 0.0;
    for (int iv = F.clu_off[c]; iv < F.clu_off[c + 1]; iv++) {
      const int v = F.clu_node[iv];
      const int k0 = F.mem_off[v], nm = F.mem_off[v + 1] - k0;
      const uint64_t fJ = first_J[v];
      const unsigned fh = first_h[v];
      if (nm == 1) {  // root family (src/beliefs.jl:803-807)
        const int pos = F.mem_pos[k0];
        if (pos < 0) continue;
        const bool proper = kind == 1.0;  // fixed root handled by pos < 0; improper prior: factor == 1
#pragma unroll
        for (int cc = 0; cc < P; cc++) {
#pragma unroll
          for (int r = 0; lead && r <= cc; r++) {
            const double x = proper ? th[(int64_t)(tr.rootP() + cc * P + r) * ldp] : 0.0;
            double* d = st + (js + pk(pos + r, pos + cc)) * ld;
            if (fJ & 1) *d = 0.0 + x;
            else if (proper) *d += x;
          }
          const double xh = proper ? th[(int64_t)(tr.rooth() + cc) * ldp] : 0.0;
          double* dh = st + (hs + pos + cc) * ld;
          if (fh & 1) *dh = 0.0 + xh;
          else if (proper) *dh += xh;
        }
        if (proper) g += th[(int64_t)tr.rootg() * ldp];
        continue;
      }
      // precision block j (symmetric: upper triangle kept, 36 registers at P = 8) and log-normaliser
      constexpr int NJ = P * (P + 1) / 2;
      double ju[SH ? 1 : NJ];  // (element pass of a shared-precision batch: the block is read from the cache, never built)
      double* juc = jucache ? jucache + (int64_t)v * (NJ + 2) * juG + (SH ? e / gen.gs : e) : nullptr;
      const int64_t jus = juG;  // stride between the entries of one cached block
#define PGBP_JU(r_, c_) (SH ? juc[(int64_t)((r_) <= (c_) ? pk((r_), (c_)) : pk((c_), (r_))) * jus] \
                            : ju[SH ? 0 : ((r_) <= (c_) ? pk((r_), (c_)) : pk((c_), (r_)))])
      double gv;
      if constexpr (SH) {  // element pass of a shared-precision batch: the group pass left j, g0 and the failure code
        const double info = juc[(int64_t)(NJ + 1) * jus];
        if (info != 0.0) { status_fail(gen.status, e, PGBP_STATUS(0x7ffffc, (int)info)); st[gs * ld] = NAN; return; }
        gv = juc[(int64_t)NJ * jus];
      } else {
      bool samecolor = true;
      for (int k = k0 + 2; k < k0 + nm; k++) if (F.mem_color[k] != F.mem_color[k0 + 1]) samecolor = false;
      if (samecolor) {
        const int col = F.mem_color[k0 + 1];
        double t0 = 0.0;
        if (nm == 2) t0 = F.mem_length[k0 + 1];
        else for (int k = k0 + 1; k < k0 + nm; k++) t0 += F.mem_gamma[k] * F.mem_gamma[k] * F.mem_length[k];
        // x / t0 for 36 values with one divisor: r = RN(1/t0), q0 = x r, q = q0 + r (x - t0 q0)
        // (Markstein: correctly rounded quotient from a correctly rounded reciprocal), 3 FMA-class
        // operations per entry instead of a ~20-instruction division sequence
        const double rt = 1.0 / t0;
#pragma unroll
        for (int cc = 0; cc < P; cc++) {
#pragma unroll
          for (int r = 0; r <= cc; r++) {
            const double x = th[(int64_t)(tr.P(col) + cc * P + r) * ldp];
            const double q0 = x * rt;
            ju[pk(r, cc)] = fma(fma(-t0, q0, x), rt, q0);
          }
        }
        gv = th[(int64_t)tr.g0(col) * ldp] - 0.5 * P * log(t0);
      } else {  // heterogeneous hybrid: j = (sum gamma^2 t R_c)^-1
        double w[P * P], jl[P * P];
        for (int q = 0; q < P * P; q++) w[q] = 0.0;
        for (int k = k0 + 1; k < k0 + nm; k++) {
          const double f = F.mem_gamma[k] * F.mem_gamma[k] * F.mem_length[k];
          const int col = F.mem_color[k];
          for (int q = 0; q < P * P; q++) w[q] += f * th[(int64_t)(tr.R(col) + q) * ldp];
        }
        double ldv;
        const int info = spd_inverse_logdet(w, jl, P, &ldv);
        if (info) {
          if (!SH && juc) juc[(int64_t)(NJ + 1) * jus] = (double)info;
          status_fail(gen.status, e, PGBP_STATUS(0x7ffffc, info)); st[gs * ld] = NAN; return;
        }
#pragma unroll
        for (int cc = 0; cc < P; cc++) {
#pragma unroll
          for (int r = 0; r <= cc; r++) ju[pk(r, cc)] = jl[cc * P + r];
        }
        gv = -0.5 * (P * PGBP_LOG2PI + ldv);
      }
      if (!SH && juc) {  // group pass: leave the block for the element pass
#pragma unroll
        for (int q = 0; q < NJ; q++) juc[(int64_t)q * jus] = ju[q];
        juc[(int64_t)NJ * jus] = gv;
        juc[(int64_t)(NJ + 1) * jus] = 0.0;
      }
      }
      if constexpr (SH) {
        // Tip family (the node itself observed, its one parent free) on the element side of a shared-precision batch:
        // the same operations as the general code below, row by row -- j z is consumed as it is produced instead of
        // living in an array next to z and sixteen loads in flight (ncu on C5: the 96-register kernel spilled 66
        // local stores per warp, and those, not the h rows, were half of its DRAM writes)
        if (nm == 2 && F.mem_pos[k0] < 0 && F.mem_pos[k0 + 1] >= 0) {
          const int row = F.node_datarow[v];
          const int pa = F.mem_pos[k0 + 1];
          const bool first = (fh >> 1) & 1;
          double z[P];
#pragma unroll
          for (int t = 0; t < P; t++) z[t] = 0.0 + 1.0 * td[(int64_t)(row * P + t) * ldd];
#pragma unroll
          for (int t = 0; t < P; t++) if (z[t] != z[t]) status_fail(gen.status, e, PGBP_STATUS(0x7ffffa, t + 1));
          const uint32_t ld8 = (uint32_t)(ld * 8);
          char* stb = (char*)st;
          double quad = 0.0;
#pragma unroll
          for (int r = 0; r < P; r++) {
            double s = 0.0;
#pragma unroll
            for (int cc = 0; cc < P; cc++) s += PGBP_JU(r, cc) * z[cc];
            quad += z[r] * s;
            double* dh = kaddr(stb, (uint32_t)(hs + pa + r), ld8);
            if (first) *dh = 0.0 - (-1.0) * s;
            else *dh = *dh - (-1.0) * s;
#if defined(__CUDA_ARCH__)
            asm volatile("" ::: "memory");  // keep the loads of row r + 1 behind the store of row r
#endif
          }
          gv -= 0.5 * quad;
          g += gv;
          continue;
        }
      }
      if constexpr (SH) {
        // Family without evidence (every member free: the internal nodes, half of a big network's clusters): the h
        // segments this family writes first are zero, nothing else moves on the element side.  Same stores as the
        // general code below, without its z / j z arrays.
        bool nofixed = true;
        for (int a = 0; a < nm; a++) if (F.mem_pos[k0 + a] < 0) nofixed = false;
        if (nofixed) {
          g += gv;
          const uint32_t ld8 = (uint32_t)(ld * 8);
          char* stb = (char*)st;
          for (int a = 0; a < nm; a++) {
            if (!((fh >> a) & 1)) continue;
            const int pa = F.mem_pos[k0 + a];
#pragma unroll
            for (int t = 0; t < P; t++) *kaddr(stb, (uint32_t)(hs + pa + t), ld8) = 0.0;
          }
          continue;
        }
      }
      // evidence: z = sum over fixed members of c_a * value_a
      bool anyfixed = false;
      double z[P], jz[P];
#pragma unroll
      for (int t = 0; t < P; t++) { z[t] = 0.0; jz[t] = 0.0; }
      for (int a = 0; a < nm; a++) {
        if (F.mem_pos[k0 + a] >= 0) continue;
        anyfixed = true;
        const double ca = a == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + a]);
        if (a == 0) {
          const int row = F.node_datarow[v];
#pragma unroll
          for (int t = 0; t < P; t++) z[t] += ca * td[(int64_t)(row * P + t) * ldd];
        } else {
#pragma unroll
          for (int t = 0; t < P; t++) z[t] += ca * th[(int64_t)(tr.mu() + t) * ldp];
        }
      }
      if (anyfixed) {
#pragma unroll
        for (int t = 0; t < P; t++) if (z[t] != z[t]) status_fail(gen.status, e, PGBP_STATUS(0x7ffffa, t + 1));
        double quad = 0.0;
#pragma unroll
        for (int r = 0; r < P; r++) {
          double s = 0.0;
#pragma unroll
          for (int cc = 0; cc < P; cc++) s += PGBP_JU(r, cc) * z[cc];
          jz[r] = s;
          quad += z[r] * s;
        }
        gv -= 0.5 * quad;
      }
      g += gv;
      const uint32_t ld8 = (uint32_t)(ld * 8);
      char* stb = (char*)st;
      for (int a = 0; a < nm; a++) {
        const int pa = F.mem_pos[k0 + a];
        if (pa < 0) continue;
        const double ca = a == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + a]);
        if ((fh >> a) & 1) {
#pragma unroll
          for (int t = 0; t < P; t++) *kaddr(stb, (uint32_t)(hs + pa + t), ld8) = anyfixed ? 0.0 - ca * jz[t] : 0.0;
        } else if (anyfixed) {
          double oldh[P];
#pragma unroll
          for (int t = 0; t < P; t++) oldh[t] = *kaddr(stb, (uint32_t)(hs + pa + t), ld8);
#pragma unroll
          for (int t = 0; t < P; t++) *kaddr(stb, (uint32_t)(hs + pa + t), ld8) = oldh[t] - ca * jz[t];
        }
        for (int bq = a; lead && bq < nm; bq++) {
          const int pb = F.mem_pos[k0 + bq];
          if (pb < 0) continue;
          const double cb = bq == 0 ? 1.0 : (nm == 2 ? -1.0 : -F.mem_gamma[k0 + bq]);
          const double cab = ca * cb;
          const bool diag = bq == a;
          const bool first = (fJ >> (a * 8 + bq)) & 1;
          if (first) {
#pragma unroll
            for (int tb = 0; tb < P; tb++) {
              const uint32_t colslot = (uint32_t)js + (uint32_t)tri(pb + tb) + (uint32_t)pa;  // pk(pa + ta, pb + tb)
#pragma unroll
              for (int ta = 0; ta < P; ta++)
                if (!diag || ta <= tb) *kaddr(stb, colslot + ta, ld8) = cab * PGBP_JU(ta, tb);
            }
          } else {
            // read-modify-write of a block another family wrote first: the P loads of a column are issued
            // together, then the adds and stores (a load cannot be hoisted above a store the compiler cannot
            // disambiguate: entry-by-entry "+=" exposed one L2 round trip per entry, 60 % long_sb in ncu)
#pragma unroll
            for (int tb = 0; tb < P; tb++) {
              const uint32_t colslot = (uint32_t)js + (uint32_t)tri(pb + tb) + (uint32_t)pa;
              double old[P];
#pragma unroll
              for (int ta = 0; ta < P; ta++)
                if (!diag || ta <= tb) old[ta] = *kaddr(stb, colslot + ta, ld8);
#pragma unroll
              for (int ta = 0; ta < P; ta++)
                if (!diag || ta <= tb) *kaddr(stb, colslot + ta, ld8) = old[ta] + cab * PGBP_JU(ta, tb);
            }
          }
        }
      }
#undef PGBP_JU
    }
    st[gs * ld] = g;
  }
};

// --------------------------------------------------------------------------
// K4: factored energy (src/score.jl:162-182)
// --------------------------------------------------------------------------
template <int MAXM>
struct EnergyClusterBody {
  const double* state;
  const double* factor;
  int32_t* status;
  const int64_t* cl_jslot;
  const int64_t* cl_hslot;
  const int64_t* cl_gslot;
  const int32_t* cl_dim;
  const int32_t* list;  // clusters handled by this instantiation
  double* part;         // [2*nclusters + nsepsets][ld]: energy_c, entropy_c, entropy_s
  int nclusters;
  int64_t ld;
  JSide sj{nullptr, 0, 0}, fj{nullptr, 0, 0};  // shared-precision batches: J rows of beliefs / factors in the group batch
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const {
    const int c = list[y + y0];
    const int M = cl_dim[c];
    const double* st = state + e;
    const double* fa = factor + e;
    const double* stj = sj.base ? jcolumn(sj, e) : st;
    const double* faj = fj.base ? jcolumn(fj, e) : fa;
    const int64_t ldj = sj.base ? sj.ld : ld;
    const int64_t js = cl_jslot[c], hs = cl_hslot[c], gs = cl_gslot[c];
    const double gf = fa[gs * ld];
    if (M == 0) {  // src/score.jl:170-171
      part[(int64_t)c * ld + e] = -gf;
      part[(int64_t)(nclusters + c) * ld + e] = 0.0;
      return;
    }
    constexpr int NA = MAXM * (MAXM + 1) / 2;
    double A[NA], mu[MAXM], x[MAXM];
    const int SM = tri(M);
    for (int q = 0; q < SM; q++) A[q] = stj[(js + q) * ldj];
    for (int k = 0; k < M; k++) mu[k] = st[(hs + k) * ld];
    double logdet = 0.0;
    for (int k = 0; k < M; k++) {  // U'U = J_b; forward solve w = U^-T h
      const double d = A[pk(k, k)];
      if (!(d > 0.0)) {
        status_fail(status, e, PGBP_STATUS(0x7ffffb, k + 1));
        part[(int64_t)c * ld + e] = NAN;
        part[(int64_t)(nclusters + c) * ld + e] = NAN;
        return;
      }
      logdet += log(d);
      const double rinv = 1.0 / sqrt(d);
      A[pk(k, k)] = rinv;  // store 1/U_kk
      for (int cc = k + 1; cc < M; cc++) A[pk(k, cc)] *= rinv;
      mu[k] *= rinv;
      for (int cc = k + 1; cc < M; cc++) {
        const double akc = A[pk(k, cc)];
        for (int r = k + 1; r <= cc; r++) A[pk(r, cc)] = nfma(A[pk(k, r)], akc, A[pk(r, cc)]);
        mu[cc] = nfma(akc, mu[k], mu[cc]);
      }
    }
    for (int k = M - 1; k >= 0; k--) {  // U mu = w
      double s = mu[k];
      for (int cc = k + 1; cc < M; cc++) s = nfma(A[pk(k, cc)], mu[cc], s);
      mu[k] = s * A[pk(k, k)];
    }
    // tr(J_b^-1 J_f) = sum_k |U^-T f_k|^2-weighted ... computed as sum_k e_k' U^-1 U^-T J_f e_k:
    // for each column k of J_f solve U' x = f_k, U y = x, take y_k.
    double trace = 0.0, quad = 0.0, hfmu = 0.0;
    for (int k = 0; k < M; k++) {
      double fk_mu = 0.0;
      for (int r = 0; r < M; r++) {
        const double f = faj[(js + (r <= k ? pk(r, k) : pk(k, r))) * ldj];
        x[r] = f;
        fk_mu = fma(f, mu[r], fk_mu);
      }
      quad += mu[k] * fk_mu;
      for (int r = 0; r < M; r++) {  // U' x = f_k
        double s = x[r];
        for (int q = 0; q < r; q++) s = nfma(A[pk(q, r)], x[q], s);
        x[r] = s * A[pk(r, r)];
      }
      for (int r = M - 1; r >= k; r--) {  // U y = x, only down to row k
        double s = x[r];
        for (int q = r + 1; q < M; q++) s = nfma(A[pk(r, q)], x[q], s);
        x[r] = s * A[pk(r, r)];
      }
      trace += x[k];
      hfmu += fa[(hs + k) * ld] * mu[k];
    }
    part[(int64_t)c * ld + e] = 0.5 * (trace + quad) - hfmu - gf;               // average_energy, :114-117
    part[(int64_t)(nclusters + c) * ld + e] = 0.5 * (M * (PGBP_LOG2PI + 1.0) - logdet);  // entropy, :58-62
  }
};

template <int MAXM>
struct EntropySepsetBody {
  const double* state;
  const int64_t* jslot;  // per belief
  const int32_t* dim;
  const int32_t* list;
  double* part;
  int nclusters;
  int64_t ld;
  JSide sj{nullptr, 0, 0};
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const {
    const int j = list[y + y0];
    const int M = dim[nclusters + j];
    double* out = part + (int64_t)(2 * nclusters + j) * ld + e;
    if (M == 0) { *out = 0.0; return; }
    constexpr int NA = MAXM * (MAXM + 1) / 2;
    double A[NA];
    const double* st = sj.base ? jcolumn(sj, e) : state + e;
    const int64_t ldj = sj.base ? sj.ld : ld;
    const int64_t js = jslot[nclusters + j];
    for (int q = 0; q < tri(M); q++) A[q] = st[(js + q) * ldj];
    double logdet = 0.0;
    for (int k = 0; k < M; k++) {
      const double d = A[pk(k, k)];
      if (!(d > 0.0)) {  // logdet(Symmetric(J)) of a singular / indefinite sepset (src/score.jl:66)
        logdet = (d == 0.0) ? -INFINITY : NAN;
        break;
      }
      logdet += log(d);
      const double rinv = 1.0 / sqrt(d);
      for (int cc = k + 1; cc < M; cc++) A[pk(k, cc)] *= rinv;
      for (int cc = k + 1; cc < M; cc++) {
        const double akc = A[pk(k, cc)];
        for (int r = k + 1; r <= cc; r++) A[pk(r, cc)] = nfma(A[pk(k, r)], akc, A[pk(r, cc)]);
      }
    }
    *out = 0.5 * (M * (PGBP_LOG2PI + 1.0) - logdet);
  }
};

struct EnergyReduceBody {
  const double* part;
  double* out;  // SoA [3][ldo]
  int nclusters, nsepsets;
  int64_t ld, ldo;
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int) const {
    double en = 0.0, ent = 0.0;
    for (int c = 0; c < nclusters; c++) en += part[(int64_t)c * ld + e];
    for (int c = 0; c < nclusters; c++) ent += part[(int64_t)(nclusters + c) * ld + e];
    for (int j = 0; j < nsepsets; j++) ent -= part[(int64_t)(2 * nclusters + j) * ld + e];
    out[e] = en;
    out[ldo + e] = ent;
    out[2 * ldo + e] = -(en - ent);  // factored_energy = -free_energy, src/score.jl:151-154
  }
};

// --------------------------------------------------------------------------
// K5: regularisation
// --------------------------------------------------------------------------
PGBP_HD double maxabs_packed(const double* st, int64_t js, int M, int64_t ld) {
  double mx = 0.0;
  for (int q = 0; q < tri(M); q++) absmax(mx, st[(js + q) * ld]);
  return mx;
}

// by cluster, step A: eps_c = max(eps, max|J_c|) once, then bump the cluster's
// diagonal once per incident sepset variable (src/clustergraphbeliefs.jl:240-249, 264-273)
struct RegClusterBody {
  double* state;
  double* eps;  // [nclusters][ld]
  const int64_t* jslot;
  const int32_t* dim;
  const int32_t* reg_off;
  const int32_t* reg_pos;
  int64_t ld;
  double floor_eps;
  int64_t gs = 0;  // shared-precision mode: only group leaders own J rows
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const {
    if (gs > 1 && e % gs) return;
    const int c = y + y0;
    double* st = state + e;
    const int64_t js = jslot[c];
    double ep = maxabs_packed(st, js, dim[c], ld);
    if (!(ep >= floor_eps)) ep = (ep != ep) ? ep : floor_eps;
    eps[(int64_t)c * ld + e] = ep;
    for (int k = reg_off[c]; k < reg_off[c + 1]; k++) {
      const int u = reg_pos[k];
      st[(js + pk(u, u)) * ld] += ep;
    }
  }
};
// by cluster, step B: sepset diagonal += eps of its two clusters, in cluster order
struct RegSepsetBody {
  double* state;
  const double* eps;
  const int64_t* jslot;
  const int32_t* dim;
  const int32_t* sep_a;
  const int32_t* sep_b;
  int nclusters;
  int64_t ld;
  int64_t gs = 0;  // shared-precision mode: only group leaders own J rows
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int y) const {
    if (gs > 1 && e % gs) return;
    const int j = y + y0;
    const int M = dim[nclusters + j];
    if (M == 0) return;
    const int a = sep_a[j] < sep_b[j] ? sep_a[j] : sep_b[j];
    const int b2 = sep_a[j] < sep_b[j] ? sep_b[j] : sep_a[j];
    const double e1 = eps[(int64_t)a * ld + e], e2 = eps[(int64_t)b2 * ld + e];
    double* st = state + e;
    const int64_t js = jslot[nclusters + j];
    for (int k = 0; k < M; k++) {
      double* d = st + (js + pk(k, k)) * ld;
      *d = (*d + e1) + e2;
    }
  }
};

// on schedule: eps of one cluster (src/clustergraphbeliefs.jl:386)
struct EpsOneBody {
  const double* state;
  double* eps;  // [ld]
  int64_t js, ld;
  int M;
  double floor_eps;
  int64_t gs = 0;  // shared-precision mode: only group leaders own J rows
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int) const {
    if (gs > 1 && e % gs) return;
    double ep = maxabs_packed(state + e, js, M, ld);
    if (!(ep >= floor_eps)) ep = (ep != ep) ? ep : floor_eps;
    eps[e] = ep;
  }
};
// regularizebeliefs_1clustersepset! with a per-element eps (:264-275)
struct RegOneBody {
  double* state;
  const double* eps;
  const int32_t* upind;  // device table: cluster positions of the sepset's variables
  int64_t cjs, sjs, ld;
  int S;
  int64_t gs = 0;  // shared-precision mode: only group leaders own J rows
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int) const {
    if (gs > 1 && e % gs) return;
    double* st = state + e;
    const double ep = eps[e];
    for (int k = 0; k < S; k++) {
      const int u = upind[k];
      st[(cjs + pk(u, u)) * ld] += ep;
      st[(sjs + pk(k, k)) * ld] += ep;
    }
  }
};

// by node subtree: one launch per network node (src/clustergraphbeliefs.jl:314-340)
struct RegNodeBody {
  double* state;
  const int64_t* jslot;
  const int32_t* dim;
  const int32_t *eps_cluster, *step_off, *step_cluster, *step_sepset, *idx_off, *idx_cluster, *idx_sepset;
  int e0, e1, s0, s1;  // ranges of this node in eps_cluster / steps
  int nclusters;
  int64_t ld;
  int64_t gs = 0;  // shared-precision mode: only group leaders own J rows
  int y0 = 0;
  PGBP_HD void operator()(int64_t e, int) const {
    if (gs > 1 && e % gs) return;
    double* st = state + e;
    double ep = PGBP_EPS;
    for (int k = e0; k < e1; k++) {
      const int c = eps_cluster[k];
      const double m = maxabs_packed(st, jslot[c], dim[c], ld);
      if (m > ep || m != m) ep = m;
    }
    for (int s = s0; s < s1; s++) {
      const int64_t cj = jslot[step_cluster[s]], sj = jslot[nclusters + step_sepset[s]];
      for (int k = idx_off[s]; k < idx_off[s + 1]; k++) {
        const int uc = idx_cluster[k], us = idx_sepset[k];
        st[(cj + pk(uc, uc)) * ld] += ep;
        st[(sj + pk(us, us)) * ld] += ep;
      }
    }
  }
};

// --------------------------------------------------------------------------
// device copies of plan tables, built lazily per batch
// --------------------------------------------------------------------------
struct DevTables {
  int64_t* jslot = nullptr;  // per belief
  int64_t* hslot = nullptr;
  int64_t* gslot = nullptr;
  int32_t* dim = nullptr;
  int32_t *sep_a = nullptr, *sep_b = nullptr;
  int32_t *reg_off = nullptr, *reg_pos = nullptr;
  // families
  int32_t *node_cluster = nullptr, *mem_off = nullptr, *mem_pos = nullptr, *mem_color = nullptr,
          *node_datarow = nullptr, *clu_off = nullptr, *clu_node = nullptr;
  uint8_t* clu_flag = nullptr;
  uint64_t* first_J = nullptr;
  uint8_t* first_h = nullptr;
  double *mem_length = nullptr, *mem_gamma = nullptr;
  int32_t* mem_tpos = nullptr;    // trait-level scopes (scoped plans only)
  uint8_t* tip_missing = nullptr;
  // parameter / data staging
  double* theta = nullptr;
  int64_t theta_rows = 0, ldp = 0;
  double* tip = nullptr;
  int64_t tip_rows = 0, ldd = 0;
  std::vector<void*> owned;
};

template <class T>
static int upload(pgbp_batch* b, DevTables* dt, T** dst, const std::vector<T>& src) {
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, std::max<size_t>(1, src.size()) * sizeof(T)));
  dt->owned.push_back(v);
  *dst = (T*)v;
  b->device_bytes += (int64_t)(src.size() * sizeof(T));
  return h2d(v, src.data(), src.size() * sizeof(T), b->stream);
}

static int get_tables(pgbp_batch* b, DevTables** out) {
  if (b->d_fam) { *out = (DevTables*)b->d_fam; return 0; }
  const pgbp_plan* p = b->plan;
  std::unique_ptr<DevTables> dt(new DevTables);
  PGBP_TRY(upload(b, dt.get(), &dt->jslot, p->jslot));
  if (b->jb) {  // shared-precision batch: the element array holds h and g only, in compact rows
    std::vector<int64_t> hr(p->nbeliefs), gr(p->nbeliefs);
    for (int i = 0; i < p->nbeliefs; i++) { hr[i] = batch_hrow(b, i); gr[i] = batch_grow(b, i); }
    PGBP_TRY(upload(b, dt.get(), &dt->hslot, hr));
    PGBP_TRY(upload(b, dt.get(), &dt->gslot, gr));
  } else {
    PGBP_TRY(upload(b, dt.get(), &dt->hslot, p->hslot));
    PGBP_TRY(upload(b, dt.get(), &dt->gslot, p->gslot));
  }
  PGBP_TRY(upload(b, dt.get(), &dt->dim, p->dim));
  PGBP_TRY(upload(b, dt.get(), &dt->sep_a, p->sep_a));
  PGBP_TRY(upload(b, dt.get(), &dt->sep_b, p->sep_b));
  std::vector<int32_t> ro(1, 0), rp;
  for (int c = 0; c < p->nclusters; c++) {
    for (auto& nb : p->nbrs[c]) {  // neighbor_labels order
      const int j = nb.second;
      const std::vector<int32_t>& up = (p->sep_a[j] == c) ? p->up_a[j] : p->up_b[j];
      rp.insert(rp.end(), up.begin(), up.end());
    }
    ro.push_back((int32_t)rp.size());
  }
  PGBP_TRY(upload(b, dt.get(), &dt->reg_off, ro));
  PGBP_TRY(upload(b, dt.get(), &dt->reg_pos, rp));
  if (p->has_families) {
    const FamilyTable& F = p->fam;
    PGBP_TRY(upload(b, dt.get(), &dt->node_cluster, F.node_cluster));
    PGBP_TRY(upload(b, dt.get(), &dt->mem_off, F.mem_off));
    PGBP_TRY(upload(b, dt.get(), &dt->mem_pos, F.mem_pos));
    if (F.scoped) {
      PGBP_TRY(upload(b, dt.get(), &dt->mem_tpos, F.mem_tpos));
      PGBP_TRY(upload(b, dt.get(), &dt->tip_missing, F.tip_missing));
    }
    PGBP_TRY(upload(b, dt.get(), &dt->mem_color, F.mem_color));
    PGBP_TRY(upload(b, dt.get(), &dt->node_datarow, F.node_datarow));
    PGBP_TRY(upload(b, dt.get(), &dt->clu_off, F.clu_off));
    PGBP_TRY(upload(b, dt.get(), &dt->clu_node, F.clu_node));
    PGBP_TRY(upload(b, dt.get(), &dt->mem_length, F.mem_length));
    PGBP_TRY(upload(b, dt.get(), &dt->mem_gamma, F.mem_gamma));
    PGBP_TRY(upload(b, dt.get(), &dt->clu_flag, F.clu_flag));
    PGBP_TRY(upload(b, dt.get(), &dt->first_J, F.first_J));
    PGBP_TRY(upload(b, dt.get(), &dt->first_h, F.first_h));
  }
  PGBP_TRY(stream_sync(b->stream));
  b->d_fam = dt.release();
  *out = (DevTables*)b->d_fam;
  return 0;
}

void free_tables(pgbp_batch* b) {
  DevTables* dt = (DevTables*)b->d_fam;
  if (!dt) return;
  for (void* v : dt->owned) dev_free(v);
  dev_free(dt->theta);
  dev_free(dt->tip);
  delete dt;
  b->d_fam = nullptr;
}

static int ensure_rows(pgbp_batch* b, double** arr, int64_t* rows_have, int64_t* ld_have, int64_t rows, int64_t n) {
  const int64_t ld = (n + 31) / 32 * 32;
  if (*arr && *rows_have >= rows && *ld_have == ld) return 0;
  PGBP_TRY(stream_sync(b->stream));
  dev_free(*arr);
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, sizeof(double) * (size_t)rows * (size_t)ld));
  *arr = (double*)v;
  *rows_have = rows;
  *ld_have = ld;
  return 0;
}

template <int MAXM>
static int launch_energy_bucket(pgbp_batch* b, DevTables* dt, const std::vector<int32_t>& cl, const std::vector<int32_t>& sp,
                                double* part, int32_t* d_list) {
  const pgbp_plan* p = b->plan;
  if (!cl.empty()) {
    PGBP_TRY(h2d(d_list, cl.data(), cl.size() * sizeof(int32_t), b->stream));
    EnergyClusterBody<MAXM> body{b->state, b->factor, b->status, dt->jslot, dt->hslot, dt->gslot, dt->dim, d_list,
                                 part, p->nclusters, b->ld};
    if (b->jb) {
      body.sj = batch_jside(b);
      body.fj = JSide{b->jb->factor, b->jb->ld, b->group_size};
    }
    PGBP_TRY(launch_generic(b, "k_energy_cluster", b->B, (int)cl.size(), body));
  }
  if (!sp.empty()) {
    int32_t* d_list2 = d_list + p->nclusters;
    PGBP_TRY(h2d(d_list2, sp.data(), sp.size() * sizeof(int32_t), b->stream));
    EntropySepsetBody<MAXM> body{b->state, dt->jslot, dt->dim, d_list2, part, p->nclusters, b->ld};
    if (b->jb) body.sj = batch_jside(b);
    PGBP_TRY(launch_generic(b, "k_entropy_sepset", b->B, (int)sp.size(), body));
  }
  return 0;
}

static int factored_energy_launch(pgbp_batch* b, double* d_out_soa, int64_t ldo) {
  const pgbp_plan* p = b->plan;
  PGBP_TRY(batch_materialize_sepsets(b));
  if (!b->factor) PGBP_FAIL(PGBP_ESTATE, "batch was created without PGBP_BATCH_FACTORS");
  PGBP_TRY(batch_materialize_factors(b));
  if (b->jb) {  // the J rows of beliefs and factors are read from the group batch
    b->jb->stream = b->stream;
    PGBP_TRY(batch_materialize_sepsets(b->jb));
    PGBP_TRY(batch_materialize_factors(b->jb));
  }
  DevTables* dt;
  PGBP_TRY(get_tables(b, &dt));
  const size_t nrows = 2 * (size_t)p->nclusters + p->nsepsets;
  const size_t part_bytes = sizeof(double) * nrows * (size_t)b->ld;
  const size_t list_bytes = sizeof(int32_t) * (size_t)(p->nclusters + p->nsepsets) * 4;
  PGBP_TRY(batch_need_scratch(b, part_bytes + list_bytes + 3 * sizeof(double) * (size_t)b->ld));
  double* part = b->scratch;
  int32_t* d_list = (int32_t*)((char*)b->scratch + part_bytes);
  // bucket clusters / sepsets by dimension so small ones use small local arrays
  const int caps[4] = {4, 12, 32, PGBP_MAX_DIM};
  std::vector<int32_t> cl[4], sp[4];
  auto bucket = [&](int m) { for (int k = 0; k < 4; k++) if (m <= caps[k]) return k; return 3; };
  for (int c = 0; c < p->nclusters; c++) cl[bucket(p->dim[c])].push_back(c);
  for (int j = 0; j < p->nsepsets; j++) sp[bucket(p->dim[p->nclusters + j])].push_back(j);
  const int stride = p->nclusters + p->nsepsets;
  PGBP_TRY(launch_energy_bucket<4>(b, dt, cl[0], sp[0], part, d_list));
  PGBP_TRY(launch_energy_bucket<12>(b, dt, cl[1], sp[1], part, d_list + stride));
  PGBP_TRY(launch_energy_bucket<32>(b, dt, cl[2], sp[2], part, d_list + 2 * stride));
  PGBP_TRY(launch_energy_bucket<PGBP_MAX_DIM>(b, dt, cl[3], sp[3], part, d_list + 3 * stride));
  PGBP_TRY(stream_sync(b->stream));  // host lists are temporaries
  EnergyReduceBody red{part, d_out_soa, p->nclusters, p->nsepsets, b->ld, ldo};
  return launch_generic(b, "k_energy_reduce", b->B, 1, red);
}

}  // namespace pgbp

extern "C" {

// shared argument checks + table / staging setup of the two assign_factors entry points
static int assign_prepare(pgbp_batch* b, int32_t ncolors, int64_t nparamsets, int64_t ndatasets, int32_t pairing,
                          pgbp::DevTables** dt_out) {
  const pgbp_plan* p = b->plan;
  if (!p->has_families) PGBP_FAIL(PGBP_ESTATE, "the plan has no node-family table");
  const FamilyTable& F = p->fam;
  const int pt = p->ntraits;
  if (pt > PGBP_MAX_TRAITS) PGBP_FAIL(PGBP_EINVAL, "ntraits %d > %d", pt, PGBP_MAX_TRAITS);
  if (ncolors < F.ncolors_min) PGBP_FAIL(PGBP_EINVAL, "ncolors %d but the family table uses colour %d", ncolors, F.ncolors_min - 1);
  const int64_t B = b->B;
  if (pairing == PGBP_PAIR_PRODUCT) {
    if (nparamsets * ndatasets != B) PGBP_FAIL(PGBP_EINVAL, "product pairing needs nparamsets*ndatasets == B");
  } else if (pairing == PGBP_PAIR_ZIP) {
    if ((nparamsets != 1 && nparamsets != B) || (ndatasets != 1 && ndatasets != B))
      PGBP_FAIL(PGBP_EINVAL, "zip pairing needs nparamsets, ndatasets in {1, B}");
  } else PGBP_FAIL(PGBP_EINVAL, "unknown pairing %d", pairing);
  if (b->group_size > 1) {  // shared-precision mode: the elements of a group must use one parameter vector
    const bool ok = (pairing == PGBP_PAIR_ZIP && nparamsets == 1) ||
                    (pairing == PGBP_PAIR_PRODUCT && ndatasets % b->group_size == 0);
    if (!ok) PGBP_FAIL(PGBP_EINVAL, "shared-precision batch: every group of %lld elements needs a single parameter vector "
                       "(zip with 1 parameter set, or product with ndatasets a multiple of the group size)", (long long)b->group_size);
  }
  PGBP_TRY(set_device(b->device));
  b->lazy_factors.pending = false;  // the tables a pending snapshot would be recomputed from are about to change
  b->lazy_factors.valid = false;
  DevTables* dt;
  PGBP_TRY(get_tables(b, &dt));
  ThetaRows tr{pt, ncolors};
  PGBP_TRY(ensure_rows(b, &dt->theta, &dt->theta_rows, &dt->ldp, tr.nrows(), nparamsets));
  const int64_t tiprows = (int64_t)F.ntips * pt;
  PGBP_TRY(ensure_rows(b, &dt->tip, &dt->tip_rows, &dt->ldd, std::max<int64_t>(1, tiprows), ndatasets));
  *dt_out = dt;
  return 0;
}

static int assign_launch(pgbp_batch* b, pgbp::DevTables* dt, double* out, int32_t ncolors, int64_t nparamsets,
                         int64_t ndatasets, int32_t pairing);

// K1 proper, everything on the device, enqueue only: d_params / d_tip are the AoS records of the header
static int assign_enqueue(pgbp_batch* b, pgbp::DevTables* dt, int32_t ncolors, const double* d_params, int64_t nparamsets,
                          const double* d_tip, int64_t ndatasets, int32_t pairing) {
  const pgbp_plan* p = b->plan;
  const FamilyTable& F = p->fam;
  const int pt = p->ntraits;
  ThetaRows tr{pt, ncolors};
  ThetaPrep prep{d_params, dt->theta, dt->ldp, tr};
  PGBP_TRY(launch_generic(b, "k_theta_prep", nparamsets, 1, prep));
  const int64_t tiprows = (int64_t)F.ntips * pt;
  if (tiprows > 0) {  // tip data AoS [nd][ntips*p] -> SoA [ntips*p][ldd]
    const int64_t saveB = b->B;
    b->B = ndatasets;  // transpose over the data-set axis
    int rc = aos_to_soa(b, d_tip, (int)tiprows, nullptr, dt->tip, dt->ldd);
    b->B = saveB;
    PGBP_TRY(rc);
  }
  if (b->jb) {
    // shared-precision batch: the J rows are assigned once per group in the group batch, from the same prepared
    // tables (group g = elements [g gs, (g+1) gs): its parameter set, any of its data sets -- J does not depend on
    // the data); that pass also leaves the family precision blocks for the element pass, which writes h and g
    pgbp_batch* jb = b->jb;
    jb->stream = b->stream;
    jb->jparent = b;
    DevTables* jdt;
    PGBP_TRY(get_tables(jb, &jdt));
    const int64_t jnd = pairing == PGBP_PAIR_PRODUCT ? ndatasets / b->group_size : 1;
    std::swap(jdt->theta, dt->theta); std::swap(jdt->ldp, dt->ldp); std::swap(jdt->tip, dt->tip); std::swap(jdt->ldd, dt->ldd);
    const int rc = assign_launch(jb, jdt, jb->state, ncolors, nparamsets, jnd, pairing);
    std::swap(jdt->theta, dt->theta); std::swap(jdt->ldp, dt->ldp); std::swap(jdt->tip, dt->tip); std::swap(jdt->ldd, dt->ldd);
    PGBP_TRY(rc);
    jb->lazy_factors.pending = false;
    jb->lazy_factors.valid = false;
    PGBP_TRY(assign_launch(b, dt, b->state, ncolors, nparamsets, ndatasets, pairing));
    PGBP_TRY(batch_zero_sepsets(b, true));  // lazily: the first postorder traversal treats the sepsets as 0
    if (b->factor) {
      PGBP_TRY(d2d(jb->factor, jb->state, sizeof(double) * (size_t)p->nslots_factor * (size_t)jb->ld, b->stream));
      PGBP_TRY(d2d(b->factor, b->state, sizeof(double) * (size_t)b->nrows_efactor * (size_t)b->ld, b->stream));
    }
    return 0;
  }
  PGBP_TRY(assign_launch(b, dt, b->state, ncolors, nparamsets, ndatasets, pairing));
  // sepsets <- 0 (src/beliefs.jl:796), lazily; factor snapshot (src/clustergraphbeliefs.jl:106), lazily
  PGBP_TRY(batch_zero_sepsets(b, true));
  if (b->factor) b->lazy_factors = pgbp_batch::LazyFactors{true, true, ncolors, nparamsets, ndatasets, pairing};
  return 0;
}

// the K1 kernel: cluster beliefs (J, h, g) from the prepared tables dt->theta / dt->tip, written to `out`
// (the state array, or the factor array when a lazy snapshot is materialised: same layout)
static int assign_launch(pgbp_batch* b, pgbp::DevTables* dt, double* out, int32_t ncolors, int64_t nparamsets,
                         int64_t ndatasets, int32_t pairing) {
  const pgbp_plan* p = b->plan;
  const FamilyTable& F = p->fam;
  const int pt = p->ntraits;
  ThetaRows tr{pt, ncolors};
  FamDev fd{dt->node_cluster, dt->mem_off, dt->mem_pos, dt->mem_length, dt->mem_gamma, dt->mem_color,
            dt->node_datarow, dt->clu_off, dt->clu_node, dt->jslot, dt->hslot, dt->gslot, dt->dim,
            pt, ncolors, F.root_fixed};
  AssignBody body{fd, dt->theta, dt->ldp, dt->tip, dt->ldd, out, b->status, b->ld, nparamsets, ndatasets, pairing, tr};
  body.gs = b->group_size;
  if (F.scoped)  // trait-level scopes (missing data): the reference's absorb / marginalise sequence
    return launch_generic(b, "k_assign_scoped", b->B, p->nclusters, AssignScoped{body, dt->mem_tpos, dt->tip_missing});
  // shared-precision batches: cache of the family precision blocks, written by the group pass (this function called
  // on the group batch: b->jparent set) and read by the element pass (b->jb set)
  double* juc = nullptr;
  int64_t juG = 0;
  {
    pgbp_batch* owner = b->jb ? b : b->jparent;
    if (owner && out == b->state) {
      const size_t need = (size_t)F.nnodes * (size_t)(pt * (pt + 1) / 2 + 2) * (size_t)owner->ngroups;
      if (owner->jucache_len < need) {
        PGBP_TRY(stream_sync(b->stream));
        dev_free(owner->jucache);
        owner->jucache = nullptr; owner->jucache_len = 0;
        void* v = nullptr;
        PGBP_TRY(dev_malloc(&v, need * sizeof(double)));
        owner->jucache = (double*)v;
        owner->jucache_len = need;
        owner->device_bytes += (int64_t)(need * sizeof(double));
      }
      juc = owner->jucache;
      juG = owner->ngroups;
    }
  }
  switch (pt) {
#define PGBP_FAST_CASE(P_) \
  case P_: \
    if (b->group_size > 1) PGBP_TRY((launch_generic<AssignFast<P_, true>, 5>(b, "k_assign_factors", b->B, p->nclusters, AssignFast<P_, true>{body, dt->clu_flag, dt->first_J, dt->first_h, juc, juG}))); \
    else PGBP_TRY((launch_generic<AssignFast<P_>, 3>(b, "k_assign_factors", b->B, p->nclusters, AssignFast<P_>{body, dt->clu_flag, dt->first_J, dt->first_h, juc, juG}))); \
    break;
    PGBP_FAST_CASE(1) PGBP_FAST_CASE(2) PGBP_FAST_CASE(3) PGBP_FAST_CASE(4) PGBP_FAST_CASE(5) PGBP_FAST_CASE(6)
    PGBP_FAST_CASE(7) PGBP_FAST_CASE(8)
    // p = 16 (C5): the family precision (136 doubles) no longer fits the register file and lives in
    // thread-local memory (L1-resident), which still beats the generic body's global read-modify-write
    PGBP_FAST_CASE(12) PGBP_FAST_CASE(16)
#undef PGBP_FAST_CASE
    default: PGBP_TRY(launch_generic(b, "k_assign_factors", b->B, p->nclusters, body));
  }
  return 0;
}

}  // extern "C"
namespace pgbp {
int batch_materialize_factors(pgbp_batch* b) {
  if (!b->lazy_factors.pending) return 0;
  if (!b->factor) { b->lazy_factors.pending = false; return 0; }
  DevTables* dt;
  PGBP_TRY(get_tables(b, &dt));
  const pgbp_batch::LazyFactors lf = b->lazy_factors;
  PGBP_TRY(assign_launch(b, dt, b->factor, lf.ncolors, lf.nparamsets, lf.ndatasets, lf.pairing));
  b->lazy_factors.pending = false;
  return 0;
}
int batch_reset_by_assign(pgbp_batch* b) {
  if (!b->lazy_factors.valid) return 0;
  if (b->plan->fam.scoped) return 0;  // the scoped (missing-data) K1 is a slow thread-local path: copy instead
  DevTables* dt;
  PGBP_TRY(get_tables(b, &dt));
  const pgbp_batch::LazyFactors lf = b->lazy_factors;
  int rc = assign_launch(b, dt, b->state, lf.ncolors, lf.nparamsets, lf.ndatasets, lf.pairing);
  return rc ? rc : 1;
}
}  // namespace pgbp
extern "C" {

int32_t pgbp_assign_factors_ou(pgbp_batch* b, const double* params, int64_t nparamsets, const double* tipdata,
                               int64_t ndatasets, int32_t pairing) {
  if (!b || !params) PGBP_FAIL(PGBP_EINVAL, "null argument");
  if (b->plan->ntraits != 1) PGBP_FAIL(PGBP_EINVAL, "the Ornstein-Uhlenbeck model of the reference is univariate");
  if (b->plan->has_families && b->plan->fam.ntips > 0 && !tipdata) PGBP_FAIL(PGBP_EINVAL, "null tip data");
  pgbp::DevTables* dt;
  PGBP_TRY(assign_prepare(b, 1, nparamsets, ndatasets, pairing, &dt));
  const pgbp_plan* p = b->plan;
  const FamilyTable& F = p->fam;
  const size_t nparam = (size_t)(5 * nparamsets), ntip = (size_t)((int64_t)F.ntips * ndatasets);
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (nparam + ntip + 1)));
  PGBP_TRY(h2d(b->scratch, params, sizeof(double) * nparam, b->stream));
  if (ntip) {
    PGBP_TRY(h2d(b->scratch + nparam, tipdata, sizeof(double) * ntip, b->stream));
    const int64_t saveB = b->B;
    b->B = ndatasets;
    int rc = aos_to_soa(b, b->scratch + nparam, F.ntips, nullptr, dt->tip, dt->ldd);
    b->B = saveB;
    PGBP_TRY(rc);
  }
  FamDev fd{dt->node_cluster, dt->mem_off, dt->mem_pos, dt->mem_length, dt->mem_gamma, dt->mem_color,
            dt->node_datarow, dt->clu_off, dt->clu_node, dt->jslot, dt->hslot, dt->gslot, dt->dim, 1, 1, F.root_fixed};
  AssignOU body{fd, b->scratch, dt->tip, dt->ldd, b->state, b->status, b->ld, nparamsets, ndatasets, pairing};
  body.gs = b->group_size;
  PGBP_TRY(launch_generic(b, "k_assign_ou", b->B, p->nclusters, body));
  b->lazy_factors.pending = false;  // (the OU parameters live in scratch memory: eager snapshot)
  b->lazy_factors.valid = false;
  if (b->jb) {  // shared-precision batch: J rows once per group in the group batch (see assign_enqueue)
    pgbp_batch* jb = b->jb;
    jb->stream = b->stream;
    DevTables* jdt;
    PGBP_TRY(get_tables(jb, &jdt));
    FamDev jfd{jdt->node_cluster, jdt->mem_off, jdt->mem_pos, jdt->mem_length, jdt->mem_gamma, jdt->mem_color,
               jdt->node_datarow, jdt->clu_off, jdt->clu_node, jdt->jslot, jdt->hslot, jdt->gslot, jdt->dim, 1, 1, F.root_fixed};
    const int64_t jnd = pairing == PGBP_PAIR_PRODUCT ? ndatasets / b->group_size : 1;
    AssignOU jbody{jfd, b->scratch, dt->tip, dt->ldd, jb->state, jb->status, jb->ld, nparamsets, jnd, pairing};
    PGBP_TRY(launch_generic(jb, "k_assign_ou", jb->B, p->nclusters, jbody));
    jb->lazy_factors.pending = false;
    jb->lazy_factors.valid = false;
    PGBP_TRY(batch_zero_sepsets(b, false));
    if (b->factor) {
      PGBP_TRY(d2d(jb->factor, jb->state, sizeof(double) * (size_t)p->nslots_factor * (size_t)jb->ld, b->stream));
      PGBP_TRY(d2d(b->factor, b->state, sizeof(double) * (size_t)b->nrows_efactor * (size_t)b->ld, b->stream));
    }
    return stream_sync(b->stream);
  }
  PGBP_TRY(batch_zero_sepsets(b, true));
  if (b->factor) PGBP_TRY(d2d(b->factor, b->state, sizeof(double) * (size_t)p->nslots_factor * (size_t)b->ld, b->stream));
  return stream_sync(b->stream);
}

int32_t pgbp_assign_factors_device(pgbp_batch* b, int32_t ncolors, const double* d_params, int64_t nparamsets,
                                   const double* d_tipdata, int64_t ndatasets, int32_t pairing) {
  if (!b || !d_params) PGBP_FAIL(PGBP_EINVAL, "null argument");
  if (b->plan->has_families && b->plan->fam.ntips > 0 && !d_tipdata) PGBP_FAIL(PGBP_EINVAL, "null tip data");
  pgbp::DevTables* dt;
  PGBP_TRY(assign_prepare(b, ncolors, nparamsets, ndatasets, pairing, &dt));
  return assign_enqueue(b, dt, ncolors, d_params, nparamsets, d_tipdata, ndatasets, pairing);
}

int32_t pgbp_assign_factors(pgbp_batch* b, int32_t ncolors, const double* params, int64_t nparamsets,
                            const double* tipdata, int64_t ndatasets, int32_t pairing) {
  if (!b || !params) PGBP_FAIL(PGBP_EINVAL, "null argument");
  if (b->plan->has_families && b->plan->fam.ntips > 0 && !tipdata) PGBP_FAIL(PGBP_EINVAL, "null tip data");
  pgbp::DevTables* dt;
  PGBP_TRY(assign_prepare(b, ncolors, nparamsets, ndatasets, pairing, &dt));
  const pgbp_plan* p = b->plan;
  const int pt = p->ntraits;
  const int64_t plen = (int64_t)ncolors * pt * pt + pt + (int64_t)pt * pt;
  const int64_t tiprows = (int64_t)p->fam.ntips * pt;
  const size_t nparam = (size_t)(plen * nparamsets), ntip = (size_t)(tiprows * ndatasets);
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (nparam + ntip)));
  PGBP_TRY(h2d(b->scratch, params, sizeof(double) * nparam, b->stream));
  if (ntip) PGBP_TRY(h2d(b->scratch + nparam, tipdata, sizeof(double) * ntip, b->stream));
  PGBP_TRY(assign_enqueue(b, dt, ncolors, b->scratch, nparamsets, b->scratch + nparam, ndatasets, pairing));
  return stream_sync(b->stream);
}

int32_t pgbp_factored_energy_device(pgbp_batch* b, double* d_out_soa) {
  if (!b || !d_out_soa) PGBP_FAIL(PGBP_EINVAL, "null argument");
  PGBP_TRY(set_device(b->device));
  return factored_energy_launch(b, d_out_soa, b->ld);
}

int32_t pgbp_factored_energy(pgbp_batch* b, double* out) {
  if (!b || !out) PGBP_FAIL(PGBP_EINVAL, "null argument");
  PGBP_TRY(set_device(b->device));
  const pgbp_plan* p = b->plan;
  // output rows live behind the partial sums in the scratch buffer
  const size_t nrows = 2 * (size_t)p->nclusters + p->nsepsets;
  const size_t part_bytes = sizeof(double) * nrows * (size_t)b->ld;
  const size_t list_bytes = sizeof(int32_t) * (size_t)(p->nclusters + p->nsepsets) * 4;
  const size_t off = (part_bytes + list_bytes + 7) / 8 * 8;
  PGBP_TRY(batch_need_scratch(b, off + 6 * sizeof(double) * (size_t)b->ld));
  double* d_soa = (double*)((char*)b->scratch + off);
  PGBP_TRY(factored_energy_launch(b, d_soa, b->ld));
  double* d_aos = d_soa + 3 * b->ld;
  PGBP_TRY(soa_to_aos(b, d_soa, b->ld, d_aos, 3, nullptr));
  double* pin = (double*)batch_pinned(b, sizeof(double) * 3 * (size_t)b->B);  // results through pinned memory
  PGBP_TRY(d2h(pin ? pin : out, d_aos, sizeof(double) * 3 * (size_t)b->B, b->stream));
  PGBP_TRY(stream_sync(b->stream));
  if (pin) memcpy(out, pin, sizeof(double) * 3 * (size_t)b->B);
  return 0;
}

int32_t pgbp_regularize_bycluster(pgbp_batch* b) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  PGBP_TRY(set_device(b->device));
  if (b->jb) {  // the regularisers only touch J: the group batch's
    b->jb->stream = b->stream;
    PGBP_TRY(batch_materialize_sepsets(b));
    return pgbp_regularize_bycluster(b->jb);
  }
  PGBP_TRY(batch_materialize_sepsets(b));
  const pgbp_plan* p = b->plan;
  DevTables* dt;
  PGBP_TRY(get_tables(b, &dt));
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (size_t)p->nclusters * (size_t)b->ld));
  RegClusterBody a{b->state, b->scratch, dt->jslot, dt->dim, dt->reg_off, dt->reg_pos, b->ld, PGBP_EPS};
  PGBP_TRY(launch_generic(b, "k_reg_cluster", b->B, p->nclusters, a));
  RegSepsetBody s{b->state, b->scratch, dt->jslot, dt->dim, dt->sep_a, dt->sep_b, p->nclusters, b->ld};
  return launch_generic(b, "k_reg_sepset", b->B, p->nsepsets, s);
}

int32_t pgbp_regularize_onschedule(pgbp_batch* b) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  PGBP_TRY(set_device(b->device));
  PGBP_TRY(batch_materialize_sepsets(b));
  const pgbp_plan* p = b->plan;
  DevTables* dt;
  PGBP_TRY(get_tables(b, &dt));
  // the op list of src/clustergraphbeliefs.jl:376-403
  struct Op { int kind, c, j, nb; };
  std::vector<Op> ops;
  std::set<std::pair<int, int>> sent;  // (from, to)
  std::vector<MsgDesc> msgs;
  std::vector<int32_t> uptab;
  std::vector<int32_t> upoff;
  for (int c = 0; c < p->nclusters; c++) {
    ops.push_back({0, c, 0, 0});
    std::vector<Op> tosend;
    for (auto& nbj : p->nbrs[c]) {
      const int nb = nbj.first, j = nbj.second;
      if (!sent.count({nb, c})) {
        ops.push_back({1, c, j, (int)upoff.size()});
        const std::vector<int32_t>& up = (p->sep_a[j] == c) ? p->up_a[j] : p->up_b[j];
        upoff.push_back((int32_t)uptab.size());
        uptab.insert(uptab.end(), up.begin(), up.end());
        sent.insert({nb, c});
      }
      if (!sent.count({c, nb})) {
        tosend.push_back({2, c, j, nb});
        sent.insert({c, nb});
      }
    }
    for (auto& o : tosend) {
      MsgDesc md;
      PGBP_TRY(p->make_msg(o.c, o.j, o.nb, &md));
      md.ref = (int32_t)msgs.size();
      ops.push_back({2, o.c, o.j, (int)msgs.size()});
      msgs.push_back(md);
    }
  }
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, std::max<size_t>(1, msgs.size()) * sizeof(MsgDesc)));
  MsgDesc* d_msgs = (MsgDesc*)v;
  PGBP_TRY(dev_malloc(&v, std::max<size_t>(1, uptab.size()) * sizeof(int32_t)));
  int32_t* d_up = (int32_t*)v;
  int rc = h2d(d_msgs, msgs.data(), msgs.size() * sizeof(MsgDesc), b->stream);
  if (!rc) rc = h2d(d_up, uptab.data(), uptab.size() * sizeof(int32_t), b->stream);
  // eps and the diagonal bumps only touch J: on a shared-precision batch they run on the group batch
  pgbp_batch* jt = b->jb ? b->jb : b;
  if (b->jb) { jt->stream = b->stream; if (!rc) rc = batch_materialize_sepsets(jt); }
  if (!rc) rc = batch_need_scratch(jt, sizeof(double) * (size_t)jt->ld);
  const double eps0 = sqrt(PGBP_EPS);
  for (size_t k = 0; k < ops.size() && !rc; k++) {
    const Op& o = ops[k];
    if (o.kind == 0) {
      EpsOneBody body{jt->state, jt->scratch, p->jslot[o.c], jt->ld, p->dim[o.c], eps0};
      rc = launch_generic(jt, "k_eps_one", jt->B, 1, body);
    } else if (o.kind == 1) {
      const int S = p->dim[p->nclusters + o.j];
      if (S == 0) continue;  // isempty(upind) && return
      RegOneBody body{jt->state, jt->scratch, d_up + upoff[o.nb], p->jslot[o.c], p->jslot[p->nclusters + o.j], jt->ld, S};
      rc = launch_generic(jt, "k_reg_one", jt->B, 1, body);
    } else if (b->jb) {
      rc = shared_propagate(b, msgs[o.nb], 0, 0x3ffff0);  // residual stored, flags untouched (:400)
    } else {
      const MsgDesc& md = msgs[o.nb];
      LaunchGroup g;
      g.step = 0; g.first = o.nb; g.count = 1;
      shape_class(md.mF - md.s, md.s, &g.ci, &g.cs, &g.maxm);
      MsgArgs a = make_args(b, 0, 0x3ffff0, false);  // residual stored, flags untouched (:400)
      rc = launch_group(b, a, d_msgs, g);
    }
  }
  if (!rc) rc = stream_sync(b->stream);
  dev_free(d_msgs);
  dev_free(d_up);
  return rc;
}

int32_t pgbp_regularize_bynodesubtree(pgbp_batch* b, int32_t nnodes, const int32_t* eps_off, const int32_t* eps_cluster,
                                      const int32_t* step_off, const int32_t* step_cluster, const int32_t* step_sepset,
                                      const int32_t* idx_off, const int32_t* idx_cluster, const int32_t* idx_sepset) {
  if (!b || nnodes < 0 || !eps_off || !step_off) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  PGBP_TRY(set_device(b->device));
  if (b->jb) {  // J only: the group batch's
    b->jb->stream = b->stream;
    PGBP_TRY(batch_materialize_sepsets(b));
    return pgbp_regularize_bynodesubtree(b->jb, nnodes, eps_off, eps_cluster, step_off, step_cluster, step_sepset, idx_off,
                                         idx_cluster, idx_sepset);
  }
  PGBP_TRY(batch_materialize_sepsets(b));
  const pgbp_plan* p = b->plan;
  DevTables* dt;
  PGBP_TRY(get_tables(b, &dt));
  const int ne = eps_off[nnodes], ns = step_off[nnodes];
  const int ni = ns ? idx_off[ns] : 0;
  for (int k = 0; k < ne; k++) if (eps_cluster[k] < 0 || eps_cluster[k] >= p->nclusters) PGBP_FAIL(PGBP_EINVAL, "eps_cluster out of range");
  for (int s = 0; s < ns; s++) {
    if (step_cluster[s] < 0 || step_cluster[s] >= p->nclusters || step_sepset[s] < 0 || step_sepset[s] >= p->nsepsets)
      PGBP_FAIL(PGBP_EINVAL, "step %d out of range", s);
    for (int k = idx_off[s]; k < idx_off[s + 1]; k++)
      if (idx_cluster[k] < 0 || idx_cluster[k] >= p->dim[step_cluster[s]] || idx_sepset[k] < 0 ||
          idx_sepset[k] >= p->dim[p->nclusters + step_sepset[s]])
        PGBP_FAIL(PGBP_EINVAL, "step %d: diagonal index out of range", s);
  }
  std::vector<int32_t> all;
  all.insert(all.end(), eps_cluster, eps_cluster + ne);
  const size_t o_sc = all.size(); all.insert(all.end(), step_cluster, step_cluster + ns);
  const size_t o_ss = all.size(); all.insert(all.end(), step_sepset, step_sepset + ns);
  const size_t o_io = all.size(); all.insert(all.end(), idx_off, idx_off + ns + 1);
  const size_t o_ic = all.size(); all.insert(all.end(), idx_cluster, idx_cluster + ni);
  const size_t o_is = all.size(); all.insert(all.end(), idx_sepset, idx_sepset + ni);
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, std::max<size_t>(1, all.size()) * sizeof(int32_t)));
  int32_t* d = (int32_t*)v;
  int rc = h2d(d, all.data(), all.size() * sizeof(int32_t), b->stream);
  for (int n = 0; n < nnodes && !rc; n++) {
    if (step_off[n + 1] == step_off[n]) continue;
    RegNodeBody body{b->state, dt->jslot, dt->dim, d, nullptr, d + o_sc, d + o_ss, d + o_io, d + o_ic, d + o_is,
                     eps_off[n], eps_off[n + 1], step_off[n], step_off[n + 1], p->nclusters, b->ld};
    rc = launch_generic(b, "k_reg_node", b->B, 1, body);
  }
  if (!rc) rc = stream_sync(b->stream);
  dev_free(d);
  return rc;
}

}  // extern "C"
