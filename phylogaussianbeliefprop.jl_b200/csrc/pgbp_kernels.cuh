// Per-thread bodies of the hot kernels.  One thread = one batch element of one
// message / belief.  All global accesses are `base[slot * ld + e]`: consecutive
// threads touch consecutive doubles (batch-innermost SoA), so every warp load
// or store is one fully coalesced 256-byte transaction.
#pragma once
#include <type_traits>
#include <utility>

#include "pgbp_internal.h"

namespace pgbp {

#define PGBP_LOG2PI 1.8378770664093454835606594728112
#define PGBP_EPS 2.220446049250313e-16

struct MsgArgs {
  const MsgDesc* msgs;
  const int32_t* tab;
  double* state;
  double* resid;     // may be null
  uint8_t* calflag;  // may be null
  int32_t* status;
  const uint8_t* done;  // may be null
  int64_t B, ld;     // elements [e0, B) are processed (e0 > 0: one chunk of a pipelined calibration)
  uint32_t opts;     // PGBP_CAL_RESIDNORM | PGBP_CAL_RESIDKLDIV | PGBP_OPT_SEPZERO
  int32_t ref_base;
  int64_t e0;
};

// NaN-propagating running maximum of |x| (Julia's maximum(abs, x))
PGBP_HD void absmax(double& m, double x) {
  const double a = fabs(x);
  if (a > m || a != a) m = a;
}

// c - a*b with ONE rounding.  The library is compiled with -fmad=false, so the
// only fused operations are the explicit ones: every kernel variant (register,
// generic, walk, cooperative) that applies the same per-entry update order gives
// bit-identical results.
PGBP_HD double nfma(double a, double b, double c) { return fma(-a, b, c); }

// compile-time loop: f(std::integral_constant<int, k>) for k = 0..N-1
template <class F, int... Is>
PGBP_HD void static_for_impl(F&& f, std::integer_sequence<int, Is...>) {
  (f(std::integral_constant<int, Is>{}), ...);
}
template <int N, class F>
PGBP_HD void static_for(F&& f) {
  static_for_impl(f, std::make_integer_sequence<int, (N > 0 ? N : 0)>{});
}
// column of packed index q (q = c(c+1)/2 + r, r <= c)
PGBP_HD constexpr int colof(int q) {
  int c = 0;
  while ((c + 1) * (c + 2) / 2 <= q) ++c;
  return c;
}

#ifndef PGBP_CHUNK
#define PGBP_CHUNK 8  // measured on B200: 12 / 16 entries per chunk are slower (DESIGN.md section 6)
#endif
// internal option bit: every sepset written by this traversal is known to be identically zero (first
// postorder traversal after factor assignment / reset): the old sepset value is not loaded, and the
// zero-fill of the sepsets is skipped by the caller.  x - 0.0 == x, so results are unchanged.
#define PGBP_OPT_SEPZERO 0x100u

// calibration flag of one residual (src/beliefs.jl:994-1003):
// max|dh|/sqrt(s) <= 1e-5 && max|dJ|/sqrt(s^2) <= 1e-5.  max_i(|x_i|/c) == (max_i|x_i|)/c
// exactly (division by c > 0 is monotone, so is rounding).
PGBP_HD void store_flag(const MsgArgs& a, int dmsg, int64_t e, int S, double maxJ, double maxh) {
  if ((a.opts & PGBP_CAL_RESIDNORM) && a.calflag) {
    const bool okh = S > 0 ? (maxh / sqrt((double)S) <= 1e-5) : true;
    const bool okJ = S > 0 ? (maxJ / (double)S <= 1e-5) : true;
    a.calflag[(int64_t)dmsg * a.ld + e] = (okh && okJ) ? 1 : 0;
  }
}

// slot k of this element: base + k * (8*ld); 32-bit slot x 32-bit pitch -> one IMAD.WIDE.U32
PGBP_HD double* slot_ptr(char* base, uint32_t slot, uint32_t ld8) {
  return (double*)(base + (uint64_t)slot * (uint64_t)ld8);
}

// Every slot row a register-class message (I, S) reads, numbered in one fixed order: sender J in gather order
// [FJ, FH), sender h in [I;K] order [FH, FG), sender g, receiver g, receiver J and h at the sepset's positions
// [TJ, TH) and [TH, SG), then the old sepset g, J and h [SG, N).  The sepset rows come last because they are not
// read under PGBP_OPT_SEPZERO: the staged kernel then stages the first SG rows only.
template <int I, int S>
struct T0Rows {
  static constexpr int M = I + S, SMM = M * (M + 1) / 2, SS = S * (S + 1) / 2;
  static constexpr int FJ = 0, FH = SMM, FG = SMM + M, TG = FG + 1, TJ = TG + 1, TH = TJ + SS, SG = TH + S,
                       SJ = SG + 1, SH = SJ + SS, N = SH + S;
  // slot of row n (in the unrolled body n is a compile-time constant and the branches fold away)
  static PGBP_HD uint32_t slot(const MsgDesc& md, const int32_t* __restrict__ gat, const int32_t* __restrict__ sca, int n) {
    if (n < FG) return (n < FH ? (uint32_t)md.fJ : (uint32_t)md.fh) + (uint32_t)gat[n];
    if (n == FG) return (uint32_t)md.fg;
    if (n == TG) return (uint32_t)md.tg;
    if (n < SG) return (n < TH ? (uint32_t)md.tJ : (uint32_t)md.th) + (uint32_t)sca[n - TJ];
    if (n == SG) return (uint32_t)md.sg;
    return n < SH ? (uint32_t)md.sJ + (uint32_t)(n - SJ) : (uint32_t)md.sh + (uint32_t)(n - SH);
  }
};

// Operand sources of message_body_t0: slot(n) is the slot of row n (T0Rows numbering), at(n, slot) its value for
// this element.  T0Global reads the state array (host emulation, k_walk); the staged kernel's source reads a tile
// staged in shared memory (pgbp_msg_t0.cuh), the tile walk's values loaded before the body runs (pgbp_message.cu).
template <int I, int S>
struct T0Global {
  const MsgDesc& md;
  const int32_t* __restrict__ gat;
  const int32_t* __restrict__ sca;
  char* st;
  uint32_t ld8;
  PGBP_HD uint32_t slot(int n) const { return T0Rows<I, S>::slot(md, gat, sca, n); }
  PGBP_HD double at(int, uint32_t s) const { return *slot_ptr(st, s, ld8); }
};

// Register-resident message kernel body, compile-time shape (I >= 1 integrated
// out, S kept).  marginalize (src/beliefupdates.jl:55-83) -> divide! (:579-587)
// -> mult! (:483-488) -> residual (:646-647) -> flag (src/beliefs.jl:994-1003).
//
// Only J_II (packed), J_IK and h_I stay in registers.  They are factorised in
// place (right-looking U'U on the I rows): afterwards AI holds U, Bm holds
// Z' = U^-T J_IK and hI holds w = U^-T h_I.  The kept block is then STREAMED in
// chunks of PGBP_CHUNK packed entries: the sender's J_KK entry, the sepset's old
// value and the receiver's old value are all loaded first (3*CHUNK independent
// loads in flight per thread), then  new = J_KK - z_r.z_c,  delta = new - old,
// and the three stores.  h and g follow the same pattern.  Operands come from src
// (T0Global, a staged tile or the tile walk's registers); results are stored to the state array at the
// destination rows of md (a MsgDesc, or the tile walk's TwDesc: same field names).
template <int CI, int CS, class Desc, class Src>
PGBP_HD void message_body_t0(const MsgArgs& a, const Desc& md, int64_t e, const Src& src) {
  constexpr int I = CI, S = CS, SI = I * (I + 1) / 2, SS = S * (S + 1) / 2;
  using R = T0Rows<I, S>;
  const uint32_t ld8 = (uint32_t)(a.ld * 8);  // (batches with 8*ld >= 2^32 are refused at creation)
  char* st = (char*)(a.state + e);
  char* rs = a.resid ? (char*)(a.resid + e) : nullptr;
  auto ld = [&](int n) { return src.at(n, src.slot(n)); };
  double AI[SI > 0 ? SI : 1];
  double Bm[I * S > 0 ? I * S : 1];  // Bm[k*S + c] = J[I_k, K_c]
  double hI[I > 0 ? I : 1];
#pragma unroll
  for (int c = 0; c < I; c++) {
#pragma unroll
    for (int r = 0; r <= c; r++) AI[pk(r, c)] = ld(R::FJ + pk(r, c));
  }
#pragma unroll
  for (int c = 0; c < S; c++) {
#pragma unroll
    for (int k = 0; k < I; k++) Bm[k * S + c] = ld(R::FJ + pk(k, I + c));
  }
#pragma unroll
  for (int k = 0; k < I; k++) hI[k] = ld(R::FH + k);
  double g = ld(R::FG);
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;
  const double sg_old = sz ? 0.0 : ld(R::SG);
  const double tg_old = ld(R::TG);

  // "Ji = Jki = hi = 0 if missing data" shortcut, src/beliefupdates.jl:62-66
  bool allzero = true;
#pragma unroll
  for (int q = 0; q < SI; q++)
    if (!(fabs(AI[q]) <= PGBP_EPS)) allzero = false;
#pragma unroll
  for (int q = 0; q < I * S; q++)
    if (!(fabs(Bm[q]) <= PGBP_EPS)) allzero = false;
#pragma unroll
  for (int k = 0; k < I; k++)
    if (!(fabs(hI[k]) <= PGBP_EPS)) allzero = false;

  if (!allzero) {
    double logdet = 0.0, ww = 0.0;
#pragma unroll
    for (int k = 0; k < I; k++) {
      const double d = AI[pk(k, k)];
      if (!(d > 0.0)) {  // LAPACK potrf: info = k+1 (also catches NaN)
        status_fail(a.status, e, PGBP_STATUS(a.ref_base + (int32_t)md.ref, k + 1));
        return;
      }
      logdet += log(d);
      const double rinv = 1.0 / sqrt(d);
#pragma unroll
      for (int c = k + 1; c < I; c++) AI[pk(k, c)] *= rinv;
#pragma unroll
      for (int c = 0; c < S; c++) Bm[k * S + c] *= rinv;
      const double wk = hI[k] * rinv;
      hI[k] = wk;
      ww = fma(wk, wk, ww);
#pragma unroll
      for (int c = k + 1; c < I; c++) {
        const double akc = AI[pk(k, c)];
#pragma unroll
        for (int r = k + 1; r <= c; r++) AI[pk(r, c)] = nfma(AI[pk(k, r)], akc, AI[pk(r, c)]);
        hI[c] = nfma(akc, wk, hI[c]);
      }
#pragma unroll
      for (int c = 0; c < S; c++) {
        const double bkc = Bm[k * S + c];
#pragma unroll
        for (int r = k + 1; r < I; r++) Bm[r * S + c] = nfma(AI[pk(k, r)], bkc, Bm[r * S + c]);
      }
    }
    g += 0.5 * ((double)I * PGBP_LOG2PI - logdet + ww);
  } else {
#pragma unroll
    for (int q = 0; q < I * S; q++) Bm[q] = 0.0;  // message = (h_K, J_KK, g) unchanged
#pragma unroll
    for (int k = 0; k < I; k++) hI[k] = 0.0;
  }

  double maxJ = 0.0, maxh = 0.0;
  constexpr int NCH = (SS + PGBP_CHUNK - 1) / PGBP_CHUNK;
  static_for<NCH>([&](auto chc) {
    constexpr int q0 = decltype(chc)::value * PGBP_CHUNK;
    constexpr int n = (SS - q0) < PGBP_CHUNK ? (SS - q0) : PGBP_CHUNK;
    double jo[PGBP_CHUNK], so[PGBP_CHUNK], to[PGBP_CHUNK];
    uint32_t ta[PGBP_CHUNK];
    static_for<n>([&](auto kc) {
      constexpr int k = decltype(kc)::value, q = q0 + k, c = colof(q), r = q - c * (c + 1) / 2;
      ta[k] = src.slot(R::TJ + q);
      jo[k] = ld(R::FJ + pk(I + r, I + c));
      so[k] = sz ? 0.0 : ld(R::SJ + q);
      to[k] = src.at(R::TJ + q, ta[k]);
    });
    static_for<n>([&](auto kc) {
      constexpr int k = decltype(kc)::value, q = q0 + k, c = colof(q), r = q - c * (c + 1) / 2;
      double nv = jo[k];
#pragma unroll
      for (int i = 0; i < I; i++) nv = nfma(Bm[i * S + r], Bm[i * S + c], nv);
      const double d = nv - so[k];
      *slot_ptr(st, (uint32_t)md.sJ + q, ld8) = nv;  // (md read at the store: the tile walk's is in shared memory)
      *slot_ptr(st, ta[k], ld8) = to[k] + d;
      if (rs) *slot_ptr(rs, (uint32_t)md.rJ + q, ld8) = d;
      absmax(maxJ, d);
    });
  });
  {
    double ho[S > 0 ? S : 1], so[S > 0 ? S : 1], to[S > 0 ? S : 1];
    uint32_t ta[S > 0 ? S : 1];
#pragma unroll
    for (int k = 0; k < S; k++) {
      ta[k] = src.slot(R::TH + k);
      ho[k] = ld(R::FH + I + k);
      so[k] = sz ? 0.0 : ld(R::SH + k);
      to[k] = src.at(R::TH + k, ta[k]);
    }
#pragma unroll
    for (int k = 0; k < S; k++) {
      double nv = ho[k];
#pragma unroll
      for (int i = 0; i < I; i++) nv = nfma(Bm[i * S + k], hI[i], nv);
      const double d = nv - so[k];
      *slot_ptr(st, (uint32_t)md.sh + k, ld8) = nv;
      *slot_ptr(st, ta[k], ld8) = to[k] + d;
      if (rs) *slot_ptr(rs, (uint32_t)md.rh + k, ld8) = d;
      absmax(maxh, d);
    }
  }
  *slot_ptr(st, (uint32_t)md.sg, ld8) = g;
  *slot_ptr(st, (uint32_t)md.tg, ld8) = tg_old + (g - sg_old);
  store_flag(a, (int)md.dmsg, e, S, maxJ, maxh);
}

// One (message, element) of the register class with operands read from global memory.
template <int CI, int CS>
PGBP_HD void message_thread_t0(const MsgArgs& a, int msg_index, int64_t e) {
  const MsgDesc md = a.msgs[msg_index];  // by value: lives in registers, never re-read after a store
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  const T0Global<CI, CS> src{md, a.tab + md.gat, a.tab + md.sca, (char*)(a.state + e), (uint32_t)(a.ld * 8)};
  message_body_t0<CI, CS>(a, md, e, src);
}

// Runtime-shape variants share this tail: divide / multiply / residual / flag with
// chunked prefetch.  newJ(r,c,q), newh(k) give the outgoing message.
template <class FJ, class FH>
PGBP_HD void divide_mult_store(const MsgArgs& a, const MsgDesc& md, int64_t e, int S, FJ newJ, FH newh,
                               double newg) {
  const int64_t ld = a.ld;
  double* st = a.state + e;
  double* rs = a.resid ? a.resid + e : nullptr;
  const int32_t* __restrict__ sca = a.tab + md.sca;
  const int SS = tri(S);
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;
  const double sg_old = sz ? 0.0 : st[md.sg * ld], tg_old = st[md.tg * ld];
  double maxJ = 0.0, maxh = 0.0;
  int r = 0, c = 0;  // (r,c) of packed index q, advanced incrementally
  for (int q0 = 0; q0 < SS; q0 += PGBP_CHUNK) {
    double nv[PGBP_CHUNK], so[PGBP_CHUNK], to[PGBP_CHUNK];
    int64_t ta[PGBP_CHUNK];
#pragma unroll
    for (int k = 0; k < PGBP_CHUNK; k++) {
      const int q = q0 + k;
      if (q < SS) {
        ta[k] = (md.tJ + sca[q]) * ld;
        nv[k] = newJ(r, c, q);
        so[k] = sz ? 0.0 : st[(md.sJ + q) * ld];
        to[k] = st[ta[k]];
        if (++r > c) { r = 0; c++; }
      }
    }
#pragma unroll
    for (int k = 0; k < PGBP_CHUNK; k++) {
      const int q = q0 + k;
      if (q < SS) {
        const double d = nv[k] - so[k];
        st[(md.sJ + q) * ld] = nv[k];
        st[ta[k]] = to[k] + d;
        if (rs) rs[(md.rJ + q) * ld] = d;
        absmax(maxJ, d);
      }
    }
  }
  for (int k0 = 0; k0 < S; k0 += PGBP_CHUNK) {
    double nv[PGBP_CHUNK], so[PGBP_CHUNK], to[PGBP_CHUNK];
    int64_t ta[PGBP_CHUNK];
#pragma unroll
    for (int k = 0; k < PGBP_CHUNK; k++)
      if (k0 + k < S) {
        ta[k] = (md.th + sca[SS + k0 + k]) * ld;
        nv[k] = newh(k0 + k);
        so[k] = sz ? 0.0 : st[(md.sh + k0 + k) * ld];
        to[k] = st[ta[k]];
      }
#pragma unroll
    for (int k = 0; k < PGBP_CHUNK; k++)
      if (k0 + k < S) {
        const double d = nv[k] - so[k];
        st[(md.sh + k0 + k) * ld] = nv[k];
        st[ta[k]] = to[k] + d;
        if (rs) rs[(md.rh + k0 + k) * ld] = d;
        absmax(maxh, d);
      }
  }
  st[md.sg * ld] = newg;
  st[md.tg * ld] = tg_old + (newg - sg_old);
  store_flag(a, md.dmsg, e, S, maxJ, maxh);
}

struct TrailJ {
  const double* A;
  int I;
  PGBP_HD double operator()(int r, int c, int) const { return A[pk(I + r, I + c)]; }
};
struct TrailH {
  const double* hv;
  int I;
  PGBP_HD double operator()(int k) const { return hv[I + k]; }
};
struct GatherJ {
  const double* st;
  const int32_t* gat;
  int64_t base, ld;
  PGBP_HD double operator()(int, int, int q) const { return st[(base + gat[q]) * ld]; }
};
struct GatherH {
  const double* st;
  const int32_t* gat;
  int64_t base, ld;
  PGBP_HD double operator()(int k) const { return st[(base + gat[k]) * ld]; }
};

// Generic message kernel body: runtime shape, the whole sender belief gathered in
// [I;K] order into thread-local memory sized for MAXM, right-looking partial
// Cholesky over the first i pivots; the trailing block is the outgoing message.
template <int MAXM>
PGBP_HD void message_thread_rt(const MsgArgs& a, int msg_index, int64_t e) {
  constexpr int NA = MAXM * (MAXM + 1) / 2;
  const MsgDesc md = a.msgs[msg_index];
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  const int I = md.mF - md.s, S = md.s, M = md.mF;
  const int64_t ld = a.ld;
  const double* st = a.state + e;
  const double* stj = st;
  const int32_t* __restrict__ gat = a.tab + md.gat;
  double A[NA];
  double hv[MAXM];
  const int SM = tri(M);
#pragma unroll 8
  for (int q = 0; q < SM; q++) A[q] = stj[(md.fJ + gat[q]) * ld];
#pragma unroll 8
  for (int k = 0; k < M; k++) hv[k] = st[(md.fh + gat[SM + k]) * ld];
  double g = st[md.fg * ld];
  bool allzero = true;
  for (int c = 0; c < M; c++) {
    const int rmax = c < I ? c + 1 : I;
    for (int r = 0; r < rmax; r++)
      if (!(fabs(A[pk(r, c)]) <= PGBP_EPS)) allzero = false;
  }
  for (int k = 0; k < I; k++)
    if (!(fabs(hv[k]) <= PGBP_EPS)) allzero = false;
  if (!allzero) {
    double logdet = 0.0, ww = 0.0;
    for (int k = 0; k < I; k++) {
      const double d = A[pk(k, k)];
      if (!(d > 0.0)) {
        status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, k + 1));
        return;
      }
      logdet += log(d);
      const double rinv = 1.0 / sqrt(d);
      for (int c = k + 1; c < M; c++) A[pk(k, c)] *= rinv;
      const double wk = hv[k] * rinv;
      ww = fma(wk, wk, ww);
      for (int c = k + 1; c < M; c++) {
        const double akc = A[pk(k, c)];
        for (int r = k + 1; r <= c; r++) A[pk(r, c)] = nfma(A[pk(k, r)], akc, A[pk(r, c)]);
        hv[c] = nfma(akc, wk, hv[c]);
      }
    }
    g += 0.5 * ((double)I * PGBP_LOG2PI - logdet + ww);
  }
  divide_mult_store(a, md, e, S, TrailJ{A, I}, TrailH{hv, I}, g);
}

// Reference-order message body (PGBP_CAL_REFORDER): the same message computed in the REFERENCE's operation
// order instead of the fused right-looking form above -- marginalize as PDMats does it (src/beliefupdates.jl:68-81):
// left-looking upper Cholesky of J_I in LAPACK dpotf2 order with a division by the pivot, Z = J_KI / U by forward
// substitution, X_invA_Xt = Z Z' accumulated from 0 with un-fused products and subtracted once, mu_I = U \ (U' \ h_I),
// h_K - J_KI mu_I, logdet = 2 sum log U_kk, h_I' mu_I.  A validation mode: it removes every difference in rounding
// ORDER between this library and a LAPACK-style evaluation of the reference, so that on ill-conditioned loopy
// configurations (BASELINE configs[2] on the Bethe graph, DESIGN.md section 2) J and h can be compared bit for
// bit.  One thread per (message, element), thread-local storage: slow, never selected automatically.
template <int MAXM>
PGBP_HD void message_thread_ref(const MsgArgs& a, int msg_index, int64_t e) {
  constexpr int NA = MAXM * (MAXM + 1) / 2, NZ = (MAXM / 2) * (MAXM - MAXM / 2) > 0 ? (MAXM / 2) * (MAXM - MAXM / 2) : 1;
  const MsgDesc md = a.msgs[msg_index];
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  const int I = md.mF - md.s, S = md.s, M = md.mF;
  const int64_t ld = a.ld;
  const double* st = a.state + e;
  const int32_t* __restrict__ gat = a.tab + md.gat;
  double A[NA], hv[MAXM], Z[NZ], mu[MAXM];
  const int SM = tri(M);
  for (int q = 0; q < SM; q++) A[q] = st[(md.fJ + gat[q]) * ld];
  for (int k = 0; k < M; k++) hv[k] = st[(md.fh + gat[SM + k]) * ld];
  double g = st[md.fg * ld];
  bool allzero = true;
  for (int c = 0; c < M; c++) {
    const int rmax = c < I ? c + 1 : I;
    for (int r = 0; r < rmax; r++)
      if (!(fabs(A[pk(r, c)]) <= PGBP_EPS)) allzero = false;
  }
  for (int k = 0; k < I; k++)
    if (!(fabs(hv[k]) <= PGBP_EPS)) allzero = false;
  if (I > 0 && !allzero) {
    for (int j = 0; j < I; j++) {  // dpotf2('U')
      double ajj = A[pk(j, j)];
      for (int k = 0; k < j; k++) ajj -= A[pk(k, j)] * A[pk(k, j)];
      if (!(ajj > 0.0)) {
        status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, j + 1));
        return;
      }
      ajj = sqrt(ajj);
      A[pk(j, j)] = ajj;
      for (int c = j + 1; c < I; c++) {
        double s = A[pk(j, c)];
        for (int k = 0; k < j; k++) s -= A[pk(k, j)] * A[pk(k, c)];
        A[pk(j, c)] = s / ajj;
      }
    }
    for (int r = 0; r < S; r++) {  // row r of Z solves U' z = J_KI[r, :]'
      for (int c = 0; c < I; c++) {
        double s = A[pk(c, I + r)];
        for (int k = 0; k < c; k++) s -= A[pk(k, c)] * Z[r * I + k];
        Z[r * I + c] = s / A[pk(c, c)];
      }
    }
    for (int c = 0; c < S; c++)
      for (int r = 0; r <= c; r++) {
        double d = 0.0;
        for (int k = 0; k < I; k++) d += Z[r * I + k] * Z[c * I + k];
        A[pk(I + r, I + c)] -= d;
      }
    for (int r = 0; r < I; r++) {  // U' y = h_I
      double s = hv[r];
      for (int k = 0; k < r; k++) s -= A[pk(k, r)] * mu[k];
      mu[r] = s / A[pk(r, r)];
    }
    for (int r = I - 1; r >= 0; r--) {  // U mu = y
      double s = mu[r];
      for (int k = r + 1; k < I; k++) s -= A[pk(r, k)] * mu[k];
      mu[r] = s / A[pk(r, r)];
    }
    double logdet = 0.0, quad = 0.0;
    for (int k = 0; k < I; k++) {
      logdet += log(A[pk(k, k)]);
      quad += hv[k] * mu[k];
    }
    logdet *= 2.0;
    for (int r = 0; r < S; r++) {
      double d = 0.0;
      for (int c = 0; c < I; c++) d += A[pk(c, I + r)] * mu[c];
      hv[I + r] -= d;
    }
    g = g + ((double)I * PGBP_LOG2PI - logdet + quad) / 2;
  }
  divide_mult_store(a, md, e, S, TrailJ{A, I}, TrailH{hv, I}, g);
}

// Message with nothing to integrate out (src/beliefupdates.jl:56): the outgoing
// message is the sender's belief re-ordered; streamed, no local storage.
PGBP_HD void message_copy_thread(const MsgArgs& a, int msg_index, int64_t e) {
  const MsgDesc md = a.msgs[msg_index];
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  const int S = md.s;
  const int64_t ld = a.ld;
  const double* st = a.state + e;
  const int32_t* __restrict__ gat = a.tab + md.gat;
  const int SS = tri(S);
  const double g = st[md.fg * ld];
  divide_mult_store(a, md, e, S, GatherJ{st, gat, md.fJ, ld}, GatherH{st, gat + SS, md.fh, ld}, g);
}

// residual_kldiv! (src/beliefs.jl:1060-1075): KL divergence between the message just sent (the new
// sepset belief, J0 = J_s) and the sepset belief before the update (J1 = J_s - dJ, h1 = h_s - dh):
//   ( -tr(J0^-1 dJ) + (mu1-mu0)' J1 (mu1-mu0) + logdet J0 - logdet J1 ) / 2.
// If either matrix is not positive definite nothing is updated (the reference returns false silently).
// stj / rsj / ldj: where the J rows of the sepset and of the residual live (shared-precision batches keep them per
// group, in their own arrays with their own pitch); null = the element's own column of a.state / a.resid.
template <int MAXM>
PGBP_HD void kldiv_thread(const MsgArgs& a, double* kldiv, int msg_index, int64_t e, const double* stj = nullptr,
                          const double* rsj = nullptr, int64_t ldj = 0) {
  constexpr int NA = MAXM * (MAXM + 1) / 2;
  const MsgDesc md = a.msgs[msg_index];
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  const int S = md.s;
  if (S == 0) return;  // empty sepsets are born calibrated (kldiv = 0, src/beliefs.jl:919-922)
  const int64_t ld = a.ld;
  const double* st = a.state + e;
  const double* rs = a.resid + e;
  if (!stj) { stj = a.state + e; rsj = a.resid + e; ldj = ld; }
  double U0[NA], U1[NA], D[NA], m0[MAXM], m1[MAXM];
  const int SS = tri(S);
  for (int q = 0; q < SS; q++) {
    const double j0 = stj[(md.sJ + q) * ldj], dj = rsj[(md.rJ + q) * ldj];
    U0[q] = j0; D[q] = dj; U1[q] = j0 - dj;
  }
  for (int k = 0; k < S; k++) {
    const double h0 = st[(md.sh + k) * ld];
    m0[k] = h0; m1[k] = h0 - rs[(md.rh + k) * ld];
  }
  double ld0 = 0.0, ld1 = 0.0;
  for (int pass = 0; pass < 2; pass++) {  // U'U factorisation + mean of both beliefs
    double* A = pass ? U1 : U0;
    double* hv = pass ? m1 : m0;
    double lg = 0.0;
    for (int k = 0; k < S; k++) {
      const double d = A[pk(k, k)];
      if (!(d > 0.0)) return;
      lg += log(d);
      const double rinv = 1.0 / sqrt(d);
      A[pk(k, k)] = rinv;  // 1 / U_kk
      for (int c = k + 1; c < S; c++) A[pk(k, c)] *= rinv;
      hv[k] *= rinv;
      for (int c = k + 1; c < S; c++) {
        const double akc = A[pk(k, c)];
        for (int r = k + 1; r <= c; r++) A[pk(r, c)] = nfma(A[pk(k, r)], akc, A[pk(r, c)]);
        hv[c] = nfma(akc, hv[k], hv[c]);
      }
    }
    for (int k = S - 1; k >= 0; k--) {  // U mu = w
      double s = hv[k];
      for (int c = k + 1; c < S; c++) s = nfma(A[pk(k, c)], hv[c], s);
      hv[k] = s * A[pk(k, k)];
    }
    if (pass) ld1 = lg; else ld0 = lg;
  }
  // tr(J0^-1 dJ): column k of dJ solved through U0
  double trace = 0.0, x[MAXM];
  for (int k = 0; k < S; k++) {
    for (int r = 0; r < S; r++) x[r] = D[r <= k ? pk(r, k) : pk(k, r)];
    for (int r = 0; r < S; r++) {  // U0' y = d_k
      double s = x[r];
      for (int q = 0; q < r; q++) s = nfma(U0[pk(q, r)], x[q], s);
      x[r] = s * U0[pk(r, r)];
    }
    for (int r = S - 1; r >= k; r--) {  // U0 z = y, down to row k
      double s = x[r];
      for (int q = r + 1; q < S; q++) s = nfma(U0[pk(r, q)], x[q], s);
      x[r] = s * U0[pk(r, r)];
    }
    trace += x[k];
  }
  // (mu1-mu0)' J1 (mu1-mu0) with J1 = J0 - dJ rebuilt from the inputs (U1 now holds its factor)
  double quad = 0.0;
  for (int r = 0; r < S; r++) {
    double s = 0.0;
    for (int c = 0; c < S; c++) {
      const int q = r <= c ? pk(r, c) : pk(c, r);
      const double j1 = stj[(md.sJ + q) * ldj] - D[q];
      s = fma(j1, m1[c] - m0[c], s);
    }
    quad = fma(m1[r] - m0[r], s, quad);
  }
  kldiv[(int64_t)md.dmsg * ld + e] = 0.5 * (-trace + quad + ld0 - ld1);
}

// ---- integratebelief pieces, shared by integrate_thread and marginal_thread (one arithmetic, bit-identical results)
// Load the packed J (from stj, pitch ldj) and h of one belief into A / hv; true if every entry is zero.
template <int MAXM>
PGBP_HD bool integrate_load(const double* st, int64_t ld, const double* stj, int64_t ldj, int64_t jslot, int64_t hslot,
                            int M, double* A, double* hv) {
  const int SM = tri(M);
  bool zero = true;
  for (int q = 0; q < SM; q++) {
    A[q] = stj[(jslot + q) * ldj];
    if (A[q] != 0.0) zero = false;
  }
  for (int k = 0; k < M; k++) {
    hv[k] = st[(hslot + k) * ld];
    if (hv[k] != 0.0) zero = false;
  }
  return zero;
}
// Right-looking Cholesky J = U'U in place (A keeps U with 1/U_kk on the diagonal) and forward solve U'w = h in hv.
// Returns 0, or the 1-based pivot at which J is not positive definite.
template <int MAXM>
PGBP_HD int integrate_factor(double* A, double* hv, int M, double* logdet_out, double* ww_out) {
  double logdet = 0.0, ww = 0.0;
  for (int k = 0; k < M; k++) {
    const double d = A[pk(k, k)];
    if (!(d > 0.0)) return k + 1;
    logdet += log(d);
    const double rinv = 1.0 / sqrt(d);
    A[pk(k, k)] = rinv;
    for (int c = k + 1; c < M; c++) A[pk(k, c)] *= rinv;
    const double wk = hv[k] * rinv;
    hv[k] = wk;
    ww = fma(wk, wk, ww);
    for (int c = k + 1; c < M; c++) {
      const double akc = A[pk(k, c)];
      for (int r = k + 1; r <= c; r++) A[pk(r, c)] = nfma(A[pk(k, r)], akc, A[pk(r, c)]);
      hv[c] = nfma(akc, wk, hv[c]);
    }
  }
  *logdet_out = logdet;
  *ww_out = ww;
  return 0;
}
// Back substitution U mu = w in place in hv; each mu_k is also stored to mu_soa row k when mu_soa is given.
template <int MAXM>
PGBP_HD void integrate_solve(const double* A, double* hv, int M, double* mu_soa, int64_t ld_out, int64_t e) {
  for (int k = M - 1; k >= 0; k--) {
    double s = hv[k];
    for (int c = k + 1; c < M; c++) s = nfma(A[pk(k, c)], hv[c], s);
    hv[k] = s * A[pk(k, k)];
    if (mu_soa) mu_soa[k * ld_out + e] = hv[k];
  }
}
// inv(J) = V V' with V = U^-1 (the conditional covariance that calibrate_exact_cliquetree! reads with
// inv(b.J), src/calibration.jl:463).  In place: A holds U with 1/U_kk on the diagonal; columns
// descending, rows descending, so column c only reads U entries of columns < c and V of column c.
template <int MAXM>
PGBP_HD void integrate_invert(double* A, int M) {
  for (int c = M - 1; c >= 0; c--) {
    for (int r = c - 1; r >= 0; r--) {
      double s = A[pk(r, c)] * A[pk(c, c)];
      for (int k = r + 1; k < c; k++) s = fma(A[pk(r, k)], A[pk(k, c)], s);
      A[pk(r, c)] = -s * A[pk(r, r)];
    }
  }
}
// Entry (i, j), i <= j, of inv(J) = V V' from the V that integrate_invert leaves in A.
PGBP_HD double integrate_cov_entry(const double* A, int M, int i, int j) {
  double s = 0.0;
  for (int k = j; k < M; k++) s = fma(A[pk(i, k)], A[pk(j, k)], s);
  return s;
}

// integratebelief (src/beliefupdates.jl:187-200): mu = J^-1 h,
// norm = g + (m log2pi - logdet J + h'mu)/2; all-zero (h,J) -> (Inf.., g).
template <int MAXM>
PGBP_HD void integrate_thread(const double* state, int32_t* status, int64_t ld, int64_t e, int64_t jslot,
                              int64_t hslot, int64_t gslot, int M, double* mu_soa, double* norm, int64_t ld_out,
                              double* cov_soa = nullptr, const double* stj = nullptr, int64_t ldj = 0) {
  constexpr int NA = MAXM * (MAXM + 1) / 2;
  double A[NA > 0 ? NA : 1];
  double hv[MAXM > 0 ? MAXM : 1];
  const double* st = state + e;
  if (!stj) { stj = st; ldj = ld; }  // (shared-precision batches: J rows of the element's group, own array and pitch)
  const bool zero = integrate_load<MAXM>(st, ld, stj, ldj, jslot, hslot, M, A, hv);
  const double g = st[gslot * ld];
  if (zero) {
    if (mu_soa)
      for (int k = 0; k < M; k++) mu_soa[k * ld_out + e] = INFINITY;
    norm[e] = g;
    return;
  }
  double logdet = 0.0, ww = 0.0;
  const int pivot = integrate_factor<MAXM>(A, hv, M, &logdet, &ww);
  if (pivot) {
    status_fail(status, e, PGBP_STATUS(0x7ffffe, pivot));
    if (mu_soa)
      for (int q = 0; q < M; q++) mu_soa[q * ld_out + e] = NAN;
    norm[e] = NAN;
    return;
  }
  norm[e] = g + 0.5 * ((double)M * PGBP_LOG2PI - logdet + ww);
  if (mu_soa) integrate_solve<MAXM>(A, hv, M, mu_soa, ld_out, e);
  if (cov_soa) {
    integrate_invert<MAXM>(A, M);
    for (int j = 0; j < M; j++)
      for (int i = 0; i <= j; i++) cov_soa[(int64_t)pk(i, j) * ld_out + e] = integrate_cov_entry(A, M, i, j);
  }
}

// Posterior moments of position subsets of one belief (pgbp_marginal_moments): the belief is read and factorised
// once per element, then every query [t0, t1) of it gets mu[pos] and the packed upper triangle of inv(J)[pos, pos],
// with the arithmetic of integrate_thread (same entries bit for bit).  qtab[4t..4t+3] = (k, offset of the positions
// in qpos, first mu row, first covariance row).  All-zero (J, h): +Inf everywhere; J not positive definite: status
// 0x7ffffe and NaN everywhere.
struct MargDesc {
  int64_t jslot, hrow;  // J slot (plan layout; the group batch's array for shared-precision batches), first h row
  int32_t m, t0, t1, pad;
};
template <int MAXM>
PGBP_HD void marginal_thread(const double* state, int32_t* status, int64_t ld, int64_t e, const MargDesc& d,
                             const int32_t* qtab, const int32_t* qpos, double* mu_soa, double* cov_soa,
                             int64_t ld_out, const double* stj, int64_t ldj) {
  constexpr int NA = MAXM * (MAXM + 1) / 2;
  double A[NA > 0 ? NA : 1];
  double hv[MAXM > 0 ? MAXM : 1];
  const double* st = state + e;
  if (!stj) { stj = st; ldj = ld; }
  const int M = d.m;
  double fillv = INFINITY;
  bool ok = !integrate_load<MAXM>(st, ld, stj, ldj, d.jslot, d.hrow, M, A, hv);
  if (ok) {
    double logdet, ww;
    const int pivot = integrate_factor<MAXM>(A, hv, M, &logdet, &ww);
    if (pivot) {
      status_fail(status, e, PGBP_STATUS(0x7ffffe, pivot));
      fillv = NAN;
      ok = false;
    }
  }
  if (!ok) {
    for (int t = d.t0; t < d.t1; t++) {
      const int k = qtab[4 * t];
      for (int r = 0; r < k; r++) mu_soa[(int64_t)(qtab[4 * t + 2] + r) * ld_out + e] = fillv;
      if (cov_soa)
        for (int r = 0; r < tri(k); r++) cov_soa[(int64_t)(qtab[4 * t + 3] + r) * ld_out + e] = fillv;
    }
    return;
  }
  integrate_solve<MAXM>(A, hv, M, nullptr, 0, e);
  if (cov_soa) integrate_invert<MAXM>(A, M);
  for (int t = d.t0; t < d.t1; t++) {
    const int k = qtab[4 * t];
    const int32_t* pos = qpos + qtab[4 * t + 1];
    const int64_t mr = qtab[4 * t + 2], cr = qtab[4 * t + 3];
    for (int r = 0; r < k; r++) mu_soa[(mr + r) * ld_out + e] = hv[pos[r]];
    if (cov_soa)
      for (int c = 0; c < k; c++)
        for (int r = 0; r <= c; r++) {
          const int a = pos[r], b = pos[c];
          cov_soa[(cr + pk(r, c)) * ld_out + e] = a <= b ? integrate_cov_entry(A, M, a, b) : integrate_cov_entry(A, M, b, a);
        }
  }
}

}  // namespace pgbp
