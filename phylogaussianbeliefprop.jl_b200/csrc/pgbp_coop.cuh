// K2, cooperative class: medium message shapes (sender dimension 13..32), G lanes per
// batch element.
//
// Why: one thread per element needs S(m_F)+m_F doubles of live state (m_F = 24: 324 doubles =
// 648 registers) -- it spills to local memory and thrashes L1/L2 (measured 260 GB/s on
// (i,s) = (16,8)).  Here the sender belief is spread column-cyclically over G lanes of one
// warp: lane g owns columns c = g, g+G, g+2G, .. of the [I;K]-ordered upper triangle (rows
// 0..c) and the matching entries of h.  m_F = 24, G = 8: at most 8+16+24 (+3) doubles per lane.
//
// Memory: the state layout is unchanged (batch-innermost SoA).  A warp holds 32/G consecutive
// elements; lanes with the same g are adjacent, so every warp-level load/store touches G slots x
// (32/G consecutive doubles): full 32-byte sectors for G <= 8.
//
// Arithmetic: right-looking U'U elimination of the first I pivots.  At pivot k every lane scales
// its own row-k entries (U[k,c] = A[k,c] / sqrt(d_k)) and publishes them in a per-element row
// buffer in shared memory; after one __syncwarp every lane reads U[k,r] (broadcast reads: the G
// lanes of an element read the same word) and applies  A[r,c] -= U[k,r] U[k,c]  to its columns.
// Each entry therefore receives its updates in ascending k with the same operands as in the
// register-resident (T0) and generic kernels: results are bit-identical to theirs.
// After I pivots the trailing block IS the outgoing message (src/beliefupdates.jl:77-82); each
// lane then does divide! / mult! / residual (src/beliefupdates.jl:579-587,483-488,646-647) for its
// own columns.
#pragma once
#include "pgbp_bulk.cuh"
#include "pgbp_kernels.cuh"

namespace pgbp {

#ifndef PGBP_HOST_EMUL

template <int MAXM, int G>
__global__ void __launch_bounds__(128) k_message_coop(MsgArgs a) {
  constexpr int RPW = 32 / G;               // elements per warp
  constexpr int RPB = 128 / G;              // elements per block
  constexpr int NJ = (MAXM + G - 1) / G;    // column slots per lane
  constexpr unsigned FULL = 0xffffffffu;
  __shared__ double rowbuf[2][MAXM + 1][RPB];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane / RPW, rw = lane % RPW;  // lane = g * RPW + rw
  const int rb = warp * RPW + rw;
  const int64_t e = a.e0 + (int64_t)blockIdx.x * RPB + rb;
  const MsgDesc md = a.msgs[blockIdx.y];
  const int I = md.mF - md.s, S = md.s, M = md.mF;
  const int64_t ld = a.ld;
  bool active = e < a.B;
  if (active) active = a.status[e] == 0 && !(a.done && a.done[e]);
  double* st = a.state + (active ? e : 0);
  double* rs = a.resid ? a.resid + (active ? e : 0) : nullptr;
  const int32_t* __restrict__ gat = a.tab + md.gat;
  const int32_t* __restrict__ sca = a.tab + md.sca;
  const int SM = tri(M), SS = tri(S);
  // lanes of this element: bit (gg * RPW + rw) for gg < G
  unsigned repmask = 0;
#pragma unroll
  for (int gg = 0; gg < G; gg++) repmask |= 1u << (gg * RPW + rw);

  // ---- gather my columns (rows 0..c) and my h entries ---------------------------------
  double A[NJ][MAXM];
  double hc[NJ];
  bool nz = false;  // some entry of J_II, J_IK, h_I is not within eps of 0 (src/beliefupdates.jl:63)
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    const int c = g + G * j;
    const bool cv = active && c < M;
    const int RJ = (G * j + G < MAXM) ? (G * j + G) : MAXM;
#pragma unroll
    for (int r = 0; r < RJ; r++) {
      double v = 0.0;
      if (cv && r <= c) v = st[(md.fJ + gat[pk(r, c)]) * ld];
      A[j][r] = v;
      if (r < I && !(fabs(v) <= PGBP_EPS)) nz = true;
    }
    double hv = 0.0;
    if (cv) hv = st[(md.fh + gat[SM + c]) * ld];
    hc[j] = hv;
    if (c < I && !(fabs(hv) <= PGBP_EPS)) nz = true;
  }
  const double g_old = st[md.fg * ld];
  const bool skip = (__ballot_sync(FULL, nz) & repmask) == 0;  // message = (h_K, J_KK, g) unchanged

  // ---- eliminate the first I pivots -----------------------------------------------------
  double dk[NJ];  // pivots I own (k = g + G*j), for the log-determinant
#pragma unroll
  for (int j = 0; j < NJ; j++) dk[j] = 1.0;
  double ww = 0.0;
  int fail_pivot = 0;
  // (static_for: the pivot index must be a compile-time constant for the register arrays, also at MAXM = 48
  //  where a pragma-unrolled loop is left rolled by the compiler)
  static_for<MAXM>([&](auto kc_) {
    constexpr int k = decltype(kc_)::value;
    if (k < I) {
    constexpr int jk = k / G, gk = k % G;
    const int src = gk * RPW + rw;
    const double d = __shfl_sync(FULL, A[jk][k], src);
    if (!skip && fail_pivot == 0 && !(d > 0.0)) fail_pivot = k + 1;  // LAPACK potrf info (also NaN)
    if (g == gk) dk[jk] = d;
    const double rinv = skip ? 0.0 : 1.0 / sqrt(d);
    double(*row)[RPB] = rowbuf[k & 1];
    // scale my row-k entries, publish them
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const int RJ = (G * j + G < MAXM) ? (G * j + G) : MAXM;
      if (k < RJ) {
        const int c = g + G * j;
        if (c > k) {
          const double u = A[j][k] * rinv;
          A[j][k] = u;
          if (c < M) row[c][rb] = u;
        } else if (c == k) {
          row[MAXM][rb] = hc[j] * rinv;  // w_k
        }
      }
    }
    __syncwarp();
    const double wk = row[MAXM][rb];
    ww = fma(wk, wk, ww);
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const int RJ = (G * j + G < MAXM) ? (G * j + G) : MAXM;
      if (k + 1 < RJ) {
        const int c = g + G * j;
        if (c > k) {
          const double ukc = A[j][k];
#pragma unroll
          for (int r = k + 1; r < RJ; r++)
            if (r <= c && c < M) A[j][r] = nfma(row[r][rb], ukc, A[j][r]);
          hc[j] = nfma(ukc, wk, hc[j]);
        }
      }
    }
    }
  });
  if (fail_pivot) {
    if (active && g == 0) status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, fail_pivot));
    active = false;
  }

  // ---- log-normaliser: logs of my pivots in parallel, summed in pivot order ---------------
  double lg[NJ];
#pragma unroll
  for (int j = 0; j < NJ; j++) lg[j] = (G * j < MAXM && g + G * j < I) ? log(dk[j]) : 0.0;
  double logdet = 0.0;
  static_for<MAXM>([&](auto kc_) {
    constexpr int k = decltype(kc_)::value;
    if (k < I) logdet += __shfl_sync(FULL, lg[k / G], (k % G) * RPW + rw);
  });
  double gnew = g_old;
  if (!skip) gnew += 0.5 * ((double)I * PGBP_LOG2PI - logdet + ww);

  // ---- divide! / mult! / residual for my kept columns -----------------------------------------
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;
  double maxJ = 0.0, maxh = 0.0;
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    const int RJ = (G * j + G < MAXM) ? (G * j + G) : MAXM;
    const int c = g + G * j;
    const bool cv = active && c >= I && c < M;
    const int cc = c - I;
#pragma unroll
    for (int r0 = 0; r0 < RJ; r0 += PGBP_CHUNK) {
      double so[PGBP_CHUNK], to[PGBP_CHUNK];
      int64_t ta[PGBP_CHUNK], sa[PGBP_CHUNK];
#pragma unroll
      for (int u = 0; u < PGBP_CHUNK; u++) {
        const int r = r0 + u;
        if (r < RJ) {
          const bool v = cv && r >= I && r <= c;
          const int q = v ? pk(r - I, cc) : 0;
          sa[u] = (md.sJ + q) * ld;
          ta[u] = (md.tJ + (v ? sca[q] : 0)) * ld;
          so[u] = (v && !sz) ? st[sa[u]] : 0.0;
          to[u] = v ? st[ta[u]] : 0.0;
        }
      }
#pragma unroll
      for (int u = 0; u < PGBP_CHUNK; u++) {
        const int r = r0 + u;
        if (r < RJ) {
          const bool v = cv && r >= I && r <= c;
          if (v) {
            const double nv = A[j][r];
            const double d = nv - so[u];
            st[sa[u]] = nv;
            st[ta[u]] = to[u] + d;
            if (rs) rs[(md.rJ + pk(r - I, cc)) * ld] = d;
            absmax(maxJ, d);
          }
        }
      }
    }
    if (cv) {
      const int64_t sa = (md.sh + cc) * ld, ta = (md.th + sca[SS + cc]) * ld;
      const double so = sz ? 0.0 : st[sa], to = st[ta];
      const double nv = hc[j];
      const double d = nv - so;
      st[sa] = nv;
      st[ta] = to + d;
      if (rs) rs[(md.rh + cc) * ld] = d;
      absmax(maxh, d);
    }
  }
  // NaN-propagating max over the G lanes of the element
#pragma unroll
  for (int gg = 1; gg < G; gg <<= 1) {
    const int src = ((g ^ gg) * RPW + rw);
    const double oJ = __shfl_sync(FULL, maxJ, src), oh = __shfl_sync(FULL, maxh, src);
    if (oJ > maxJ || oJ != oJ) maxJ = (maxJ != maxJ) ? maxJ : oJ;
    if (oh > maxh || oh != oh) maxh = (maxh != maxh) ? maxh : oh;
  }
  if (active && g == 0) {
    const double sg_old = sz ? 0.0 : st[md.sg * ld], tg_old = st[md.tg * ld];
    st[md.sg * ld] = gnew;
    st[md.tg * ld] = tg_old + (gnew - sg_old);
    store_flag(a, md.dmsg, e, S, maxJ, maxh);
  }
}

#endif  // !PGBP_HOST_EMUL

// =====================================================================================
// K2, shared-memory class ("T0S"): the register-resident algorithm of message_thread_t0 with its
// working set (U = chol(J_II) rows, Z = U^-T J_IK, w = U^-T h_I) held in SHARED memory instead of
// registers, one thread per batch element, one warp per block.
//
// Why this and not more lanes per element: the cooperative kernel above spends ~0.19 warp
// instructions per byte moved (every lane repeats the pivot bookkeeping and runs predicated-off
// work) and the SM's issue rate, not HBM, bounds it.  One thread per element costs ~0.04, so the
// kernel can be HBM-bound; what a thread lacks is storage (m_F = 16: 108 live doubles), and that
// is what shared memory provides: tri(I) + I*S + I doubles per element, laid out [entry][lane], so
// every LDS/STS of a warp is one conflict-free 256-byte row and no two threads ever touch the same
// word -- no barrier anywhere in the kernel.
//
//   A  the I-rows of the sender (J_II upper, J_IK, h_I) go global -> shared with 8-byte cp.async:
//      all loads of the element are in flight at once, no registers staged;
//   B  left-looking U'U: one column at a time in registers (at most MAXI doubles), previous rows
//      read back from shared memory: one LDS per FMA, one STS per finished entry;
//   C  the kept block is STREAMED column by column, like in message_thread_t0: sender J_KK, old
//      sepset and old receiver values are loaded together (24 independent loads per thread), then
//      new = J_KK - z_r.z_c, delta = new - old, three stores.
// Per-entry update order and operands equal message_thread_t0 / message_thread_rt: bit-identical.
// =====================================================================================
// doubles of shared memory per element
PGBP_HD int smem_doubles(int I, int S) { return I * (I + 1) / 2 + I * S + I; }
// 16-bit index tables of one message, staged in shared memory (+ 4 entries of slack)
PGBP_HD size_t smem_table_bytes(int I, int S) {
  const int M = I + S;
  return sizeof(uint16_t) * (size_t)(M * (M + 1) / 2 + M + S * (S + 1) / 2 + S + 4);
}
// bytes of shared memory per block (one warp) of k_message_smem<I>: element data + index tables
PGBP_HD size_t smem_block_bytes(int I, int S) {
  return sizeof(double) * 32 * (size_t)smem_doubles(I, S) + smem_table_bytes(I, S);
}
// bytes of shared memory per tile of k_message_smem_mw<I, NW, TILE, .>: factor rows + 2 scalar rows (x TILE lanes x
// 8 bytes), per-lane int32 flags (active, failed pivot, one non-zero flag per warp), index tables; 16 bytes of slack
// on narrow tiles
PGBP_HD size_t smem_tile_bytes(int I, int S, int NW, int TILE) {
  return sizeof(double) * TILE * (size_t)(smem_doubles(I, S) + 2) + sizeof(int32_t) * TILE * (size_t)(2 + NW) +
         smem_table_bytes(I, S) + (TILE < 32 ? 16 : 0);
}

#ifndef PGBP_HOST_EMUL

__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p)); }

// Phase C of every shared-memory kernel below: the kept block streamed like in message_thread_t0.  For a chunk of CH
// kept entries the sender's J_KK (h_K) entry, the old sepset value and the old receiver value are loaded together,
// then  nv = J_KK - z_r.z_c  (h_K - Z'w) with nfma over i ascending,  d = nv - old sepset,  and three stores: the
// sepset gets nv, the receiver old + d, the residual d.  Per entry the operands and their order are those of
// message_thread_t0 / message_thread_rt, so each kernel that streams through here is bit-identical to them.
//   LS  lane stride of the Z tile: Z(k, cc) = Z[(cc * I + k) * LS], column S holds w = U^-T h_I
//   MI  compile-time bound on the integrated dimension I (MI == I where I is a template argument: the guards fold)
//   MS  0: S is a runtime value, chunks of PGBP_CHUNK entries; > 0: S <= MS, a kept column or the h part is one chunk
//   T   element type of the index tables (uint16_t staged in shared memory, or int32_t read from global memory)
template <int LS, int MI, int MS, class T>
struct KeptStream {
  static constexpr int CH = MS > 0 ? MS : PGBP_CHUNK;
  const double* Z;
  int I, S;
  const T* gat;  // sender slots in [I;K] order: J (tri(M) entries), then h
  const T* sca;  // receiver slots at the sepset's positions: J (tri(S) entries), then h
  char* st;
  char* rs;      // may be null
  uint32_t ld8, fJ, fh, sJ, sh, tJ, th, rJ, rh;
  bool sz;       // PGBP_OPT_SEPZERO: the old sepset is zero and not loaded

  __device__ __forceinline__ KeptStream(const double* Z_, int I_, const MsgDesc& md, const T* gat_, const T* sca_,
                                        char* st_, char* rs_, uint32_t ld8_, bool sz_)
      : Z(Z_), I(I_), S(md.s), gat(gat_), sca(sca_), st(st_), rs(rs_), ld8(ld8_), fJ((uint32_t)md.fJ),
        fh((uint32_t)md.fh), sJ((uint32_t)md.sJ), sh((uint32_t)md.sh), tJ((uint32_t)md.tJ), th((uint32_t)md.th),
        rJ((uint32_t)md.rJ), rh((uint32_t)md.rh), sz(sz_) {}

  // kept column cc: entries (rr, cc), rr = 0..cc.  (MS > 0: z_c is read after the column's loads and reused for the
  // diagonal entry -- the same values, in the order that keeps the unrolled kernels at their register budget.)
  __device__ __forceinline__ void column(int cc, double& maxJ) const {
    double zc[MI];
    auto load_zc = [&] {
#pragma unroll
      for (int i = 0; i < MI; i++) zc[i] = i < I ? Z[(cc * I + i) * LS] : 0.0;
    };
    if (MS == 0) load_zc();
    const T* gc = gat + tri(I + cc) + I;  // sender slots of (I+rr, I+cc), rr = 0..cc
    const int qc = tri(cc);
    for (int r0 = 0; r0 <= cc; r0 += CH) {
      double jo[CH], so[CH], to[CH];
      double* ta[CH];
#pragma unroll
      for (int u = 0; u < CH; u++) {
        const int rr = r0 + u;
        if (rr <= cc) {
          ta[u] = slot_ptr(st, tJ + sca[qc + rr], ld8);
          jo[u] = *slot_ptr(st, fJ + gc[rr], ld8);
          so[u] = sz ? 0.0 : *slot_ptr(st, sJ + qc + rr, ld8);
          to[u] = *ta[u];
        }
      }
      if (MS > 0) load_zc();
#pragma unroll
      for (int u = 0; u < CH; u++) {
        const int rr = r0 + u;
        if (rr <= cc) {
          double nv = jo[u];
          const double* zr = Z + rr * I * LS;
#pragma unroll
          for (int i = 0; i < MI; i++)
            if (i < I) nv = nfma(MS > 0 && rr == cc ? zc[i] : zr[i * LS], zc[i], nv);
          const double d = nv - so[u];
          *slot_ptr(st, sJ + qc + rr, ld8) = nv;
          *ta[u] = to[u] + d;
          if (rs) *slot_ptr(rs, rJ + qc + rr, ld8) = d;
          absmax(maxJ, d);
        }
      }
      if (MS > 0) break;  // cc < MS: one chunk
    }
  }

  // h entries in chunks [k0, k0 + CH), [k0 + kstep, k0 + kstep + CH), ...
  __device__ __forceinline__ void hpart(int k0, int kstep, double& maxh) const {
    double w[MI];
#pragma unroll
    for (int i = 0; i < MI; i++) w[i] = i < I ? Z[(S * I + i) * LS] : 0.0;
    const T* gh = gat + tri(I + S) + I;
    const T* sh_ = sca + tri(S);
    for (; k0 < S; k0 += kstep) {
      double ho[CH], so[CH], to[CH];
      double* ta[CH];
#pragma unroll
      for (int u = 0; u < CH; u++) {
        const int k = k0 + u;
        if (k < S) {
          ta[u] = slot_ptr(st, th + sh_[k], ld8);
          ho[u] = *slot_ptr(st, fh + gh[k], ld8);
          so[u] = sz ? 0.0 : *slot_ptr(st, sh + k, ld8);
          to[u] = *ta[u];
        }
      }
#pragma unroll
      for (int u = 0; u < CH; u++) {
        const int k = k0 + u;
        if (k < S) {
          double nv = ho[u];
          const double* zr = Z + k * I * LS;
#pragma unroll
          for (int i = 0; i < MI; i++)
            if (i < I) nv = nfma(zr[i * LS], w[i], nv);
          const double d = nv - so[u];
          *slot_ptr(st, sh + k, ld8) = nv;
          *ta[u] = to[u] + d;
          if (rs) *slot_ptr(rs, rh + k, ld8) = d;
          absmax(maxh, d);
        }
      }
      if (MS > 0) break;  // S <= MS: one chunk
    }
  }

  // L2 prefetch of everything column(cc) and h entry cc read (kept block of the sender, old sepset, old receiver):
  // issued before the factorisation, the HBM -> L2 transfers overlap it and phase C then waits on L2 only.  UNROLL:
  // unroll count of the loop over the column's entries (the single-warp kernel keeps it rolled, the multi-warp kernel
  // unrolls it 4 x: measured on C5, rolled there it was 0.4 % slower)
  template <int UNROLL>
  __device__ __forceinline__ void prefetch(int cc) const {
    const T* gc = gat + tri(I + cc) + I;
    const int qc = tri(cc);
#pragma unroll(UNROLL)
    for (int rr = 0; rr <= cc; rr++) {
      prefetch_l2(slot_ptr(st, fJ + gc[rr], ld8));
      if (!sz) prefetch_l2(slot_ptr(st, sJ + qc + rr, ld8));
      prefetch_l2(slot_ptr(st, tJ + sca[qc + rr], ld8));
    }
    prefetch_l2(slot_ptr(st, fh + gat[tri(I + S) + I + cc], ld8));
    if (!sz) prefetch_l2(slot_ptr(st, sh + cc, ld8));
    prefetch_l2(slot_ptr(st, th + sca[tri(S) + cc], ld8));
  }
};

// TILE < 32: narrow tiles for shapes whose 32-element factor exceeds the SM's shared memory (C5's (32,16)
// messages: 274 KB at 32 lanes, 206 KB at 24): lanes >= TILE idle, rows of TILE doubles (whole 32-byte sectors
// for TILE = 16, 24).  No warp-level synchronisation anywhere in this kernel.
template <int MAXI, int TILE = 32>
__global__ void __launch_bounds__(32) k_message_smem_rt(MsgArgs a) {
  extern __shared__ double sm[];
  const int tid = threadIdx.x;
  if (TILE < 32 && tid >= TILE) return;
  const int64_t e = a.e0 + (int64_t)blockIdx.x * TILE + tid;
  if (e >= a.B) return;
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  const MsgDesc md = a.msgs[blockIdx.y];
  const int I = md.mF - md.s, S = md.s, M = md.mF;
  const int64_t ld = a.ld;
  double* st = a.state + e;
  const int32_t* __restrict__ gat = a.tab + md.gat;
  const int TI = tri(I), SMM = tri(M);
  const int ZB = TI, WB = TI + I * S;  // region bases: Z(k, cc) = ZB + cc*I + k, w(k) = WB + k
#define PGBP_SM(ent) sm[(ent) * TILE + tid]

  // ---- A: I-rows of the sender -> shared (asynchronous) ---------------------------------
  for (int c = 0; c < M; c++) {
    const int kmax = c < I ? c + 1 : I;
    const int base = c < I ? tri(c) : ZB + (c - I) * I;
    const int32_t* gc = gat + tri(c);
#pragma unroll 4
    for (int k = 0; k < kmax; k++) cp_async8(&PGBP_SM(base + k), st + (md.fJ + gc[k]) * ld);
  }
#pragma unroll 4
  for (int k = 0; k < I; k++) cp_async8(&PGBP_SM(WB + k), st + (md.fh + gat[SMM + k]) * ld);
  double g = st[md.fg * ld];
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;
  const double sg_old = sz ? 0.0 : st[md.sg * ld], tg_old = st[md.tg * ld];
  cp_async_wait_all();

  // "Ji = Jki = hi = 0 if missing data" shortcut (src/beliefupdates.jl:62-66)
  bool allzero = true;
  {
    const int n = WB + I;
#pragma unroll 4
    for (int q = 0; q < n; q++)
      if (!(fabs(PGBP_SM(q)) <= PGBP_EPS)) allzero = false;
  }

  if (!allzero) {
    // ---- B: left-looking factorisation, column c in registers ------------------------------
    double rinv[MAXI];
#pragma unroll
    for (int k = 0; k < MAXI; k++) rinv[k] = 0.0;
    double logdet = 0.0, ww = 0.0;
    for (int c = 0; c <= M; c++) {  // c == M: the h column
      const bool isp = c < I, ish = c == M;
      const int kmax = isp ? c + 1 : I;      // rows held
      const int nelim = isp ? c : I;         // pivots applied
      const int base = isp ? tri(c) : (ish ? WB : ZB + (c - I) * I);
      double v[MAXI];
#pragma unroll
      for (int k = 0; k < MAXI; k++) v[k] = k < kmax ? PGBP_SM(base + k) : 0.0;
#pragma unroll
      for (int k = 0; k < MAXI; k++) {
        if (k >= nelim) break;
        const double u = v[k] * rinv[k];
        v[k] = u;
        PGBP_SM(base + k) = u;
        if (ish) ww = fma(u, u, ww);
#pragma unroll
        for (int r = k + 1; r < MAXI; r++)
          if (r < kmax) v[r] = nfma(PGBP_SM(pk(k, r)), u, v[r]);
      }
      if (isp) {
        double d = 0.0;
#pragma unroll
        for (int k = 0; k < MAXI; k++)
          if (k == c) d = v[k];
        if (!(d > 0.0)) {  // LAPACK potrf: info = c+1 (also catches NaN)
          status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, c + 1));
          return;
        }
        logdet += log(d);
        const double ri = 1.0 / sqrt(d);
#pragma unroll
        for (int k = 0; k < MAXI; k++)
          if (k == c) rinv[k] = ri;
      }
    }
    g += 0.5 * ((double)I * PGBP_LOG2PI - logdet + ww);
  } else {
    const int n = WB + I;  // message = (h_K, J_KK, g) unchanged: Z = 0, w = 0
    for (int q = TI; q < n; q++) PGBP_SM(q) = 0.0;
  }

  // ---- C: stream the kept block ---------------------------------------------------------------
  const KeptStream<TILE, MAXI, 0, int32_t> ks(&PGBP_SM(ZB), I, md, gat, a.tab + md.sca, (char*)st,
                                              a.resid ? (char*)(a.resid + e) : nullptr, (uint32_t)(ld * 8), sz);
  double maxJ = 0.0, maxh = 0.0;
  for (int cc = 0; cc < S; cc++) ks.column(cc, maxJ);
  ks.hpart(0, PGBP_CHUNK, maxh);
  st[md.sg * ld] = g;
  st[md.tg * ld] = tg_old + (g - sg_old);
  store_flag(a, md.dmsg, e, S, maxJ, maxh);
#undef PGBP_SM
}


// -------------------------------------------------------------------------------------
// Same kernel with the integrated dimension I known at compile time (I <= 16): no predicated
// work (every loop over pivots / rows has constant bounds), shared-memory offsets are immediates,
// global addresses are one IMAD.WIDE.U32 each (slot * 8*ld + base), and the Z columns (and the h
// column, which is simply column S of the right-hand sides) are solved TWO at a time so that one
// LDS of U[k,r] feeds two independent FMA chains.  ncu on the runtime-I version: 12.8k warp
// instructions per warp-message, 55% of them integer address / predicate work, IPC 1.2; this
// version: see profiles/.
// The "all zero" test of src/beliefupdates.jl:62-66 is folded into the loads of phase B; a failed
// pivot is only reported once the whole I-part has been seen to be non-zero.
// -------------------------------------------------------------------------------------
// MS = 0: kept dimension S is a runtime value (loops over kept columns stay loops);
// MS > 0: S <= MS and every loop over kept columns / rows is fully unrolled with uniform early exits --
// straight-line code whose table offsets and shared-memory offsets are immediates and whose loads the
// scheduler can hoist across columns.
template <int I, int MS>
__global__ void __launch_bounds__(32) k_message_smem(MsgArgs a) {
  extern __shared__ double sm[];
  const int tid = threadIdx.x;
  const int64_t e = a.e0 + (int64_t)blockIdx.x * 32 + tid;
  const MsgDesc md = a.msgs[blockIdx.y];
  const int S = md.s, M = md.mF;
  constexpr int TI = I * (I + 1) / 2;
  const int SMM = tri(M), SS = tri(S);
  // index tables of the message -> shared memory, one coalesced pass per warp (they are the same
  // for all elements): afterwards every lookup is a broadcast LDS instead of a dependent LDG
  const int ngat = SMM + M, nsca = SS + S;
  // (16-bit entries: slot offsets inside one belief are < tri(64) + 64; keeps 8 blocks per SM at (8,8))
  uint16_t* tgat = (uint16_t*)(sm + 32 * (TI + I * (S + 1)));
  uint16_t* tsca = tgat + ngat;
  {
    const int32_t* __restrict__ g0 = a.tab + md.gat;
    const int32_t* __restrict__ s0 = a.tab + md.sca;
    for (int q = tid; q < ngat; q += 32) tgat[q] = (uint16_t)g0[q];
    for (int q = tid; q < nsca; q += 32) tsca[q] = (uint16_t)s0[q];
  }
  __syncwarp();
  if (e >= a.B) return;  // (no warp-level synchronisation below this point)
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  const uint32_t ld8 = (uint32_t)(a.ld * 8);
  char* stb = (char*)(a.state + e);
  const uint16_t* gat = tgat;
  double* smt = sm + tid;             // entry n of this thread: smt[n * 32]
  double* Z = smt + TI * 32;          // Z(k, cc) = Z[(cc * I + k) * 32]; column S holds h_I / w
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;
  const KeptStream<32, I, MS, uint16_t> ks(Z, I, md, tgat, tsca, stb, a.resid ? (char*)(a.resid + e) : nullptr, ld8, sz);

  // ---- A: I-rows of the sender -> shared (asynchronous) ---------------------------------
#pragma unroll
  for (int c = 0; c < I; c++) {
#pragma unroll
    for (int k = 0; k <= c; k++) cp_async8(smt + pk(k, c) * 32, slot_ptr(stb, ks.fJ + gat[pk(k, c)], ld8));
  }
#pragma unroll(MS > 0 ? MS : 1)
  for (int cc = 0; cc < (MS > 0 ? MS : S); cc++) {
    if (MS > 0 && cc >= S) break;
    const uint16_t* gc = gat + tri(I + cc);
    double* zc = Z + cc * I * 32;
#pragma unroll
    for (int k = 0; k < I; k++) cp_async8(zc + k * 32, slot_ptr(stb, ks.fJ + gc[k], ld8));
  }
  {
    double* zc = Z + S * I * 32;
#pragma unroll
    for (int k = 0; k < I; k++) cp_async8(zc + k * 32, slot_ptr(stb, ks.fh + gat[SMM + k], ld8));
  }
  double g = *slot_ptr(stb, (uint32_t)md.fg, ld8);
  const double sg_old = sz ? 0.0 : *slot_ptr(stb, (uint32_t)md.sg, ld8), tg_old = *slot_ptr(stb, (uint32_t)md.tg, ld8);
#pragma unroll(MS > 0 ? MS : 1)
  for (int cc = 0; cc < (MS > 0 ? MS : S); cc++) {
    if (MS > 0 && cc >= S) break;
    ks.template prefetch<(MS > 0 ? MS : 1)>(cc);
  }
  cp_async_wait_all();

  // ---- B1: U'U = J_II, left-looking, fully unrolled ------------------------------------------
  double rinv[I];
  double logdet = 0.0;
  bool nz = false;
  int fail = 0;
#pragma unroll
  for (int c = 0; c < I; c++) {
    double v[I];
#pragma unroll
    for (int k = 0; k <= c; k++) {
      v[k] = smt[pk(k, c) * 32];
      if (!(fabs(v[k]) <= PGBP_EPS)) nz = true;
    }
#pragma unroll
    for (int k = 0; k < c; k++) {
      const double u = v[k] * rinv[k];
      v[k] = u;
      smt[pk(k, c) * 32] = u;
#pragma unroll
      for (int r = k + 1; r <= c; r++) v[r] = nfma(r == c ? u : smt[pk(k, r) * 32], u, v[r]);
    }
    const double d = v[c];
    if (!(d > 0.0) && fail == 0) fail = c + 1;  // LAPACK potrf info (also NaN); reported below
    logdet += log(d);
    rinv[c] = 1.0 / sqrt(d);
  }
  // ---- B2: Z = U^-T [J_IK | h_I], two right-hand sides at a time --------------------------------
  double ww = 0.0;
  const int nrhs = S + 1;
  constexpr int NPAIR = (I <= 10) ? 2 : 1;  // larger I: one column at a time (register budget)
  for (int c0 = 0; c0 < nrhs; c0 += NPAIR) {
    const bool two = NPAIR == 2 && c0 + 1 < nrhs;
    double* z0 = Z + c0 * I * 32;
    double* z1 = two ? z0 + I * 32 : z0;
    double v0[I], v1[I];
#pragma unroll
    for (int k = 0; k < I; k++) {
      v0[k] = z0[k * 32];
      v1[k] = z1[k * 32];
      if (!(fabs(v0[k]) <= PGBP_EPS) || !(fabs(v1[k]) <= PGBP_EPS)) nz = true;
    }
#pragma unroll
    for (int k = 0; k < I; k++) {
      const double u0 = v0[k] * rinv[k], u1 = v1[k] * rinv[k];
      v0[k] = u0;
      v1[k] = u1;
#pragma unroll
      for (int r = k + 1; r < I; r++) {
        const double ukr = smt[pk(k, r) * 32];
        v0[r] = nfma(ukr, u0, v0[r]);
        if (NPAIR == 2) v1[r] = nfma(ukr, u1, v1[r]);
      }
    }
#pragma unroll
    for (int k = 0; k < I; k++) {
      z0[k * 32] = v0[k];
      if (two) z1[k * 32] = v1[k];
    }
    if (c0 == S || (NPAIR == 2 && c0 + 1 == S)) {  // the h column: w = U^-T h_I
      const double* w = (c0 == S) ? v0 : v1;
#pragma unroll
      for (int k = 0; k < I; k++) ww = fma(w[k], w[k], ww);
    }
  }
  if (nz) {
    if (fail) {
      status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, fail));
      return;
    }
    g += 0.5 * ((double)I * PGBP_LOG2PI - logdet + ww);
  } else {  // "missing data" shortcut: message = (h_K, J_KK, g) unchanged
    for (int q = 0; q < nrhs * I; q++) Z[q * 32] = 0.0;
  }

  // ---- C: stream the kept block ---------------------------------------------------------------
  double maxJ = 0.0, maxh = 0.0;
#pragma unroll
  for (int cc = 0; cc < (MS > 0 ? MS : S); cc++) {
    if (MS > 0 && cc >= S) break;
    ks.column(cc, maxJ);
  }
  ks.hpart(0, ks.CH, maxh);
  *slot_ptr(stb, (uint32_t)md.sg, ld8) = g;
  *slot_ptr(stb, (uint32_t)md.tg, ld8) = tg_old + (g - sg_old);
  store_flag(a, md.dmsg, e, S, maxJ, maxh);
}

// -------------------------------------------------------------------------------------
// Multi-warp version of k_message_smem for LARGE integrated dimensions (I >= 12: C5's (16,16) and (16,32)
// messages, C4's (16,8); I = 32: C5's (32,16)).  There the factor of 32 elements fills 100-175 KB of shared memory
// (274 KB at I = 32), so only one or two single-warp blocks fit an SM and every phase runs at the latency of its own
// dependent chain (profiles/r1_c5_launches.txt: 49 % of the C5 step).  Here NW warps share ONE tile of TILE elements
// (lane = element, as before) and split the work by COLUMN: the asynchronous staging (phase A) by entry, the
// right-hand sides of Z = U^-T [J_IK | h_I] (phase B2) and the kept columns of the streamed Schur complement
// (phase C, paired cc / S-1-cc for balance) by warp.  Same shared-memory footprint, NW x the warps per SM.
// The Cholesky of J_II (phase B1) comes in two forms:
//   COLPAR = false  on warp 0, left-looking and fully unrolled as in k_message_smem (~12 % of the flops at I = 16);
//                   1/U_cc is kept in the (otherwise unused) diagonal slot of U for the other warps
//   COLPAR = true   right-looking, one block barrier per pivot: the owner of column c (c mod NW) applies pivot k to
//                   its column, A[r,c] -= u_kr u_kc with u_k. = A[k,.] / sqrt(A[k,k]) formed on the fly (row k is not
//                   written during step k); rows are scaled in place afterwards.  For I = 32, where B1 is 29 % of
//                   the flops and would otherwise serialise the tile on one warp.  Per entry the updates arrive in
//                   ascending k with the same operands as in the left-looking form.
// Used as <I, 4 or 8, 32, false> for I = 12..16: NW = 4 (two tiles per SM, full register budget) when two tiles fit
// the SM's shared memory, else NW = 8 (one tile per SM); measured on C5 (B200): single-warp tiles 490 ms per
// calibration step, 8 warps at 128 registers 389 ms, 4 warps at 255 registers 356 ms.  And as <32, 8, 24, true>:
// the 32-element factor does not fit, tiles of 24 elements (lanes 24..31 idle; rows of 24 doubles = six whole
// 32-byte sectors) and ONE tile of 206 KB per SM, so all the parallelism has to come from inside the tile.
// Every entry is still produced by one thread with the same operands in the same order: bit-identical.
// -------------------------------------------------------------------------------------
template <int I, int NW, int TILE, bool COLPAR>
__global__ void __launch_bounds__(32 * NW, NW <= 4 ? 2 : 1) k_message_smem_mw(MsgArgs a) {
  constexpr int TI = I * (I + 1) / 2;
  static_assert(2 * NW <= TI, "the flag reduction reuses rows [0, 2 NW) of U");
  extern __shared__ __align__(128) double sm[];  // bulk-copy destinations need 16-byte alignment
  __shared__ __align__(8) unsigned long long mbar;
  const int tid = threadIdx.x, wid = threadIdx.y;
  if (wid == 0 && tid == 0) mbar_init(&mbar, 1);  // (made visible to the other threads by the barrier after the tables)
  const bool lane_ok = TILE == 32 || tid < TILE;
  const int lane = lane_ok ? tid : 0;      // idle lanes never touch shared memory (all accesses are guarded)
  const int64_t tile0 = a.e0 + (int64_t)blockIdx.x * TILE, e = tile0 + lane;
  const MsgDesc md = a.msgs[blockIdx.y];
  const int S = md.s, M = md.mF;
  const int SMM = tri(M), SS = tri(S);
  const int nrhs = S + 1;
  const int NE = TI + I * nrhs;            // staged entries per element
  // shared layout (smem_tile_bytes): rows of TILE lanes: [0, NE) factor | ww | logdet; then per-lane int32 flags
  // ([lane] active, [TILE + lane] failed pivot, [(2 + w) TILE + lane] warp w saw a non-zero), then the index tables.
  double* smt = sm + lane;                 // entry n of this lane: smt[n * TILE]
  double* Z = smt + TI * TILE;             // Z(k, cc) = Z[(cc * I + k) * TILE]; column S holds h_I / w
  double* s_ww = smt + NE * TILE;
  double* s_logdet = s_ww + TILE;
  double* s_redJ = smt;                    // rows [0, NW) and [NW, 2 NW) of U, dead in phase C
  double* s_redh = smt + NW * TILE;
  int32_t* s_flag = (int32_t*)(sm + TILE * (NE + 2));
  uint16_t* tgat = (uint16_t*)(s_flag + TILE * (2 + NW));
  const int ngat = SMM + M, nsca = SS + S;
  uint16_t* tsca = tgat + ngat;
  {
    const int32_t* __restrict__ g0 = a.tab + md.gat;
    const int32_t* __restrict__ s0 = a.tab + md.sca;
    for (int q = wid * 32 + tid; q < ngat; q += 32 * NW) tgat[q] = (uint16_t)g0[q];
    for (int q = wid * 32 + tid; q < nsca; q += 32 * NW) tsca[q] = (uint16_t)s0[q];
    if (wid == 0 && lane_ok) {
      int act = e < a.B;
      if (act && a.status[e] != 0) act = 0;
      if (act && a.done && a.done[e]) act = 0;
      s_flag[tid] = act;
      s_flag[TILE + tid] = 0;
    }
  }
  __syncthreads();
  const bool active = lane_ok && s_flag[lane] != 0;  // same answer in every warp of the tile
  const int64_t ee = active ? e : tile0;   // inactive lanes shadow a valid element, never store
  const uint32_t ld8 = (uint32_t)(a.ld * 8);
  char* stb = (char*)(a.state + ee);
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;
  const KeptStream<TILE, I, 0, uint16_t> ks(Z, I, md, tgat, tsca, stb, a.resid ? (char*)(a.resid + ee) : nullptr, ld8, sz);

  // ---- A: staging with bulk asynchronous copies: one row of the tile (TILE elements of one slot) per instruction,
  //      rows dealt to the threads of the tile, completion counted in bytes on the tile's mbarrier ----------
  {
    const char* tileb = (const char*)(a.state + tile0);
    unsigned rowbytes = 8u * TILE;
    if (TILE < 32) {  // the last narrow tile of a row may be cut by the row pitch (a multiple of 32 elements)
      const int64_t room = a.ld - tile0;
      if (room < TILE) rowbytes = (unsigned)(room * 8);
    }
    if (wid == 0 && tid == 0) mbar_expect_tx(&mbar, (unsigned)NE * rowbytes);
    for (int n = wid * 32 + tid; n < NE; n += 32 * NW) {
      uint32_t slot;
      if (n < TI) slot = ks.fJ + tgat[n];
      else {
        const int idx = n - TI, cc = idx / I, k = idx - cc * I;
        slot = cc < S ? ks.fJ + tgat[tri(I + cc) + k] : ks.fh + tgat[SMM + k];
      }
      bulk_g2s(sm + n * TILE, tileb + (uint64_t)slot * (uint64_t)ld8, rowbytes, &mbar);
    }
  }
  double g = 0.0, sg_old = 0.0, tg_old = 0.0;
  if (lane_ok) {
    if (wid == 0) {
      g = *slot_ptr(stb, (uint32_t)md.fg, ld8);
      sg_old = sz ? 0.0 : *slot_ptr(stb, (uint32_t)md.sg, ld8);
      tg_old = *slot_ptr(stb, (uint32_t)md.tg, ld8);
    }
    for (int cc = wid; cc < S; cc += NW) ks.template prefetch<4>(cc);
  }
  mbar_wait(&mbar, 0);  // every staged row has landed (async-proxy writes are visible after the wait)
  __syncthreads();

  // ---- B1: U'U = J_II; afterwards every warp holds 1/U_kk in rinv --------------------------------
  bool nz = false;
  double rinv[I];
  if constexpr (!COLPAR) {
    if (wid == 0 && lane_ok) {
      double logdet = 0.0;
      int fail = 0;
#pragma unroll
      for (int c = 0; c < I; c++) {
        double v[I];
#pragma unroll
        for (int k = 0; k <= c; k++) {
          v[k] = smt[pk(k, c) * TILE];
          if (!(fabs(v[k]) <= PGBP_EPS)) nz = true;
        }
#pragma unroll
        for (int k = 0; k < c; k++) {
          const double u = v[k] * rinv[k];
          v[k] = u;
          smt[pk(k, c) * TILE] = u;
#pragma unroll
          for (int r = k + 1; r <= c; r++) v[r] = nfma(r == c ? u : smt[pk(k, r) * TILE], u, v[r]);
        }
        const double d = v[c];
        if (!(d > 0.0) && fail == 0) fail = c + 1;  // LAPACK potrf info (also NaN); reported below
        logdet += log(d);
        rinv[c] = 1.0 / sqrt(d);
        smt[pk(c, c) * TILE] = rinv[c];
      }
      s_logdet[0] = logdet;
      s_flag[TILE + tid] = fail;
    }
    __syncthreads();
    if (lane_ok) {
#pragma unroll
      for (int k = 0; k < I; k++) rinv[k] = smt[pk(k, k) * TILE];
    }
  } else {
    double logdet = 0.0;
    int fail = 0;
    if (lane_ok)  // "all zero" test on the original entries of this warp's columns (src/beliefupdates.jl:62-66)
      for (int c = wid; c < I; c += NW)
        for (int k = 0; k <= c; k++)
          if (!(fabs(smt[(tri(c) + k) * TILE]) <= PGBP_EPS)) nz = true;
#pragma unroll
    for (int k = 0; k < I; k++) {
      double d = 1.0;
      if (lane_ok) d = smt[pk(k, k) * TILE];  // final: every update of steps < k is behind the barrier
      if (!(d > 0.0) && fail == 0) fail = k + 1;  // LAPACK potrf info (also NaN); reported below
      if (wid == 0) logdet += log(d);
      const double ri = 1.0 / sqrt(d);
      rinv[k] = ri;
      if (lane_ok) {
        const int c0 = k + 1 + ((wid - (k + 1)) % NW + NW) % NW;  // first column > k owned by this warp
        for (int c = c0; c < I; c += NW) {
          const int tc = tri(c);
          const double ukc = smt[(tc + k) * TILE] * ri;
          // operands of 8 rows loaded before the first store: the compiler cannot move a shared-memory load above
          // a store it cannot disambiguate, and one row per iteration exposed the full LDS latency every time
          for (int r0 = k + 1; r0 <= c; r0 += 8) {
            double ur[8], av[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
              const int r = r0 + u;
              if (r <= c) {
                ur[u] = smt[(tri(r) + k) * TILE];
                av[u] = smt[(tc + r) * TILE];
              }
            }
#pragma unroll
            for (int u = 0; u < 8; u++) {
              const int r = r0 + u;
              if (r <= c) smt[(tc + r) * TILE] = nfma(ur[u] * ri, ukc, av[u]);
            }
          }
        }
      }
      __syncthreads();
    }
    if (lane_ok) {  // scale the rows in place: U(k,c) = A(k,c) / sqrt(A(k,k))
      for (int c = wid; c < I; c += NW) {
        const int tc = tri(c);
#pragma unroll
        for (int k = 0; k < I; k++)
          if (k < c) smt[(tc + k) * TILE] *= rinv[k];
      }
      if (wid == 0) {
        s_logdet[0] = logdet;
        s_flag[TILE + tid] = fail;
      }
    }
    __syncthreads();
  }

  // ---- B2: Z = U^-T [J_IK | h_I], right-hand sides dealt to the warps ---------------------------
  if (lane_ok) {
    for (int c0 = wid; c0 < nrhs; c0 += NW) {
      double* z0 = Z + c0 * I * TILE;
      double v0[I];
#pragma unroll
      for (int k = 0; k < I; k++) {
        v0[k] = z0[k * TILE];
        if (!(fabs(v0[k]) <= PGBP_EPS)) nz = true;
      }
#pragma unroll
      for (int k = 0; k < I; k++) {
        const double u0 = v0[k] * rinv[k];
        v0[k] = u0;
#pragma unroll
        for (int r = k + 1; r < I; r++) v0[r] = nfma(smt[pk(k, r) * TILE], u0, v0[r]);
      }
#pragma unroll
      for (int k = 0; k < I; k++) z0[k * TILE] = v0[k];
      if (c0 == S) {  // the h column: w = U^-T h_I
        double ww = 0.0;
#pragma unroll
        for (int k = 0; k < I; k++) ww = fma(v0[k], v0[k], ww);
        s_ww[0] = ww;
      }
    }
    s_flag[(2 + wid) * TILE + tid] = nz ? 1 : 0;
  }
  __syncthreads();
  bool nzall = false;
  int fail = 0;
  if (lane_ok) {
#pragma unroll
    for (int w = 0; w < NW; w++) nzall = nzall || s_flag[(2 + w) * TILE + tid] != 0;
    fail = s_flag[TILE + tid];
  }
  const bool dead = !active || (nzall && fail != 0);
  if (lane_ok) {
    if (nzall) {
      if (fail && active && wid == 0) status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, fail));
      if (wid == 0) g += 0.5 * ((double)I * PGBP_LOG2PI - s_logdet[0] + s_ww[0]);
    } else {  // "missing data" shortcut: message = (h_K, J_KK, g) unchanged
      for (int q = wid; q < nrhs * I; q += NW) Z[q * TILE] = 0.0;
    }
  }
  __syncthreads();  // the last read of U (B2) is behind this barrier: phase C reads Z only

  // ---- C: stream the kept block, kept columns paired (j, S-1-j) and dealt to the warps ------------
  double maxJ = 0.0, maxh = 0.0;
  const int half = (S + 1) / 2;
  for (int j = wid; j < half && !dead; j += NW) {
    for (int side = 0; side < 2; side++) {
      const int cc = side == 0 ? j : S - 1 - j;
      if (side == 1 && cc == j) break;
      ks.column(cc, maxJ);
    }
  }
  // h part: chunks of kept entries dealt to the warps, last warp first (it has the lightest J share)
  if (!dead) ks.hpart((NW - 1 - wid) * PGBP_CHUNK, NW * PGBP_CHUNK, maxh);
  if (lane_ok) {
    s_redJ[wid * TILE] = maxJ;
    s_redh[wid * TILE] = maxh;
  }
  __syncthreads();
  if (wid == 0 && !dead) {
    double mJ = 0.0, mh = 0.0;
#pragma unroll
    for (int w = 0; w < NW; w++) {  // NaN-propagating maximum, like absmax
      const double xj = s_redJ[w * TILE], xh = s_redh[w * TILE];
      if (xj > mJ || xj != xj) mJ = xj;
      if (xh > mh || xh != xh) mh = xh;
    }
    *slot_ptr(stb, (uint32_t)md.sg, ld8) = g;
    *slot_ptr(stb, (uint32_t)md.tg, ld8) = tg_old + (g - sg_old);
    store_flag(a, md.dmsg, e, S, mJ, mh);
  }
}

#endif  // !PGBP_HOST_EMUL

}  // namespace pgbp
