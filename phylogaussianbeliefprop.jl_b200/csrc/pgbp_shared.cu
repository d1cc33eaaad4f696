// Shared-precision batches: message passing in two kernels (SURVEY.md section 8f-1).
//
// In the reference only h and g of a message depend on the data (src/beliefupdates.jl:77-81): trait replicates under
// one parameter vector have the same J in every belief at every step.  A shared-precision batch therefore keeps the
// J rows once per GROUP (pgbp_batch::jb: an ordinary batch with one element per group) and only h, g per element
// (compact rows, pgbp_internal.h).  One message F -> T through sepset S is then
//
//   k_jmsg  one WARP per (message, group): gathers J_F in [I;K] order into shared memory, right-looking U'U of the
//           integrated block, Schur complement, divide / multiply / residual / flag of the J part, and leaves the
//           factor record   [info | logdet | 1/U_kk (I) | rows k < I of the scaled factor: U_k,k+1.. and Z_k,.]
//           in the traversal's cache;
//   k_hmsg  one THREAD per (message, element): w = U^-T h_I by forward substitution with the cached rows,
//           h_K - Z'w, g + (I log 2pi - logdet + w'w)/2, divide / multiply / residual / flag of the h part.
//
// Per element and message only 8 (m_F + 1 + 4 (s + 1) + s) bytes move and I^2/2 + I S fused multiply-adds are spent
// instead of the I^3/3 + .. of the factorisation.  Every entry sees the same operations in the same order as in the
// register kernels (message_thread_t0): results are bit-identical to an ordinary batch given the same inputs
// (tests/test_parity.py::test_shared_precision_batch_is_bit_identical).
#include <algorithm>

#include "pgbp_bulk.cuh"
#include "pgbp_kernels.cuh"
#include "pgbp_launch.h"
#include "pgbp_shapes.h"

namespace pgbp {

template <class T>
static int salloc(pgbp_batch* b, T** p, size_t n) {
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, std::max<size_t>(1, n) * sizeof(T)));
  *p = (T*)v;
  b->device_bytes += (int64_t)(n * sizeof(T));
  return 0;
}

struct JArgs {
  const MsgDesc* msgs;       // plan numbering (the group batch's own descriptors)
  const int32_t* tab;
  double* state;             // group batch: J rows live here
  double* resid;             // may be null
  uint8_t* calflag;          // may be null: J part of the calibration flags
  int32_t* status;           // per group
  int64_t ld, G;
  double* cache;             // [G][stride]
  const int64_t* cache_off;  // per message of the launch's descriptor array
  int64_t stride;
  uint32_t opts;
  int32_t ref_base;
};

struct HArgs {
  const MsgDesc* msgs;       // h / g rows remapped to the compact element numbering
  const int32_t* tab;
  double* state;             // element array: h, g rows
  double* resid;             // may be null (dh rows)
  uint8_t* calflag;          // may be null: h part of the calibration flags
  int32_t* status;           // per element
  int64_t B, ld, gs;
  const double* cache;
  const int64_t* cache_off;
  int64_t stride;
  uint32_t opts;
  int32_t ref_base;
};

PGBP_HD int64_t jrec_len(int I, int S) { return I == 0 ? 0 : 2 + I + (int64_t)I * (I + S) - (int64_t)I * (I + 1) / 2; }

// record slot of the single-message path (pgbp_propagate): any shape, whole 128-byte lines
static int64_t jrec_one_len() { return (jrec_len(PGBP_MAX_DIM, 0) + (int64_t)PGBP_MAX_DIM * PGBP_MAX_DIM + 31) / 16 * 16; }

// the lanes that share one (message, group): a warp on the device, a single "lane" in the host emulation
struct OneLane {
  static constexpr int n = 1;
  int lane = 0;
  PGBP_HD void sync() const {}
  PGBP_HD bool all(bool p) const { return p; }
  PGBP_HD double maxnan(double x) const { return x; }
};
#ifndef PGBP_HOST_EMUL
struct WarpLanes {
  static constexpr int n = 32;
  int lane;
  __device__ void sync() const { __syncwarp(); }
  __device__ bool all(bool p) const { return __all_sync(0xffffffffu, p); }
  __device__ double maxnan(double x) const {  // NaN-propagating maximum over the warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double y = __shfl_xor_sync(0xffffffffu, x, o);
      x = (x != x || y != y) ? NAN : (y > x ? y : x);
    }
    return x;
  }
};
// a whole block of NT threads on one (message, group): large matrices (the factorisation of a 48 x 48 belief is a
// chain of 32 dependent rank-1 updates: the more lanes per update, the shorter the chain)
template <int NT>
struct BlockLanes {
  static constexpr int n = NT;
  int lane;
  double* red;  // NT / 32 doubles of shared memory
  __device__ void sync() const { __syncthreads(); }
  __device__ bool all(bool p) const { return __syncthreads_and(p) != 0; }
  __device__ double maxnan(double x) const {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double y = __shfl_xor_sync(0xffffffffu, x, o);
      x = (x != x || y != y) ? NAN : (y > x ? y : x);
    }
    if ((lane & 31) == 0) red[lane >> 5] = x;
    __syncthreads();
    double m = red[0];
#pragma unroll
    for (int k = 1; k < NT / 32; k++) {
      const double y = red[k];
      m = (m != m || y != y) ? NAN : (y > m ? y : m);
    }
    __syncthreads();
    return m;
  }
};
#endif

// (row, column) of packed index q = c(c+1)/2 + r, q < nq, two bytes per entry
template <class W>
PGBP_HD void fill_rc(uint8_t* rc, int nq, const W& w) {
  for (int q = w.lane; q < nq; q += W::n) {
    int c = (int)((sqrt(8.0 * (double)q + 1.0) - 1.0) * 0.5);
    while ((c + 1) * (c + 2) / 2 <= q) c++;
    while (c * (c + 1) / 2 > q) c--;
    rc[2 * q] = (uint8_t)(q - c * (c + 1) / 2);
    rc[2 * q + 1] = (uint8_t)c;
  }
}

// J part of one message for one group.  A: tri(mF) doubles shared by the lanes; rc: the (row, column) table of
// fill_rc for at least tri(mF) entries.
template <class W>
PGBP_HD void jmsg_body(const JArgs& a, int mi, int64_t g, const W& w, double* A, const uint8_t* rc) {
  const MsgDesc md = a.msgs[mi];
  if (a.status[g] != 0) return;  // the group failed earlier: its J stops moving (uniform over the lanes)
  const int I = md.mF - md.s, S = md.s, M = md.mF;
  const int SM = tri(M);
  const int64_t ld = a.ld;
  double* st = a.state + g;
  const int32_t* __restrict__ gat = a.tab + md.gat;
  const int32_t* __restrict__ sca = a.tab + md.sca;
  double* rec = I > 0 ? a.cache + g * a.stride + a.cache_off[mi] : nullptr;
  for (int q0 = w.lane; q0 < SM; q0 += 4 * W::n) {  // four independent (table, entry) load pairs in flight per lane
    double v[4];
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (q0 + j * W::n < SM) v[j] = st[(md.fJ + gat[q0 + j * W::n]) * ld];
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (q0 + j * W::n < SM) A[q0 + j * W::n] = v[j];
  }
  w.sync();
  if (I > 0) {
    bool z = true;  // "Ji = Jki = 0", src/beliefupdates.jl:62-66 (the h_I part of the test is the elements')
    for (int c = 0; c < M; c++) {
      const int rmax = c < I ? c + 1 : I;
      for (int r = w.lane; r < rmax; r += W::n)
        if (!(fabs(A[pk(r, c)]) <= PGBP_EPS)) z = false;
    }
    if (!w.all(z)) {
      double logdet = 0.0;
      for (int k = 0; k < I; k++) {
        const double d = A[pk(k, k)];
        if (!(d > 0.0)) {  // LAPACK potrf: info = k+1 (also catches NaN); every element of the group fails here
          if (w.lane == 0) {
            status_fail(a.status, g, PGBP_STATUS(a.ref_base + md.ref, k + 1));
            rec[0] = (double)(k + 1);
          }
          return;
        }
        logdet += log(d);
        const double rinv = 1.0 / sqrt(d);
        for (int c = k + 1 + w.lane; c < M; c += W::n) A[pk(k, c)] *= rinv;
        if (w.lane == 0) rec[2 + k] = rinv;
        w.sync();
        // trailing update, one entry per lane and pass: A[r,c] -= A[k,r] A[k,c] for k < r <= c
        for (int q = pk(k + 1, k + 1) + w.lane; q < SM; q += W::n) {
          const int r = rc[2 * q], c = rc[2 * q + 1];
          if (r > k) A[q] = nfma(A[pk(k, r)], A[pk(k, c)], A[q]);
        }
        w.sync();
      }
      if (w.lane == 0) { rec[0] = 0.0; rec[1] = logdet; }
      int64_t off = 2 + I;
      for (int k = 0; k < I; k++) {
        for (int c = k + 1 + w.lane; c < M; c += W::n) rec[off + (c - k - 1)] = A[pk(k, c)];
        off += M - 1 - k;
      }
    } else if (w.lane == 0) {
      rec[0] = -1.0;  // shortcut: the message is (J_KK, h_K, g) as they are
    }
  }
  // divide! / mult! / residual of the J part (src/beliefupdates.jl:579-587, 483-488, 646-647)
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;  // lazy sepset zero: the old sepset value is 0, not loaded
  double* rs = a.resid ? a.resid + g : nullptr;
  double maxJ = 0.0;
  // (flattened over the packed entries: one pass of dependent global round trips per W::n entries instead of one per
  // column -- on narrow levels these round trips ARE the group pass: C2S spent 17 us per level here)
  for (int q = w.lane; q < tri(S); q += W::n) {
    const int r = rc[2 * q], c = rc[2 * q + 1];
    const double nv = A[pk(I + r, I + c)];
    double* sp = st + (md.sJ + q) * ld;
    double* tp = st + (md.tJ + sca[q]) * ld;
    const double d = nv - (sz ? 0.0 : *sp);
    *sp = nv;
    *tp = *tp + d;
    if (rs) rs[(md.rJ + q) * ld] = d;
    absmax(maxJ, d);
  }
  maxJ = w.maxnan(maxJ);
  if (w.lane == 0 && (a.opts & PGBP_CAL_RESIDNORM) && a.calflag)
    a.calflag[(int64_t)md.dmsg * ld + g] = (S > 0 ? (maxJ / (double)S <= 1e-5) : true) ? 1 : 0;
}

// Every slot row the element pass of a message (I, S), M = I + S, reads, numbered in one fixed order: sender h in [I;K]
// order [0, TH), receiver h at the sepset's positions [TH, FG), sender g, receiver g, then the old sepset g and h
// [SG, N).  The sepset rows come last because they are not read under PGBP_OPT_SEPZERO: k_hmsg_bulk then stages the
// first SG rows only.
struct HRows {
  int TH, FG, TG, SG, SH, N;
  PGBP_HD HRows(int M, int S) : TH(M), FG(M + S), TG(M + S + 1), SG(M + S + 2), SH(M + S + 3), N(M + 2 * S + 3) {}
  PGBP_HD uint32_t slot(const MsgDesc& md, const int32_t* __restrict__ gat, const int32_t* __restrict__ sca, int n) const {
    if (n < TH) return (uint32_t)md.fh + (uint32_t)gat[n];
    if (n < FG) return (uint32_t)md.th + (uint32_t)sca[n - TH];
    if (n == FG) return (uint32_t)md.fg;
    if (n == TG) return (uint32_t)md.tg;
    if (n == SG) return (uint32_t)md.sg;
    return (uint32_t)md.sh + (uint32_t)(n - SH);
  }
};

// Operand sources of hmsg_body: fslot(k) and tslot(k) are the slots of rows k and TH + k (HRows numbering),
// at(n, slot) the value of row n for this element, rec the group's factor record.  HTab reads the state array through
// the index tables, with tables and record in global memory (host emulation, k_hwalk, k_hmsg) or staged in shared
// memory by k_hmsg; HBulk reads every row from k_hmsg_bulk's tile.  ahead: the old sepset and receiver values of a
// chunk are loaded with the sender's before its arithmetic (global memory: 3 CH loads in flight), not at the stores
// (shared memory: nothing held across the arithmetic -- loaded ahead, k_hmsg_bulk<16> took 9 % longer on one B200).
struct HTab {
  static constexpr bool ahead = true;
  uint32_t fh, th;
  const int32_t* __restrict__ gat;  // sender positions of [I;K]
  const int32_t* __restrict__ sca;  // receiver positions of the sepset's variables
  const double* __restrict__ rec;
  char* st;
  uint32_t ld8;
  PGBP_HD uint32_t fslot(int k) const { return fh + (uint32_t)gat[k]; }
  PGBP_HD uint32_t tslot(int k) const { return th + (uint32_t)sca[k]; }
  PGBP_HD double at(int, uint32_t s) const { return *slot_ptr(st, s, ld8); }
};

// h, g part of one message for one element whose status is 0.  CI >= 0: compile-time integrated dimension (w in
// registers); CI < 0: runtime (thread-local array).
// CH: kept entries per streaming chunk (3 CH loads in flight per thread).  Measured on B200 for the thread-per-element
// kernels: CH = 4 beats CH = 8 (254 registers): c5s 4,801 vs 4,227 calibrations/s, c2s 137.7 vs 130.9 M/s at that
// stage; with CH = 4 k_hmsg is capped at 128 registers for I <= 16 (4 blocks per SM: 166.5 ms per C5S step against
// 178.6 with 3 and 194.0 with 5).  k_hmsg_bulk reads its operands from shared memory and takes CH = 8.
template <int CI, int CH, class Src>
PGBP_HD void hmsg_body(const HArgs& a, const MsgDesc& md, int64_t e, const Src& src) {
  const int S = md.s;
  const int I = CI >= 0 ? CI : md.mF - S, M = I + S;
  const HRows R(M, S);
  const uint32_t ld8 = (uint32_t)(a.ld * 8);
  char* st = (char*)(a.state + e);
  char* rs = a.resid ? (char*)(a.resid + e) : nullptr;
  const uint32_t sh = (uint32_t)md.sh, rh = (uint32_t)md.rh;
  const uint32_t sg = (uint32_t)md.sg, tg = (uint32_t)md.tg;
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;  // lazy sepset zero: old sepset h, g are 0, not loaded
  double g = src.at(R.FG, (uint32_t)md.fg);
  const double sg_old = sz ? 0.0 : src.at(R.SG, sg), tg_old = src.at(R.TG, tg);
  double hI[CI > 0 ? CI : (CI == 0 ? 1 : PGBP_MAX_DIM)];
  const double* __restrict__ rec = src.rec;
  bool zeroZ = true;
  if (I > 0) {
#pragma unroll
    for (int k = 0; k < I; k++) hI[k] = src.at(k, src.fslot(k));
    const double info = rec[0];
    if (info > 0.0) {  // the factorisation of the group's J_I failed at this pivot
      status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, (int)info));
      return;
    }
    if (info < 0.0) {  // J_I = J_IK = 0: the message is the kept part unchanged -- if this element's h_I is 0 too
      bool hz = true;
#pragma unroll
      for (int k = 0; k < I; k++)
        if (!(fabs(hI[k]) <= PGBP_EPS)) hz = false;
      if (!hz) {  // the reference would factorise a zero matrix here
        status_fail(a.status, e, PGBP_STATUS(a.ref_base + md.ref, 1));
        return;
      }
    } else {
      zeroZ = false;
      double ww = 0.0;
      const double* row = rec + 2 + I;
#pragma unroll
      for (int k = 0; k < I; k++) {
        const double wk = hI[k] * rec[2 + k];
        hI[k] = wk;
        ww = fma(wk, wk, ww);
#pragma unroll
        for (int c = k + 1; c < I; c++) hI[c] = nfma(row[c - k - 1], wk, hI[c]);
        row += M - 1 - k;
      }
      g += 0.5 * ((double)I * PGBP_LOG2PI - rec[1] + ww);
    }
  }
  double maxh = 0.0;
  for (int k0 = 0; k0 < S; k0 += CH) {
    double nv[CH], so[CH], to[CH];
    uint32_t ta[CH];
    auto load_old = [&](int j) {  // receiver slot, old sepset and receiver values of kept entry k0 + j
      ta[j] = src.tslot(k0 + j);
      so[j] = sz ? 0.0 : src.at(R.SH + k0 + j, sh + k0 + j);
      to[j] = src.at(R.TH + k0 + j, ta[j]);
    };
#pragma unroll
    for (int j = 0; j < CH; j++)
      if (k0 + j < S) {
        nv[j] = src.at(I + k0 + j, src.fslot(I + k0 + j));
        if constexpr (Src::ahead) load_old(j);
      }
    if (!zeroZ) {
      const double* row = rec + 2 + I;
#pragma unroll
      for (int i = 0; i < I; i++) {
        const double wi = hI[i];
#pragma unroll
        for (int j = 0; j < CH; j++)
          if (k0 + j < S) nv[j] = nfma(row[(I - 1 - i) + k0 + j], wi, nv[j]);
        row += M - 1 - i;
      }
    }
#pragma unroll
    for (int j = 0; j < CH; j++)
      if (k0 + j < S) {
        if constexpr (!Src::ahead) load_old(j);
        const double d = nv[j] - so[j];
        *slot_ptr(st, sh + k0 + j, ld8) = nv[j];
        *slot_ptr(st, ta[j], ld8) = to[j] + d;
        if (rs) *slot_ptr(rs, rh + k0 + j, ld8) = d;
        absmax(maxh, d);
      }
  }
  *slot_ptr(st, sg, ld8) = g;
  *slot_ptr(st, tg, ld8) = tg_old + (g - sg_old);
  if ((a.opts & PGBP_CAL_RESIDNORM) && a.calflag)
    a.calflag[(int64_t)md.dmsg * a.ld + e] = (S > 0 ? (maxh / sqrt((double)S) <= 1e-5) : true) ? 1 : 0;
}

// One (message, element) of the element pass with tables and record read from global memory.
template <int CI>
PGBP_HD void hmsg_thread(const HArgs& a, int mi, int64_t e) {
  const MsgDesc& md = a.msgs[mi];  // only the fields used are loaded; rows fit 32 bits (checked at creation)
  if (a.status[e] != 0) return;
  const int S = md.s, M = CI >= 0 ? CI + S : md.mF;
  const double* rec = M > S ? a.cache + (e / a.gs) * a.stride + a.cache_off[mi] : nullptr;
  hmsg_body<CI, 4>(a, md, e, HTab{(uint32_t)md.fh, (uint32_t)md.th, a.tab + md.gat + tri(M), a.tab + md.sca + tri(S), rec,
                                   (char*)(a.state + e), (uint32_t)(a.ld * 8)});
}

#ifndef PGBP_HOST_EMUL
// dynamic shared memory: tri(maxM)+1 doubles | NT/32 doubles (reduction) | 2 tri(maxM) bytes ((row, column) table)
template <int NT>
__global__ void __launch_bounds__(NT) k_jmsg(JArgs a, int maxM) {
  extern __shared__ double jA[];
  const int nq = tri(maxM);
  double* red = jA + nq + 1;
  uint8_t* rc = (uint8_t*)(red + NT / 32);
  if constexpr (NT == 32) {
    const WarpLanes w{(int)threadIdx.x};
    fill_rc(rc, nq, w);
    __syncwarp();
    for (int64_t g = blockIdx.y; g < a.G; g += gridDim.y) {
      jmsg_body(a, blockIdx.x, g, w, jA, rc);
      __syncwarp();
    }
  } else {
    const BlockLanes<NT> w{(int)threadIdx.x, red};
    fill_rc(rc, nq, w);
    __syncthreads();
    for (int64_t g = blockIdx.y; g < a.G; g += gridDim.y) {
      jmsg_body(a, blockIdx.x, g, w, jA, rc);
      __syncthreads();
    }
  }
}
// reclen > 0: every message of the launch has a factor record of `reclen` doubles; when the block's 128 elements
// belong to ONE group the record is staged in shared memory once (coalesced) and read from there (broadcast LDS)
// instead of ~I (I + 2S) / 2 dependent global loads per thread.
#ifndef PGBP_HMSG_MINB
#define PGBP_HMSG_MINB 4  // resident blocks per SM of the element pass for I <= 16 (register cap 128)
#endif
template <int CI>
__global__ void __launch_bounds__(128, (CI >= 0 && CI <= 16 ? PGBP_HMSG_MINB : 3)) k_hmsg(HArgs a, int reclen) {
  extern __shared__ double srec[];
  const int64_t e0 = (int64_t)blockIdx.x * blockDim.x;
  const int64_t e = e0 + threadIdx.x;
  bool staged = false;
  if (CI != 0 && reclen > 0) {
    const int64_t elast = (e0 + blockDim.x - 1 < a.B ? e0 + blockDim.x - 1 : a.B - 1);
    if (e0 / a.gs == elast / a.gs) {  // uniform over the block
      const MsgDesc& md = a.msgs[blockIdx.y];
      const int S = md.s, M = md.mF;
      const double* src = a.cache + (e0 / a.gs) * a.stride + a.cache_off[blockIdx.y];
      for (int q = threadIdx.x; q < reclen; q += blockDim.x) srec[q] = src[q];
      int32_t* stab = (int32_t*)(srec + reclen);
      const int32_t* gat = a.tab + md.gat + tri(M);
      const int32_t* sca = a.tab + md.sca + tri(S);
      for (int q = threadIdx.x; q < M + S; q += blockDim.x) stab[q] = q < M ? gat[q] : sca[q - M];
      __syncthreads();
      staged = true;
    }
  }
  if (e >= a.B) return;
  if (!staged) {
    hmsg_thread<CI>(a, blockIdx.y, e);
    return;
  }
  // record and tables through the shared window (LDS with immediate offsets), not through generic pointers
  const MsgDesc& md = a.msgs[blockIdx.y];
  if (a.status[e] != 0) return;
  const int32_t* stab = (const int32_t*)(srec + reclen);
  hmsg_body<CI, 4>(a, md, e, HTab{(uint32_t)md.fh, (uint32_t)md.th, stab, stab + md.mF, srec, (char*)(a.state + e),
                                  (uint32_t)(a.ld * 8)});
}

// Element pass with bulk-copy staging: the wide levels of big graphs (C5: 420k messages x 1,536 replicates) are a
// pure streaming problem -- 8 (m_F + 1 + 4 (s+1)) bytes and I^2/2 + I S FMAs per (message, element) -- and the
// thread-per-element kernel above keeps too few bytes in flight (12-16 warps per SM x ~14 loads each; ncu: long
// scoreboard 48 %, 2.8 TB/s).  Here a block of 128 threads owns 128 consecutive elements of ONE message: every slot
// row the message reads (h of the sender in [I;K] order, old sepset h, target h at the sepset's positions, the three
// g) is a contiguous 1 KB segment of the batch-innermost layout, so thread n issues ONE cp.async.bulk for row n, the
// factor record arrives by a bulk copy too, and all of them (67 rows = 69 KB for an (I,S) = (16,16) message) are in
// flight at once on one mbarrier, without holding a register.  Three blocks per SM keep ~200 KB in flight.  The
// arithmetic is hmsg_body with operands from shared memory (element = thread, conflict-free): bit-identical results.
struct HBulk {
  static constexpr bool ahead = false;
  const double* rec;
  const double* r;         // this element's column of the tile: row n at r[128 n]
  const uint32_t* sl;      // slot of every staged row
  int th;
  PGBP_HD uint32_t fslot(int k) const { return sl[k]; }
  PGBP_HD uint32_t tslot(int k) const { return sl[th + k]; }
  PGBP_HD double at(int n, uint32_t) const { return r[n * 128]; }
};
template <int CI>
__global__ void __launch_bounds__(128, (CI <= 16 ? 3 : 2)) k_hmsg_bulk(HArgs a, int reclen) {
  extern __shared__ __align__(128) double sm[];
  __shared__ __align__(8) unsigned long long mbar;
  const int tid = threadIdx.x;
  const MsgDesc& md = a.msgs[blockIdx.y];
  const int S = md.s, M = CI + S;
  const HRows R(M, S);
  const int nrows = (a.opts & PGBP_OPT_SEPZERO) ? R.SG : R.N;
  const int64_t e0 = (int64_t)blockIdx.x * 128, e = e0 + tid;
  const int64_t left = a.ld - e0;
  const uint32_t rowbytes = (uint32_t)(left < 128 ? left : 128) * 8u;
  const uint32_t ld8 = (uint32_t)(a.ld * 8);
  double* rows = sm + reclen;
  uint32_t* sslot = (uint32_t*)(rows + (size_t)nrows * 128);  // slot of every staged row
  if (tid == 0) {
    mbar_init(&mbar, 1);
    mbar_expect_tx(&mbar, (unsigned)reclen * 8u + (unsigned)nrows * rowbytes);
  }
  __syncthreads();
  const char* tileb = (const char*)(a.state + e0);
  if (tid == 0) bulk_g2s(sm, a.cache + (e0 / a.gs) * a.stride + a.cache_off[blockIdx.y], (unsigned)reclen * 8u, &mbar);
  {
    const int32_t* __restrict__ gat = a.tab + md.gat + tri(M);
    const int32_t* __restrict__ sca = a.tab + md.sca + tri(S);
    for (int n = tid; n < nrows; n += 128) {
      const uint32_t slot = R.slot(md, gat, sca, n);
      sslot[n] = slot;
      bulk_g2s(rows + (size_t)n * 128, tileb + (uint64_t)slot * (uint64_t)ld8, rowbytes, &mbar);
    }
  }
  const int32_t stat = e < a.B ? a.status[e] : 1;
  __syncthreads();       // sslot
  mbar_wait(&mbar, 0);   // every row and the record have landed (no thread leaves the block before that)
  if (stat != 0) return;
  hmsg_body<CI, 8>(a, md, e, HBulk{sm, rows + tid, sslot, M});
}
#endif

// ---------------------------------------------------------------------------------------------------------------
// Walk kernels: a RUN of consecutive narrow steps in ONE launch per pass.
// Deep schedules of narrow steps (loopy graphs, the thin ends of a clique tree's level order) spend their time in
// launch gaps and single-message latencies.  (C5's clique tree is not one of them: 62 + 45 steps, 21 of them <= 8
// messages wide -- its ~900 launches per pass are launch groups by shape; no measurable effect there.)  For a run of narrow
// steps the group pass becomes one block per group (8 warps, one message per warp, block barrier between steps) and
// the element pass one block per 128 elements that walks the run for ITS elements (elements are independent: no
// synchronisation between blocks).  The element pass of step s only needs the group pass of step s: the group walk
// publishes a per-(step, group) counter after each step (release), the element walk spins on it (acquire, bounded).
// The counters count executions, so a captured CUDA graph can be replayed: the element walk of execution k waits for
// counter >= k, k = its own per-traversal execution count kept on the device.
// Records are padded to whole 128-byte lines: a line never holds parts of two records, so reading a record after
// its flag cannot see a stale L1 line from an earlier read of its neighbour.
#define PGBP_SW_WIDE 8     // widest step (messages) of a walk run
#define PGBP_SW_MINRUN 8   // shortest run worth a walk launch
#ifndef PGBP_HOST_EMUL
__global__ void __launch_bounds__(32 * PGBP_SW_WIDE) k_jwalk(JArgs a, const int32_t* __restrict__ step_off, int s0, int s1,
                                                            unsigned* flags, int maxM) {
  extern __shared__ double jA[];
  const int nq = tri(maxM);
  const int warp = threadIdx.x >> 5;
  const WarpLanes w{(int)(threadIdx.x & 31)};
  uint8_t* rc = (uint8_t*)(jA + (size_t)PGBP_SW_WIDE * (nq + 1));
  double* A = jA + (size_t)warp * (nq + 1);
  if (warp == 0) fill_rc(rc, nq, w);
  __syncthreads();
  for (int64_t g = blockIdx.x; g < a.G; g += gridDim.x) {
    for (int s = s0; s < s1; s++) {
      const int first = step_off[s], end = step_off[s + 1];
      for (int m = first + warp; m < end; m += PGBP_SW_WIDE) {
        jmsg_body(a, m, g, w, A, rc);
        __syncwarp();
      }
      __syncthreads();  // the step's records and J rows are written (block scope) ...
      if (threadIdx.x == 0) {
        __threadfence();  // ... and visible device-wide before the counter moves
        atomicAdd(&flags[(int64_t)s * a.G + g], 1u);
      }
    }
  }
}

// (one out-of-line body per shape: inlined into one switch the nine small shapes cost 2 KB of spills and a 1 KB frame)
template <int CI>
__device__ __noinline__ void hmsg_call(const HArgs& a, int m, int64_t e) { hmsg_thread<CI>(a, m, e); }

// SMALL: every message of the run integrates at most 8 variables (C2-like graphs): exact small shapes, 128 registers,
// four resident blocks per SM; otherwise the I = 0 / 16 / 32 shapes of the p = 16 workloads at 255 registers.
template <bool SMALL>
__global__ void __launch_bounds__(128, (SMALL ? 4 : 1)) k_hwalk(HArgs a, const int32_t* __restrict__ step_off, int s0, int s1,
                                                  const unsigned* flags, unsigned* hcount, unsigned* done_blocks, int64_t G) {
  __shared__ unsigned need;
  __shared__ int timed_out;
  const int64_t e0 = (int64_t)blockIdx.x * blockDim.x;
  const int64_t e = e0 + threadIdx.x;
  const int64_t elast = (e0 + blockDim.x - 1 < a.B ? e0 + blockDim.x - 1 : a.B - 1);
  const int64_t g0 = e0 / a.gs, g1 = elast / a.gs;
  if (threadIdx.x == 0) { need = *(volatile unsigned*)hcount + 1u; timed_out = 0; }
  __syncthreads();
  for (int s = s0; s < s1; s++) {
    if (threadIdx.x == 0) {
      const long long t0 = clock64();
      for (int64_t g = g0; g <= g1; g++)
        while (*(volatile const unsigned*)&flags[(int64_t)s * G + g] < need) {
          if (clock64() - t0 > 6000000000LL) { timed_out = 1; break; }  // ~3 s: the group walk is lost
          __nanosleep(100);
        }
      __threadfence();
    }
    __syncthreads();
    if (timed_out) break;
    if (e < a.B) {
      const int first = step_off[s], end = step_off[s + 1];
      for (int m = first; m < end; m++) {
        const int I = a.msgs[m].mF - a.msgs[m].s;
        if constexpr (SMALL) {
          switch (I) {
            case 0: hmsg_call<0>(a, m, e); break;
            case 1: hmsg_call<1>(a, m, e); break;
            case 2: hmsg_call<2>(a, m, e); break;
            case 3: hmsg_call<3>(a, m, e); break;
            case 4: hmsg_call<4>(a, m, e); break;
            case 5: hmsg_call<5>(a, m, e); break;
            case 6: hmsg_call<6>(a, m, e); break;
            case 7: hmsg_call<7>(a, m, e); break;
            default: hmsg_call<8>(a, m, e); break;
          }
        } else {
          switch (I) {
            case 0: hmsg_call<0>(a, m, e); break;
            case 16: hmsg_thread<16>(a, m, e); break;
            case 32: hmsg_thread<32>(a, m, e); break;
            default: hmsg_thread<-1>(a, m, e); break;
          }
        }
      }
    }
  }
  if (timed_out && e < a.B) status_fail(a.status, e, PGBP_STATUS(0x7ffff8, 1));
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(done_blocks, 1u) == gridDim.x - 1) {  // last block of this execution
      *done_blocks = 0;
      __threadfence();
      atomicAdd(hcount, 1u);
    }
  }
}
#endif

static int launch_jmsg(pgbp_batch* b, JArgs a, int nmsg, int maxM, pgbp_stream_t stream) {
  int done = 0;
  while (done < nmsg) {
    const int n = std::min(nmsg - done, 1 << 30);
    JArgs c = a;
    c.msgs = a.msgs + done;
    c.cache_off = a.cache_off + done;
#ifdef PGBP_HOST_EMUL
    (void)stream;
    std::vector<double> A((size_t)tri(maxM) + 1);
    std::vector<uint8_t> rc(2 * (size_t)tri(maxM) + 2);
    fill_rc(rc.data(), tri(maxM), OneLane{});
    for (int m = 0; m < n; m++)
      for (int64_t g = 0; g < c.G; g++) jmsg_body(c, m, g, OneLane{}, A.data(), rc.data());
#else
    dim3 grid((unsigned)n, (unsigned)std::min<int64_t>(c.G, 65535));
    const size_t smem = sizeof(double) * (size_t)(tri(maxM) + 1 + 4) + 2 * (size_t)tri(maxM) + 8;
    // sender dimension >= 23: a 128-thread block per (message, group) shortens the chain of dependent rank-1 updates.
    // PGBP_JMSG_WIDE=n takes the one-warp kernel instead from n (message, group) pairs per launch upwards: 4.5k
    // instead of 29.5k warp instructions per 32 x 32 message, but measured no faster on C5's wide levels (138.9 vs
    // 137.1 ms per step) -- the group pass is bound by its scattered 8-byte accesses, not by instructions.
    const char* we = getenv("PGBP_JMSG_WIDE");  // (read per call: a test switches it)
    const int64_t wide = we ? atoll(we) : INT64_MAX;
    if (tri(maxM) >= 256 && (int64_t)n * c.G < wide) k_jmsg<128><<<grid, 128, smem, stream>>>(c, maxM);
    else k_jmsg<32><<<grid, 32, smem, stream>>>(c, maxM);
#endif
    b->launches++;
    PGBP_TRY(check_launch("k_jmsg"));
    done += n;
  }
  return 0;
}

template <int CI>
static int launch_hmsg_t(pgbp_batch* b, const HArgs& a, int nmsg, int reclen) {
#ifdef PGBP_HOST_EMUL
  (void)reclen;
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = 0; e < a.B; e++) hmsg_thread<CI>(a, m, e);
#else
  dim3 grid((unsigned)((a.B + 127) / 128), (unsigned)nmsg);
  if constexpr (CI == 8 || CI == 12 || CI == 16 || CI == 24 || CI == 32) {
    // bulk-copy staging (k_hmsg_bulk): every block of 128 elements inside one group, 16-byte aligned rows, one
    // message shape per launch (reclen > 0), and the rows of a message fit the shared memory of an SM
    if (reclen > 0 && (a.gs % 128 == 0 || a.gs >= a.B) && a.ld % 2 == 0 && a.B >= 64) {
      const int S = (int)((reclen - 2 - CI - (CI * (CI - 1)) / 2) / CI);  // jrec_len(I, S) solved for S
      const int reclen16 = (reclen + 15) / 16 * 16;
      const int nrows = CI + 3 * S + 3;
      const size_t smem = sizeof(double) * ((size_t)reclen16 + (size_t)nrows * 128) + sizeof(uint32_t) * (size_t)nrows;
      if (jrec_len(CI, S) == reclen && smem <= 100 * 1024) {
        static AttrOnce attr;  // per instantiation and device
        if (attr.first()) PGBP_CUDA(cudaFuncSetAttribute(k_hmsg_bulk<CI>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        k_hmsg_bulk<CI><<<grid, 128, smem, b->stream>>>(a, reclen16);
        b->launches++;
        return check_launch("k_hmsg_bulk");
      }
    }
  }
  if (reclen * 8 > 40 * 1024) reclen = 0;  // (records beyond the default dynamic shared memory: global loads)
  const size_t smem = reclen ? sizeof(double) * (size_t)reclen + sizeof(int32_t) * 2 * PGBP_MAX_DIM : 0;
  k_hmsg<CI><<<grid, 128, smem, b->stream>>>(a, reclen);
#endif
  b->launches++;
  return check_launch("k_hmsg");
}

// reclen: record length shared by every message of the launch (0: mixed shapes, no staging)
static int launch_hmsg(pgbp_batch* b, HArgs a, int nmsg, int I, int reclen) {
  int done = 0;
  while (done < nmsg) {
    const int n = std::min(nmsg - done, 65535);
    HArgs c = a;
    c.msgs = a.msgs + done;
    c.cache_off = a.cache_off + done;
    int rc;
    switch (I) {
#define PGBP_H_CASE(I_) case I_: rc = launch_hmsg_t<I_>(b, c, n, reclen); break;
      PGBP_H_CASE(0) PGBP_H_CASE(1) PGBP_H_CASE(2) PGBP_H_CASE(3) PGBP_H_CASE(4) PGBP_H_CASE(5) PGBP_H_CASE(6)
      PGBP_H_CASE(7) PGBP_H_CASE(8) PGBP_H_CASE(9) PGBP_H_CASE(10) PGBP_H_CASE(11) PGBP_H_CASE(12) PGBP_H_CASE(16)
      PGBP_H_CASE(24) PGBP_H_CASE(32)
#undef PGBP_H_CASE
      default: rc = launch_hmsg_t<-1>(b, c, n, reclen);
    }
    PGBP_TRY(rc);
    done += n;
  }
  return 0;
}

static JArgs make_jargs(pgbp_batch* b, uint32_t opts, int32_t ref_base) {
  pgbp_batch* jb = b->jb;
  JArgs a;
  a.msgs = nullptr;
  a.tab = jb->d_tab;
  a.state = jb->state;
  a.resid = jb->resid;
  a.calflag = jb->calflag;
  a.status = jb->status;
  a.ld = jb->ld;
  a.G = b->ngroups;
  a.cache = nullptr;
  a.cache_off = nullptr;
  a.stride = 0;
  a.opts = opts;
  a.ref_base = ref_base;
  return a;
}
static HArgs make_hargs(pgbp_batch* b, uint32_t opts, int32_t ref_base) {
  HArgs a;
  a.msgs = nullptr;
  a.tab = b->d_tab;
  a.state = b->state;
  a.resid = b->resid;
  a.calflag = b->calflag;
  a.status = b->status;
  a.B = b->B;
  a.ld = b->ld;
  a.gs = b->group_size;
  a.cache = nullptr;
  a.cache_off = nullptr;
  a.stride = 0;
  a.opts = opts;
  a.ref_base = ref_base;
  return a;
}

// the group batch runs on the element batch's stream (one stream, program order: group pass, element pass)
static void adopt_stream(pgbp_batch* b) { b->jb->stream = b->stream; }

int shared_run_traversal(pgbp_batch* b, int tree, int dir, uint32_t opts, int32_t ref_base) {
  const Traversal& tv = b->plan->trees[tree].trav[dir];
  const int td = 2 * tree + dir;
  if (tv.msgs.empty()) return 0;
  adopt_stream(b);
  JArgs ja = make_jargs(b, opts, ref_base);
  ja.msgs = b->jb->d_msgs[td];
  ja.cache = b->jcache[td];
  ja.cache_off = b->d_jcache_off[td];
  ja.stride = b->jcache_len[td];
  HArgs ha = make_hargs(b, opts, ref_base);
  ha.cache = b->jcache[td];
  ha.stride = b->jcache_len[td];
  pgbp_stream_t js = b->stream;
#ifndef PGBP_HOST_EMUL
  // Group pass on its own stream: fork after everything already enqueued on the batch's stream (assignment,
  // regularisation, the previous traversal's group pass is ordered by the stream itself) and after the last
  // element pass that read this traversal's records.
  if (!b->jstream) PGBP_CUDA(cudaStreamCreateWithFlags(&b->jstream, cudaStreamNonBlocking));
  if (!b->jfork_event) { cudaEvent_t ev; PGBP_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)); b->jfork_event = (void*)ev; }
  while ((int)b->jstep_events.size() < tv.nsteps) {
    cudaEvent_t ev;
    PGBP_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    b->jstep_events.push_back((void*)ev);
  }
  if (b->jcache_free.size() < b->jcache.size()) b->jcache_free.resize(b->jcache.size(), nullptr);
  if (b->jcache_used.size() < b->jcache.size()) b->jcache_used.resize(b->jcache.size(), 0);
  js = b->jstream;
  // update_residualkldiv reads the sepset's J and the residual's dJ from the group batch AFTER the element pass of
  // the message: the next traversal's group pass must not have overwritten them -- no running ahead across traversals
  if (opts & PGBP_CAL_RESIDKLDIV) b->jfork_pending = true;
  if (b->jfork_pending) {  // first traversal of a calibrate! call: after the work already enqueued on the batch's stream
    PGBP_CUDA(cudaEventRecord((cudaEvent_t)b->jfork_event, b->stream));
    PGBP_CUDA(cudaStreamWaitEvent(js, (cudaEvent_t)b->jfork_event, 0));
    b->jfork_pending = false;
    b->jcache_used.assign(b->jcache.size(), 0);  // the fork orders this call after every earlier element pass
  }
  // later traversals of the same call start as soon as the previous group pass is done (stream order): the group
  // pass runs ahead of the element pass -- except that it must not overwrite records still being read
  if (b->jcache_used[td]) PGBP_CUDA(cudaStreamWaitEvent(js, (cudaEvent_t)b->jcache_free[td], 0));  // (same call: same capture)
#endif
  // walk runs: maximal runs of >= PGBP_SW_MINRUN consecutive steps of <= PGBP_SW_WIDE messages (walk_end[s] = end of the
  // run starting at s, 0 elsewhere); only when the element walk leaves SMs free for the group walk it waits for
  std::vector<int> walk_end(tv.nsteps + 1, 0);
#ifndef PGBP_HOST_EMUL
  {
    // PGBP_SHARED_WALK: 0 = per-step launches only; default = walks where both run side by side (<= 64 element
    // blocks); 1 = also for larger batches, the element walk ordered behind the group walk's event -- measured on C2S
    // (65,536 replicates, 7 levels per direction): 0.62 ms per calibration against 0.42 ms with per-step launches
    // (one block walking 16 messages in sequence is slower than 16 launches that each fill the GPU), hence opt-in
    static const int walk_mode = [] { const char* e = getenv("PGBP_SHARED_WALK"); return e ? atoi(e) : 2; }();
    const bool walk_on = walk_mode == 1 || (walk_mode == 2 && (b->B + 127) / 128 <= 64);
    // (<= 64 element blocks: the two walks run side by side, the element walk spinning on the group walk's counters;
    // larger batches: the element walk is launched behind the group walk's event -- same kernels, nothing to spin on)
    const bool ok = walk_on && !(opts & PGBP_CAL_RESIDKLDIV) && b->ngroups <= 16;
    for (int s = 0; ok && s < tv.nsteps;) {
      int t = s;
      while (t < tv.nsteps && tv.step_off[t + 1] - tv.step_off[t] <= PGBP_SW_WIDE) t++;
      if (t - s >= PGBP_SW_MINRUN) walk_end[s] = t;
      s = t > s ? t : s + 1;
    }
    if (!b->d_walkflags.size()) { b->d_walkflags.assign(b->jcache.size(), nullptr); b->d_walkcount.assign(b->jcache.size(), nullptr); }
    if (!b->d_walkflags[td]) {
      PGBP_TRY(salloc(b, &b->d_walkflags[td], (size_t)tv.nsteps * (size_t)b->ngroups));
      PGBP_TRY(salloc(b, &b->d_walkcount[td], 2));
      PGBP_TRY(dev_memset(b->d_walkflags[td], 0, sizeof(unsigned) * (size_t)tv.nsteps * (size_t)b->ngroups, b->stream));
      PGBP_TRY(dev_memset(b->d_walkcount[td], 0, sizeof(unsigned) * 2, b->stream));
      PGBP_TRY(stream_sync(b->stream));
    }
  }
#endif
  // group pass: one launch per step (messages of a step touch disjoint beliefs), one launch per walk run
  for (int s = 0; s < tv.nsteps; s++) {
#ifndef PGBP_HOST_EMUL
    if (walk_end[s]) {
      const int s1 = walk_end[s];
      int maxM = 0;
      for (int k = tv.step_off[s]; k < tv.step_off[s1]; k++) maxM = std::max(maxM, tv.msgs[k].mF);
      const size_t smem = sizeof(double) * (size_t)PGBP_SW_WIDE * (size_t)(tri(maxM) + 1) + 2 * (size_t)tri(maxM) + 16;
      static AttrOnce attr_done;
      if (attr_done.first()) PGBP_CUDA(cudaFuncSetAttribute((const void*)k_jwalk, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
      k_jwalk<<<(unsigned)std::min<int64_t>(b->ngroups, 1024), 32 * PGBP_SW_WIDE, smem, js>>>(ja, b->jb->d_step_off[td], s, s1, b->d_walkflags[td], maxM);
      b->launches++;
      PGBP_TRY(check_launch("k_jwalk"));
      PGBP_CUDA(cudaEventRecord((cudaEvent_t)b->jstep_events[s1 - 1], js));
      s = s1 - 1;
      continue;
    }
#endif
    const int first = tv.step_off[s], count = tv.step_off[s + 1] - first;
    if (count > 0) {
      int maxM = 0;
      for (int k = first; k < first + count; k++) maxM = std::max(maxM, tv.msgs[k].mF);
      JArgs c = ja;
      c.msgs = ja.msgs + first;
      c.cache_off = ja.cache_off + first;
      PGBP_TRY(launch_jmsg(b, c, count, maxM, js));
    }
#ifndef PGBP_HOST_EMUL
    PGBP_CUDA(cudaEventRecord((cudaEvent_t)b->jstep_events[s], js));
#endif
  }
  // element pass: the plan's launch groups (same step, same shape class), each step after its records exist
  int waited = -1, walked_until = 0;
  for (const LaunchGroup& g : tv.groups) {
#ifndef PGBP_HOST_EMUL
    if (g.step < walked_until) continue;  // inside a run the element walk has been launched for
    if (walk_end[g.step]) {
      const int s1 = walk_end[g.step];
      HArgs c = ha;
      c.msgs = b->d_msgs[td];
      c.cache_off = b->d_jcache_off[td];
      const unsigned grid = (unsigned)((b->B + 127) / 128);
      if (grid > 64) {  // every SM may be taken by spinning blocks: order the element walk after the whole group walk
        PGBP_CUDA(cudaStreamWaitEvent(b->stream, (cudaEvent_t)b->jstep_events[s1 - 1], 0));
        waited = s1 - 1;
      }
      int maxI = 0;
      for (int k = tv.step_off[g.step]; k < tv.step_off[s1]; k++) maxI = std::max(maxI, tv.msgs[k].mF - tv.msgs[k].s);
#define PGBP_HWALK(SM_) k_hwalk<SM_><<<grid, 128, 0, b->stream>>>(c, b->jb->d_step_off[td], g.step, s1, b->d_walkflags[td], b->d_walkcount[td], b->d_walkcount[td] + 1, b->ngroups)
      if (maxI <= 8) PGBP_HWALK(true);
      else PGBP_HWALK(false);
#undef PGBP_HWALK
      b->launches++;
      PGBP_TRY(check_launch("k_hwalk"));
      walked_until = s1;
      continue;
    }
    if (g.step != waited) {
      PGBP_CUDA(cudaStreamWaitEvent(b->stream, (cudaEvent_t)b->jstep_events[g.step], 0));
      waited = g.step;
    }
#else
    (void)waited;
#endif
    HArgs c = ha;
    c.msgs = b->d_msgs[td] + g.first;
    c.cache_off = b->d_jcache_off[td] + g.first;
    const int gI = g.ci >= 0 ? g.ci : g.maxm;
    PGBP_TRY(launch_hmsg(b, c, g.count, gI, gI > 0 ? (int)jrec_len(gI, g.cs) : 0));
    if (opts & PGBP_CAL_RESIDKLDIV) {
      MsgArgs ma = make_args(b, opts, ref_base, false);
      PGBP_TRY(launch_kldiv(b, ma, b->d_msgs[td], g));
    }
  }
#ifndef PGBP_HOST_EMUL
  // join: whatever follows on the batch's stream (integrate, energies, the next assignment) sees the final J; the
  // last step's event was waited on above unless the traversal ended with copy-only steps
  if (waited != tv.nsteps - 1) PGBP_CUDA(cudaStreamWaitEvent(b->stream, (cudaEvent_t)b->jstep_events[tv.nsteps - 1], 0));
  if (!b->jcache_free[td]) { cudaEvent_t ev; PGBP_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)); b->jcache_free[td] = (void*)ev; }
  PGBP_CUDA(cudaEventRecord((cudaEvent_t)b->jcache_free[td], b->stream));  // this traversal's records may be overwritten after this
  b->jcache_used[td] = 1;
#endif
  return 0;
}

int shared_propagate(pgbp_batch* b, const MsgDesc& md_plan, uint32_t opts, int32_t ref_base) {
  adopt_stream(b);
  pgbp_batch* jb = b->jb;
  const MsgDesc mh = shared_remap(b, md_plan);
  PGBP_TRY(h2d(jb->d_one, &md_plan, sizeof(MsgDesc), b->stream));
  PGBP_TRY(h2d(b->d_one, &mh, sizeof(MsgDesc), b->stream));
  JArgs ja = make_jargs(b, b->jb->calflag ? opts : (opts & ~PGBP_CAL_RESIDNORM), ref_base);
  ja.msgs = jb->d_one;
  ja.cache = b->jcache_one;
  ja.cache_off = b->d_zero64;
  ja.stride = jrec_one_len();
  PGBP_TRY(launch_jmsg(b, ja, 1, md_plan.mF, b->stream));
  HArgs ha = make_hargs(b, b->calflag ? opts : (opts & ~PGBP_CAL_RESIDNORM), ref_base);
  ha.msgs = b->d_one;
  ha.cache = b->jcache_one;
  ha.cache_off = b->d_zero64;
  ha.stride = ja.stride;
  PGBP_TRY(launch_hmsg(b, ha, 1, md_plan.mF - md_plan.s, (int)jrec_len(md_plan.mF - md_plan.s, md_plan.s)));
  return stream_sync(b->stream);  // the descriptors are stack objects
}

MsgDesc shared_remap(const pgbp_batch* b, const MsgDesc& m) {
  const pgbp_plan* p = b->plan;
  auto belief_of = [&](int64_t hslot) {
    return (int)(std::lower_bound(p->hslot.begin(), p->hslot.end(), hslot) - p->hslot.begin());
  };
  const int f = belief_of(m.fh), s = belief_of(m.sh), t = belief_of(m.th);
  MsgDesc r = m;
  r.fh = b->eh[f]; r.fg = b->eh[f] + p->dim[f];
  r.sh = b->eh[s]; r.sg = b->eh[s] + p->dim[s];
  r.th = b->eh[t]; r.tg = b->eh[t] + p->dim[t];
  r.rh = b->erh[m.dmsg];
  return r;
}

// Element side of a shared-precision batch (the caller has set plan, B, ld, group_size, device, flags, stream):
// compact layout, descriptors, caches, and the group batch.
int shared_create(pgbp_batch* b) {
  const pgbp_plan* p = b->plan;
  b->ngroups = b->B / b->group_size;
  b->eh.resize(p->nbeliefs);
  int64_t row = 0;
  for (int i = 0; i < p->nbeliefs; i++) {
    if (i == p->nclusters) b->nrows_efactor = row;
    b->eh[i] = row;
    row += p->dim[i] + 1;
  }
  if (p->nsepsets == 0) b->nrows_efactor = row;
  b->nrows_e = row;
  b->erh.resize(2 * (size_t)p->nsepsets);
  row = 0;
  for (int d = 0; d < 2 * p->nsepsets; d++) { b->erh[d] = row; row += p->dim[p->nclusters + d / 2]; }
  b->nrows_eresid = row;
  const size_t ld = (size_t)b->ld;
  PGBP_TRY(salloc(b, &b->state, (size_t)b->nrows_e * ld));
  PGBP_TRY(dev_memset(b->state, 0, sizeof(double) * (size_t)b->nrows_e * ld, b->stream));
  if (b->flags & PGBP_BATCH_FACTORS) {
    PGBP_TRY(salloc(b, &b->factor, (size_t)b->nrows_efactor * ld));
    PGBP_TRY(dev_memset(b->factor, 0, sizeof(double) * (size_t)b->nrows_efactor * ld, b->stream));
  }
  if (b->flags & PGBP_BATCH_RESIDUALS) {
    const size_t nd = 2 * (size_t)p->nsepsets;
    PGBP_TRY(salloc(b, &b->resid, std::max<size_t>(1, (size_t)b->nrows_eresid) * ld));
    PGBP_TRY(dev_memset(b->resid, 0, sizeof(double) * std::max<size_t>(1, (size_t)b->nrows_eresid) * ld, b->stream));
    PGBP_TRY(salloc(b, &b->kldiv, std::max<size_t>(1, nd) * ld));
    PGBP_TRY(salloc(b, &b->calflag, std::max<size_t>(1, nd) * ld));
    PGBP_TRY(salloc(b, &b->iscal, ld));
    PGBP_TRY(salloc(b, &b->itertree, 2 * ld));
    PGBP_TRY(dev_memset(b->iscal, 0, sizeof(int32_t) * ld, b->stream));
    PGBP_TRY(dev_memset(b->itertree, 0, sizeof(int32_t) * 2 * ld, b->stream));
  }
  PGBP_TRY(salloc(b, &b->status, ld));
  PGBP_TRY(dev_memset(b->status, 0, sizeof(int32_t) * ld, b->stream));
  PGBP_TRY(salloc(b, &b->d_one, 1));
  PGBP_TRY(batch_upload_tables(b));
  // descriptors with compact h / g rows, record offsets and caches per traversal
  const size_t nt = p->trees.size();
  b->d_msgs.assign(2 * nt, nullptr);
  b->jcache.assign(2 * nt, nullptr);
  b->d_jcache_off.assign(2 * nt, nullptr);
  b->jcache_len.assign(2 * nt, 0);
  for (size_t t = 0; t < nt; t++)
    for (int dir = 0; dir < 2; dir++) {
      const Traversal& tv = p->trees[t].trav[dir];
      const size_t n = tv.msgs.size();
      std::vector<MsgDesc> rm(n);
      std::vector<int64_t> off(n + 1, 0);
      for (size_t k = 0; k < n; k++) {
        rm[k] = shared_remap(b, tv.msgs[k]);
        off[k + 1] = off[k] + (jrec_len(tv.msgs[k].mF - tv.msgs[k].s, tv.msgs[k].s) + 15) / 16 * 16;  // whole 128-byte lines
      }
      const size_t td = 2 * t + dir;
      PGBP_TRY(salloc(b, &b->d_msgs[td], n));
      PGBP_TRY(h2d(b->d_msgs[td], rm.data(), n * sizeof(MsgDesc), b->stream));
      PGBP_TRY(salloc(b, &b->d_jcache_off[td], n + 1));
      PGBP_TRY(h2d(b->d_jcache_off[td], off.data(), (n + 1) * sizeof(int64_t), b->stream));
      b->jcache_len[td] = off[n];
      PGBP_TRY(salloc(b, &b->jcache[td], (size_t)off[n] * (size_t)b->ngroups));
      PGBP_TRY(stream_sync(b->stream));  // rm / off are locals
    }
  PGBP_TRY(salloc(b, &b->jcache_one, (size_t)jrec_one_len() * (size_t)b->ngroups));
  PGBP_TRY(salloc(b, &b->d_zero64, 1));
  PGBP_TRY(dev_memset(b->d_zero64, 0, sizeof(int64_t), b->stream));
  return stream_sync(b->stream);
}

void shared_destroy(pgbp_batch* b) {
#ifndef PGBP_HOST_EMUL
  if (b->jstream) { cudaStreamSynchronize(b->jstream); cudaStreamDestroy(b->jstream); b->jstream = 0; }
  for (void* ev : b->jstep_events) cudaEventDestroy((cudaEvent_t)ev);
  for (void* ev : b->jcache_free) if (ev) cudaEventDestroy((cudaEvent_t)ev);
  if (b->jfork_event) cudaEventDestroy((cudaEvent_t)b->jfork_event);
  b->jstep_events.clear(); b->jcache_free.clear(); b->jfork_event = nullptr;
#endif
  for (auto* q : b->jcache) dev_free(q);
  for (auto* q : b->d_jcache_off) dev_free(q);
  for (auto* q : b->d_walkflags) dev_free(q);
  for (auto* q : b->d_walkcount) dev_free(q);
  dev_free(b->jcache_one);
  dev_free(b->d_zero64);
  dev_free(b->jucache);
  b->jucache = nullptr;
  if (b->jb) {
    b->jb->stream = 0;  // borrowed from the element batch
    b->jb->own_stream = false;
    pgbp_batch_destroy(b->jb);
    b->jb = nullptr;
  }
}

}  // namespace pgbp
