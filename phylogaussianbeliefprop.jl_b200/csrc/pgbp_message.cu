// K2 (message passing), K3 (integrate) and the calibrate! driver.
#include "pgbp_msg_t0.cuh"

using namespace pgbp;

namespace pgbp {

#ifndef PGBP_WALK_THREADS
#define PGBP_WALK_THREADS 128
#endif
#ifndef PGBP_WALK_MINBLOCKS
#define PGBP_WALK_MINBLOCKS 2
#endif

#ifndef PGBP_HOST_EMUL
__global__ void __launch_bounds__(256) k_message_copy(MsgArgs a) {
  const int64_t e = a.e0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.B) return;
  message_copy_thread(a, blockIdx.y, e);
}
#endif

// Walk kernel: one thread = one replicate walks the WHOLE message list of a
// calibration (postorder then preorder) in the reference's sequential order.
// Replicates are independent, so there is no inter-thread dependency at all:
// one launch per calibration, no per-message launch latency, and a belief
// written by message k is re-read by message k+1 from L1/L2 instead of HBM.
// Shapes are restricted to the trait-multiple family of pgbp_shapes.h so that
// every message still runs the register-resident specialised body.
template <int P, int A_, int B_>
PGBP_HD void walk_case(const MsgArgs& a, int m, int64_t e) {
  if constexpr (A_ == 0) message_copy_thread(a, m, e);
  else if constexpr ((A_ + B_) * P <= PGBP_T0_MAX) message_thread_t0<A_ * P, B_ * P>(a, m, e);
}
template <int P>
PGBP_HD void walk_thread(const MsgArgs& a, int nmsg, int64_t e) {
  if (a.status[e] != 0) return;
  if (a.done && a.done[e]) return;
  for (int m = 0; m < nmsg; m++) {
    switch (a.msgs[m].wid) {
      case 0: case 1: case 2: case 3: walk_case<P, 0, 0>(a, m, e); break;
      case 4: walk_case<P, 1, 0>(a, m, e); break;
      case 5: walk_case<P, 1, 1>(a, m, e); break;
      case 6: walk_case<P, 1, 2>(a, m, e); break;
      case 7: walk_case<P, 1, 3>(a, m, e); break;
      case 8: walk_case<P, 2, 0>(a, m, e); break;
      case 9: walk_case<P, 2, 1>(a, m, e); break;
      case 10: walk_case<P, 2, 2>(a, m, e); break;
      case 11: walk_case<P, 2, 3>(a, m, e); break;
      case 12: walk_case<P, 3, 0>(a, m, e); break;
      case 13: walk_case<P, 3, 1>(a, m, e); break;
      case 14: walk_case<P, 3, 2>(a, m, e); break;
      case 15: walk_case<P, 3, 3>(a, m, e); break;
      default: break;
    }
    if (a.status[e] != 0) return;  // first failed message stops the traversal (src/calibration.jl:129-131)
  }
}

// Tile-walk kernel: ONE launch for a run of consecutive steps of a deep, thin schedule of tiny messages
// (loopy BP on Bethe-type graphs: hundreds of steps of a few messages each, which per-step launches
// execute at ~9 us of pure latency apiece).  A block owns 32 elements (threadIdx.x) and LANES message
// lanes (threadIdx.y); it walks the steps in order, the lanes share the messages of a step, a block
// barrier separates the steps.  All threads that ever touch an element's beliefs are in the same block,
// so the block barrier (which also orders their global-memory accesses) is the only synchronisation: no
// launch per step, no grid-wide sync.  The walk is latency-bound per step, so everything is arranged to
// shorten the dependent chain of one message:
//  * descriptors are pre-resolved (TwDesc: slot numbers, no index-table indirection) and staged in shared
//    memory with cp.async ONE STAGE AHEAD (a stage = <= 64 messages of one step), double-buffered;
//  * a message issues ALL its loads (sender, old sepset, old receiver, status) before any arithmetic:
//    one HBM/L2 round trip per message instead of three;
//  * registers are capped (launch bounds) so that every block of the batch is resident at once.
// The arithmetic is message_body_t0<I,S> on the loaded values (I = 0 is the streaming copy): results are
// bit-identical to the per-step kernels by construction.

// Operand source of message_body_t0 in the tile walk: slots from the pre-resolved descriptor, values v[n] loaded
// by tilewalk_t0 before the body runs.
template <int I, int S>
struct T0Tile {
  using R = T0Rows<I, S>;
  const TwDesc& d;
  double v[R::N];
  PGBP_HD uint32_t slot(int n) const {
    if (n < R::FH) return d.fJ[n];
    if (n < R::FG) return d.fh[n - R::FH];
    if (n == R::FG) return d.fg;
    if (n == R::TG) return d.tg;
    if (n < R::TH) return d.tJ[n - R::TJ];
    if (n < R::SG) return d.th[n - R::TH];
    if (n == R::SG) return d.sg;
    return n < R::SH ? d.sJ + (uint32_t)(n - R::SJ) : d.sh + (uint32_t)(n - R::SH);
  }
  PGBP_HD double at(int n, uint32_t) const { return v[n]; }
};

// Loads in the order the body uses them (J_II, J_IK, h_I, g, then the kept entries with their old sepset and
// receiver values): in row order k_tilewalk spills 1,664 instead of 1,328 bytes at its 64-register cap.
template <int CI, int CS>
PGBP_HD void tilewalk_t0(const MsgArgs& a, const TwDesc& d, int64_t e) {
  constexpr int I = CI, S = CS, SS = S * (S + 1) / 2;
  using R = T0Rows<I, S>;
  const uint32_t ld8 = (uint32_t)(a.ld * 8);
  char* st = (char*)(a.state + e);
  const bool sz = (a.opts & PGBP_OPT_SEPZERO) != 0;  // the body does not read the old sepset then
  const int32_t stat = a.status[e];
  const uint8_t dn = a.done ? a.done[e] : (uint8_t)0;
  T0Tile<I, S> src{d, {}};
  auto load = [&](int n) { src.v[n] = *slot_ptr(st, src.slot(n), ld8); };
#pragma unroll
  for (int c = 0; c < I; c++) {
#pragma unroll
    for (int r = 0; r <= c; r++) load(R::FJ + pk(r, c));
  }
#pragma unroll
  for (int c = 0; c < S; c++) {
#pragma unroll
    for (int k = 0; k < I; k++) load(R::FJ + pk(k, I + c));
  }
#pragma unroll
  for (int k = 0; k < I; k++) load(R::FH + k);
  load(R::FG);
  if (!sz) load(R::SG);
  load(R::TG);
#pragma unroll
  for (int q = 0; q < SS; q++) {
    const int c = colof(q), r = q - c * (c + 1) / 2;
    load(R::FJ + pk(I + r, I + c));
    if (!sz) load(R::SJ + q);
    load(R::TJ + q);
  }
#pragma unroll
  for (int k = 0; k < S; k++) {
    load(R::FH + I + k);
    if (!sz) load(R::SH + k);
    load(R::TH + k);
  }
  if (stat != 0 || dn) return;
  message_body_t0<CI, CS>(a, d, e, src);
}

PGBP_HD void tilewalk_message(const MsgArgs& a, const TwDesc& d, int64_t e) {
  switch (d.shape) {
    case 0 * 8 + 0: tilewalk_t0<0, 0>(a, d, e); break;
    case 0 * 8 + 1: tilewalk_t0<0, 1>(a, d, e); break;
    case 0 * 8 + 2: tilewalk_t0<0, 2>(a, d, e); break;
    case 0 * 8 + 3: tilewalk_t0<0, 3>(a, d, e); break;
    case 0 * 8 + 4: tilewalk_t0<0, 4>(a, d, e); break;
    case 1 * 8 + 0: tilewalk_t0<1, 0>(a, d, e); break;
    case 1 * 8 + 1: tilewalk_t0<1, 1>(a, d, e); break;
    case 1 * 8 + 2: tilewalk_t0<1, 2>(a, d, e); break;
    case 1 * 8 + 3: tilewalk_t0<1, 3>(a, d, e); break;
    case 2 * 8 + 0: tilewalk_t0<2, 0>(a, d, e); break;
    case 2 * 8 + 1: tilewalk_t0<2, 1>(a, d, e); break;
    case 2 * 8 + 2: tilewalk_t0<2, 2>(a, d, e); break;
    case 3 * 8 + 0: tilewalk_t0<3, 0>(a, d, e); break;
    case 3 * 8 + 1: tilewalk_t0<3, 1>(a, d, e); break;
    case 4 * 8 + 0: tilewalk_t0<4, 0>(a, d, e); break;
    default: break;  // unreachable: use_tilewalk() admits sender dimensions <= 4 only
  }
}
#ifndef PGBP_HOST_EMUL
template <int P>
__global__ void __launch_bounds__(PGBP_WALK_THREADS, PGBP_WALK_MINBLOCKS) k_walk(MsgArgs a, int nmsg) {
  const int64_t e = a.e0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.B) return;
  walk_thread<P>(a, nmsg, e);
}

PGBP_D void cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem_src) : "memory");
}
PGBP_D void cp_async_commit_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory"); }

template <int LANES, int MINB>
__global__ void __launch_bounds__(32 * LANES, MINB) k_tilewalk(MsgArgs a, const TwDesc* __restrict__ descs,
                                                              const int32_t* __restrict__ stage_off, int k0, int k1) {
  __shared__ TwDesc buf[2][PGBP_TW_STAGE];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const int64_t e = a.e0 + (int64_t)blockIdx.x * 32 + threadIdx.x;
  const bool live = e < a.B;
  auto stage_load = [&](int m0, int m1, int which) {
    const uint4* src = reinterpret_cast<const uint4*>(descs + m0);
    uint4* dst = reinterpret_cast<uint4*>(&buf[which][0]);
    const int nch = (m1 - m0) * (int)(sizeof(TwDesc) / 16);
    for (int c = tid; c < nch; c += 32 * LANES) cp_async16(dst + c, src + c);
  };
  int m0 = stage_off[k0], m1 = stage_off[k0 + 1];
  stage_load(m0, m1, 0);
  for (int k = k0; k < k1; k++) {
    const int cur = (k - k0) & 1;
    const int m2 = (k + 1 < k1) ? stage_off[k + 2] : m1;  // end of the next stage
    cp_async_commit_wait_all();  // this thread's chunks of stage k have landed
    __syncthreads();             // stage k visible to all; every message of stage k-1 is complete
    if (k + 1 < k1) stage_load(m1, m2, cur ^ 1);  // overlaps the messages of stage k
    if (live) {
      const int n = m1 - m0;
      for (int j = threadIdx.y; j < n; j += LANES) tilewalk_message(a, buf[cur][j], e);
    }
    m0 = m1;
    m1 = m2;
  }
}

template <int MAXM>
__global__ void __launch_bounds__(128) k_message_ref(MsgArgs a) {
  const int64_t e = a.e0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.B) return;
  message_thread_ref<MAXM>(a, blockIdx.y, e);
}

template <int MAXM>
__global__ void __launch_bounds__(128) k_kldiv(MsgArgs a, double* kldiv, JSide js, JSide jr) {
  const int64_t e = a.e0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.B) return;
  kldiv_thread<MAXM>(a, kldiv, blockIdx.y, e, jcolumn(js, e), jcolumn(jr, e), js.ld);
}

template <int MAXM>
__global__ void __launch_bounds__(128) k_integrate(const double* state, int32_t* status, int64_t B, int64_t ld,
                                                   int64_t jslot, int64_t hslot, int64_t gslot, int M,
                                                   double* mu_soa, double* norm, int64_t ld_out, double* cov_soa,
                                                   JSide js) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  integrate_thread<MAXM>(state, status, ld, e, jslot, hslot, gslot, M, mu_soa, norm, ld_out, cov_soa, jcolumn(js, e), js.ld);
}
#endif

static int launch_copy(pgbp_batch* b, const MsgArgs& a, int nmsg) {
#ifdef PGBP_HOST_EMUL
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_copy_thread(a, m, e);
#else
  dim3 grid((unsigned)((a.B - a.e0 + 255) / 256), (unsigned)nmsg);
  k_message_copy<<<grid, 256, 0, b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message_copy");
}

// reference-order validation mode (PGBP_CAL_REFORDER): every message with something to integrate out goes
// through message_thread_ref
template <int MAXM>
static int launch_ref_t(pgbp_batch* b, const MsgArgs& a, int n) {
#ifdef PGBP_HOST_EMUL
  for (int m = 0; m < n; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_ref<MAXM>(a, m, e);
#else
  dim3 grid((unsigned)((a.B - a.e0 + 127) / 128), (unsigned)n);
  k_message_ref<MAXM><<<grid, 128, 0, b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message_ref");
}
static int launch_ref(pgbp_batch* b, const MsgArgs& a, int n, int mF) {
  if (mF <= 8) return launch_ref_t<8>(b, a, n);
  if (mF <= 16) return launch_ref_t<16>(b, a, n);
  if (mF <= 32) return launch_ref_t<32>(b, a, n);
  return launch_ref_t<PGBP_MAX_DIM>(b, a, n);
}

// One launch group (same step, same shape class).  blockIdx.y is limited to
// 65535: split larger groups.
int launch_group(pgbp_batch* b, MsgArgs a, const MsgDesc* d_msgs, const LaunchGroup& g) {
  int done = 0;
  while (done < g.count) {
    const int n = std::min(g.count - done, 65535);
    a.msgs = d_msgs + g.first + done;
    int rc = 0;
    if (g.ci == 0) {
      rc = launch_copy(b, a, n);
    } else if (a.opts & PGBP_CAL_REFORDER) {
      rc = launch_ref(b, a, n, g.ci > 0 ? g.ci + g.cs : g.maxm + g.cs);
    } else if (g.ci > 0) {
      rc = launch_t0_part0(b, a, n, g.ci, g.cs);
      if (rc == PGBP_NOT_MINE) rc = launch_t0_part1(b, a, n, g.ci, g.cs);
      if (rc == PGBP_NOT_MINE) rc = launch_t0_part2(b, a, n, g.ci, g.cs);
      if (rc == PGBP_NOT_MINE) PGBP_FAIL(PGBP_ESTATE, "no specialised kernel for shape (%d,%d)", g.ci, g.cs);
    } else {  // medium / large class: the group is uniform in (I, S) = (g.maxm, g.cs)
      rc = launch_medium(b, a, n, g.maxm, g.cs);
    }
    PGBP_TRY(rc);
    done += n;
  }
  return 0;
}

// residual_kldiv! for the n messages of a launch group (after their propagate_belief!)
template <int MAXM>
static int launch_kldiv_t(pgbp_batch* b, const MsgArgs& a, int n) {
#ifdef PGBP_HOST_EMUL
  const JSide js = batch_jside(b), jr{b->jb ? b->jb->resid : nullptr, js.ld, js.gs};
  for (int m = 0; m < n; m++)
    for (int64_t e = a.e0; e < a.B; e++) kldiv_thread<MAXM>(a, b->kldiv, m, e, jcolumn(js, e), jcolumn(jr, e), js.ld);
#else
  const JSide js = batch_jside(b), jr{b->jb ? b->jb->resid : nullptr, js.ld, js.gs};
  dim3 grid((unsigned)((a.B - a.e0 + 127) / 128), (unsigned)n);
  k_kldiv<MAXM><<<grid, 128, 0, b->stream>>>(a, b->kldiv, js, jr);
#endif
  b->launches++;
  return check_launch("k_kldiv");
}
int launch_kldiv(pgbp_batch* b, MsgArgs a, const MsgDesc* d_msgs, const LaunchGroup& g) {
  int maxs = g.ci == 0 ? PGBP_MAX_DIM : g.cs;  // copy groups mix sepset dimensions
  if (g.ci > 0) maxs = g.cs;
  int done = 0;
  while (done < g.count) {
    const int n = std::min(g.count - done, 65535);
    a.msgs = d_msgs + g.first + done;
    if (maxs <= 4) PGBP_TRY(launch_kldiv_t<4>(b, a, n));
    else if (maxs <= 12) PGBP_TRY(launch_kldiv_t<12>(b, a, n));
    else if (maxs <= 32) PGBP_TRY(launch_kldiv_t<32>(b, a, n));
    else PGBP_TRY(launch_kldiv_t<PGBP_MAX_DIM>(b, a, n));
    done += n;
  }
  return 0;
}

MsgArgs make_args(pgbp_batch* b, uint32_t opts, int32_t ref_base, bool use_done) {
  MsgArgs a;
  a.msgs = nullptr;
  a.tab = b->d_tab;
  a.state = b->state;
  a.resid = b->resid;
  a.calflag = b->calflag;
  a.status = b->status;
  a.done = use_done ? b->done : nullptr;
  a.B = b->chunk_end > 0 ? b->chunk_end : b->B;
  a.e0 = b->chunk_begin;
  a.ld = b->ld;
  a.opts = opts;
  a.ref_base = ref_base;
  return a;
}

template <int P>
static int launch_walk(pgbp_batch* b, const MsgArgs& a, int nmsg) {
#ifdef PGBP_HOST_EMUL
  for (int64_t e = a.e0; e < a.B; e++) walk_thread<P>(a, nmsg, e);
#else
  k_walk<P><<<(unsigned)((a.B - a.e0 + PGBP_WALK_THREADS - 1) / PGBP_WALK_THREADS), PGBP_WALK_THREADS, 0, b->stream>>>(a, nmsg);
#endif
  b->launches++;
  return check_launch("k_walk");
}

// post (+ pre) traversal of one tree in a single launch; first/count select the
// part of the walk list (postorder = [0,n), preorder = [n,2n))
int run_walk(pgbp_batch* b, int tree, int first, int count, uint32_t opts, int32_t ref_base, bool use_done) {
  MsgArgs a = make_args(b, opts, ref_base - first, use_done);
  a.msgs = b->d_walk[tree] + first;
  switch (b->plan->ntraits) {
    case 1: return launch_walk<1>(b, a, count);
    case 2: return launch_walk<2>(b, a, count);
    case 3: return launch_walk<3>(b, a, count);
    case 4: return launch_walk<4>(b, a, count);
    default: PGBP_FAIL(PGBP_ESTATE, "walk kernel: unsupported ntraits");
  }
}

bool use_walk(const pgbp_batch* b, int tree) {
  const Tree& tr = b->plan->trees[tree];
  if (!tr.walkable || b->plan->ntraits > PGBP_WALK_MAXP || b->jb) return false;
  // measured on B200 (lazaridis p=3, B=65536): level-parallel 70.3M calibrations/s, walk 46.5M
  // (8 warps/SM at 255 registers cannot hide HBM latency) => the walk kernel is opt-in only
  return b->walk_mode == 1;
}

// tile-walk applies to: tiny messages (sender dimension <= 4), no KL update, and a schedule deep
// enough that per-step launches are latency-bound (>= 24 steps averaging < 32 messages).  Steps wider than
// b->tw_wide messages are split off into ordinary launches (LANES lanes would serialise them); runs of
// narrower steps in between go to one tile-walk launch each.
static bool use_tilewalk(const pgbp_batch* b, const Traversal& tv, uint32_t opts) {
  if (b->tilewalk_mode == 0 || (opts & (PGBP_CAL_RESIDKLDIV | PGBP_CAL_REFORDER)) || tv.tw.empty() || b->jb) return false;
  if (b->tilewalk_mode == 1) return true;
  return tv.nsteps >= 24 && (int64_t)tv.msgs.size() < 32 * (int64_t)tv.nsteps;
}

static int launch_tilewalk(pgbp_batch* b, const MsgArgs& a, const Traversal& tv, int td, int s0, int s1) {
  const int k0 = tv.step_stage[s0], k1 = tv.step_stage[s1];
#ifdef PGBP_HOST_EMUL
  (void)td;
  for (int k = k0; k < k1; k++)
    for (int m = tv.stage_off[k]; m < tv.stage_off[k + 1]; m++)
      for (int64_t e = a.e0; e < a.B; e++) tilewalk_message(a, tv.tw[m], e);
#else
  const unsigned grid = (unsigned)((a.B - a.e0 + 31) / 32);
  const TwDesc* descs = b->d_tw[td];
  const int32_t* so = b->d_stage_off[td];
  switch (b->tw_lanes) {
    case 4: k_tilewalk<4, 8><<<grid, dim3(32, 4), 0, b->stream>>>(a, descs, so, k0, k1); break;
    case 16: k_tilewalk<16, 2><<<grid, dim3(32, 16), 0, b->stream>>>(a, descs, so, k0, k1); break;
    default: k_tilewalk<8, 4><<<grid, dim3(32, 8), 0, b->stream>>>(a, descs, so, k0, k1); break;
  }
#endif
  b->launches++;
  return check_launch("k_tilewalk");
}

int run_traversal(pgbp_batch* b, int tree, int dir, uint32_t opts, int32_t ref_base, bool use_done) {
  const Traversal& tv = b->plan->trees[tree].trav[dir];
  MsgArgs a = make_args(b, opts, ref_base, use_done);
  const MsgDesc* d = b->d_msgs[2 * tree + dir];
  if (use_tilewalk(b, tv, opts)) {
    const int wide = b->tw_wide;
    auto width = [&](int st) { return tv.step_off[st + 1] - tv.step_off[st]; };
    size_t gi = 0;  // groups are in launch order, i.e. sorted by step
    int st = 0;
    while (st < tv.nsteps) {
      int s1 = st;
      while (s1 < tv.nsteps && width(s1) <= wide) s1++;
      if (s1 - st >= 2) {  // a run of narrow steps: one launch
        a.msgs = d;
        PGBP_TRY(launch_tilewalk(b, a, tv, 2 * tree + dir, st, s1));
        while (gi < tv.groups.size() && tv.groups[gi].step < s1) gi++;
        st = s1;
        continue;
      }
      // a wide (or isolated) step: its ordinary launch groups
      while (gi < tv.groups.size() && tv.groups[gi].step < st) gi++;
      for (; gi < tv.groups.size() && tv.groups[gi].step == st; gi++) PGBP_TRY(launch_group(b, a, d, tv.groups[gi]));
      st++;
    }
    return 0;
  }
  for (const LaunchGroup& g : tv.groups) {
    PGBP_TRY(launch_group(b, a, d, g));
    if (opts & PGBP_CAL_RESIDKLDIV) PGBP_TRY(launch_kldiv(b, a, d, g));
  }
  return 0;
}

// iscalibrated_residnorm(beliefs) = AND over all directed messages
// (src/clustergraphbeliefs.jl:168-169); with auto, freeze calibrated elements.
PGBP_HD void iscal_thread(const uint8_t* calflag, int nd, int64_t ld, const int32_t* status, uint8_t* done,
                          int32_t* iscal, int32_t* itertree, int32_t it, int32_t tr, int autostop, int64_t e,
                          const uint8_t* calflagJ, int64_t ldJ, int64_t gs) {
  if (done && done[e]) return;  // frozen: keeps its (true) result
  int ok = status[e] == 0;
  for (int d = 0; d < nd && ok; d++) ok = calflag[(int64_t)d * ld + e] != 0;
  if (calflagJ) {  // shared-precision batches: the J part of every flag is the group's (jb->calflag)
    const int64_t g = e / gs;
    for (int d = 0; d < nd && ok; d++) ok = calflagJ[(int64_t)d * ldJ + g] != 0;
  }
  iscal[e] = ok;
  if (ok) {
    if (itertree && itertree[e] == 0) {
      itertree[e] = it;
      itertree[ld + e] = tr;
    }
    if (autostop && done) done[e] = 1;
  }
}

#ifndef PGBP_HOST_EMUL
__global__ void k_iscal(const uint8_t* calflag, int nd, int64_t e0, int64_t B, int64_t ld, const int32_t* status,
                        uint8_t* done, int32_t* iscal, int32_t* itertree, int32_t it, int32_t tr, int autostop,
                        const uint8_t* calflagJ, int64_t ldJ, int64_t gs) {
  const int64_t e = e0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  iscal_thread(calflag, nd, ld, status, done, iscal, itertree, it, tr, autostop, e, calflagJ, ldJ, gs);
}
#endif

int launch_iscal(pgbp_batch* b, int it, int tr, int autostop) {
  const int nd = 2 * b->plan->nsepsets;
  const int64_t e0 = b->chunk_begin, e1 = b->chunk_end > 0 ? b->chunk_end : b->B;
  const uint8_t* fJ = b->jb ? b->jb->calflag : nullptr;
  const int64_t ldJ = b->jb ? b->jb->ld : 0;
#ifdef PGBP_HOST_EMUL
  for (int64_t e = e0; e < e1; e++)
    iscal_thread(b->calflag, nd, b->ld, b->status, b->done, b->iscal, b->itertree, it, tr, autostop, e, fJ, ldJ, b->group_size);
#else
  k_iscal<<<(unsigned)((e1 - e0 + 255) / 256), 256, 0, b->stream>>>(b->calflag, nd, e0, e1, b->ld, b->status, b->done,
                                                                     b->iscal, b->itertree, it, tr, autostop, fJ, ldJ,
                                                                     b->group_size);
#endif
  b->launches++;
  return check_launch("k_iscal");
}

int integrate_launch(pgbp_batch* b, int belief, double* d_mu_soa, double* d_norm, int64_t ld_out, double* d_cov_soa) {
  const pgbp_plan* p = b->plan;
  if (belief >= p->nclusters) PGBP_TRY(batch_materialize_sepsets(b));
  const int M = p->dim[belief];
  const int64_t js = p->jslot[belief], hs = batch_hrow(b, belief), gs = batch_grow(b, belief);
  const JSide jside = batch_jside(b);
#ifdef PGBP_HOST_EMUL
  for (int64_t e = 0; e < b->B; e++)
    integrate_thread<PGBP_MAX_DIM>(b->state, b->status, b->ld, e, js, hs, gs, M, d_mu_soa, d_norm, ld_out, d_cov_soa, jcolumn(jside, e), jside.ld);
#else
  const unsigned grid = (unsigned)((b->B + 127) / 128);
  if (M <= 4)
    k_integrate<4><<<grid, 128, 0, b->stream>>>(b->state, b->status, b->B, b->ld, js, hs, gs, M, d_mu_soa, d_norm, ld_out, d_cov_soa, jside);
  else if (M <= 12)
    k_integrate<12><<<grid, 128, 0, b->stream>>>(b->state, b->status, b->B, b->ld, js, hs, gs, M, d_mu_soa, d_norm, ld_out, d_cov_soa, jside);
  else if (M <= 32)
    k_integrate<32><<<grid, 128, 0, b->stream>>>(b->state, b->status, b->B, b->ld, js, hs, gs, M, d_mu_soa, d_norm, ld_out, d_cov_soa, jside);
  else
    k_integrate<PGBP_MAX_DIM><<<grid, 128, 0, b->stream>>>(b->state, b->status, b->B, b->ld, js, hs, gs, M, d_mu_soa, d_norm, ld_out, d_cov_soa, jside);
#endif
  b->launches++;
  return check_launch("k_integrate");
}

}  // namespace pgbp

// Enqueue one calibrate! call (validated arguments) on b->stream, eagerly.  *nlaunch_est: launches of
// ONE element chunk.
static int calibrate_enqueue(pgbp_batch* b, const std::vector<int32_t>& ids, int32_t niter, uint32_t flags, bool lazy);

extern "C" {

int32_t pgbp_calibrate_async(pgbp_batch* b, const int32_t* tree_ids, int32_t ntrees, int32_t niter, uint32_t flags) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  const pgbp_plan* p = b->plan;
  if (!(flags & PGBP_CAL_BOTH)) PGBP_FAIL(PGBP_EINVAL, "flags select neither postorder nor preorder");
  if (niter < 1) PGBP_FAIL(PGBP_EINVAL, "niter < 1");
  if ((flags & (PGBP_CAL_RESIDNORM | PGBP_CAL_AUTO)) && !b->calflag)
    PGBP_FAIL(PGBP_ESTATE, "residual tracking requested but the batch was created without PGBP_BATCH_RESIDUALS");
  if (b->group_size > 1 && (flags & PGBP_CAL_AUTO))
    PGBP_FAIL(PGBP_EINVAL, "auto-stop is per element: not available in shared-precision mode (the group's J keeps moving)");
  if ((flags & PGBP_CAL_REFORDER) && b->group_size > 1)
    PGBP_FAIL(PGBP_EINVAL, "the reference-order validation mode is not available for shared-precision batches");
  if ((flags & PGBP_CAL_RESIDKLDIV) && !b->kldiv)
    PGBP_FAIL(PGBP_ESTATE, "update_residualkldiv requested but the batch was created without PGBP_BATCH_RESIDUALS");
  std::vector<int32_t> ids;
  if (tree_ids && ntrees < 0) PGBP_FAIL(PGBP_EINVAL, "ntrees < 0");
  if (tree_ids) ids.assign(tree_ids, tree_ids + ntrees);
  else for (int t = 0; t < (int)p->trees.size(); t++) ids.push_back(t);
  if (ids.empty()) PGBP_FAIL(PGBP_EINVAL, "empty schedule");
  for (int t : ids) if (t < 0 || t >= (int)p->trees.size()) PGBP_FAIL(PGBP_EINVAL, "tree id %d out of range", t);
  PGBP_TRY(set_device(b->device));
  // lazy sepset zero: usable iff the call starts with the postorder traversal of a tree that writes every
  // sepset (a spanning tree of a clique tree), through the per-step launches
  if (b->sepsets_lazy_zero) {
    const pgbp::Tree& t0 = p->trees[ids[0]];
    const bool ok = (flags & PGBP_CAL_POSTORDER) && t0.covers_sepsets && !(use_walk(b, ids[0]) && !(flags & PGBP_CAL_REFORDER)) &&
                    !(flags & PGBP_CAL_RESIDKLDIV);
    if (!ok) PGBP_TRY(batch_materialize_sepsets(b));
  }
  const bool lazy = b->sepsets_lazy_zero;
  b->sepsets_lazy_zero = false;  // after this call every sepset holds a real value
#ifndef PGBP_HOST_EMUL
  // CUDA graph replay: a calibrate! call is a fixed sequence of launches for fixed (schedule, niter,
  // flags, kernel strategy); the second call with the same key captures it, later calls replay it
  // (one cudaGraphLaunch instead of up to tens of thousands of launches for loopy schedules).
  int64_t nl = 0;
  for (int t : ids) nl += (int64_t)p->trees[t].trav[0].groups.size() + (int64_t)p->trees[t].trav[1].groups.size();
  nl *= niter;
  // (shared-precision batches small enough for the walk kernels are not captured: the element walk spins on counters
  // the group walk publishes from another stream, and a graph does not promise to run independent branches concurrently)
  const bool walkable_shared = b->jb && (b->B + 127) / 128 <= 64 && b->ngroups <= 16;
  const bool want_graph = !walkable_shared && (b->graph_mode == 1 || (b->graph_mode < 0 && nl >= 24));
  if (want_graph) {
    std::string key;
    for (int t : ids) key += std::to_string(t) + ",";
    key += "|" + std::to_string(niter) + "|" + std::to_string(flags) + "|" + std::to_string(b->walk_mode) + "|" +
           std::to_string(b->coop_mode) + "|" + std::to_string(b->pipeline) + "|" + std::to_string((int)b->want_info) +
           "|" + std::to_string(b->tilewalk_mode) + "|" + std::to_string(b->tw_lanes) + "|" + std::to_string(b->tw_wide) +
           "|" + std::to_string((int)lazy) +
           "|" + std::to_string((uintptr_t)b->stream);
    auto it = b->graphs.find(key);
    if (it == b->graphs.end()) {  // first sight: run eagerly (also performs one-time cudaFuncSetAttribute calls)
      b->graphs[key] = pgbp_batch::GraphEntry{};
      return calibrate_enqueue(b, ids, niter, flags, lazy);
    }
    pgbp_batch::GraphEntry& ge = it->second;
    if (!ge.exec && !ge.failed) {
      const int64_t l0 = b->launches;
      cudaGraph_t graph = nullptr;
      cudaError_t ce = cudaStreamBeginCapture(b->stream, cudaStreamCaptureModeThreadLocal);
      int rc = 0;
      if (ce == cudaSuccess) {
        rc = calibrate_enqueue(b, ids, niter, flags, lazy);
        ce = cudaStreamEndCapture(b->stream, &graph);
      }
      if (ce == cudaSuccess && !rc && graph) {
        cudaGraphExec_t ex = nullptr;
        ce = cudaGraphInstantiate(&ex, graph, 0);
        if (ce == cudaSuccess) { ge.exec = (void*)ex; ge.launches = b->launches - l0; }
      }
      if (graph) cudaGraphDestroy(graph);
      b->launches = l0;
      if (!ge.exec) {  // capture not possible (e.g. the caller's stream is already capturing): stay eager
        ge.failed = true;
        cudaGetLastError();
        return calibrate_enqueue(b, ids, niter, flags, lazy);
      }
    }
    if (ge.exec) {
      PGBP_CUDA(cudaGraphLaunch((cudaGraphExec_t)ge.exec, b->stream));
      b->launches += ge.launches;
      return 0;
    }
  }
#endif
  return calibrate_enqueue(b, ids, niter, flags, lazy);
}

}  // extern "C"

static int calibrate_enqueue(pgbp_batch* b, const std::vector<int32_t>& ids, int32_t niter, uint32_t flags, bool lazy) {
  const pgbp_plan* p = b->plan;
  const bool autostop = (flags & PGBP_CAL_AUTO) != 0;
  const bool track = (flags & PGBP_CAL_RESIDNORM) != 0;
  if (b->done) PGBP_TRY(dev_memset(b->done, 0, (size_t)b->ld, b->stream));
  if (b->itertree) PGBP_TRY(dev_memset(b->itertree, 0, sizeof(int32_t) * 2 * (size_t)b->ld, b->stream));
  if (b->iscal) PGBP_TRY(dev_memset(b->iscal, 0, sizeof(int32_t) * (size_t)b->ld, b->stream));
  const uint32_t opts = flags & (PGBP_CAL_RESIDNORM | PGBP_CAL_RESIDKLDIV | PGBP_CAL_REFORDER);
  b->jfork_pending = true;  // (shared-precision batches: the group pass forks off the batch's stream here)
  // the whole schedule for the element range [b->chunk_begin, b->chunk_end) on b->stream
  auto enqueue = [&]() -> int {
    int32_t ref = 0;
    for (int it = 1; it <= niter; it++) {
      for (size_t j = 0; j < ids.size(); j++) {
        const uint32_t sepzero = (lazy && it == 1 && j == 0) ? PGBP_OPT_SEPZERO : 0u;
        const int t = ids[j];
        const int n = (int)p->trees[t].parent.size();
        if (b->jb) {  // shared-precision batch: group pass (J, factor cache) + element pass (h, g) per traversal
          if (flags & PGBP_CAL_POSTORDER) { PGBP_TRY(shared_run_traversal(b, t, 0, opts | sepzero, ref)); ref += n; }
          if (flags & PGBP_CAL_PREORDER) { PGBP_TRY(shared_run_traversal(b, t, 1, opts, ref)); ref += n; }
        } else if (use_walk(b, t) && !(opts & (PGBP_CAL_RESIDKLDIV | PGBP_CAL_REFORDER))) {
          const bool po = flags & PGBP_CAL_POSTORDER, pr = flags & PGBP_CAL_PREORDER;
          const int first = po ? 0 : n, count = (po ? n : 0) + (pr ? n : 0);
          PGBP_TRY(run_walk(b, t, first, count, opts, ref, autostop));
          ref += count;
        } else {
          if (flags & PGBP_CAL_POSTORDER) { PGBP_TRY(run_traversal(b, t, 0, opts | sepzero, ref, autostop)); ref += n; }
          if (flags & PGBP_CAL_PREORDER) { PGBP_TRY(run_traversal(b, t, 1, opts, ref, autostop)); ref += n; }
        }
        const bool last = (it == niter && j + 1 == ids.size());
        if (track && (autostop || last || b->want_info)) PGBP_TRY(launch_iscal(b, it, (int)j + 1, autostop));
        if (ref > (1 << 22)) ref = 0;  // keep the status word positive
      }
    }
    return 0;
  };
  // how many element chunks?  auto: cut when one launch of the schedule cannot fill the GPU
  // (threads per launch ~ B x messages per step) and the chunks stay >= 8192 elements
  int nchunk = 1;
#ifndef PGBP_HOST_EMUL
  if (b->jb) nchunk = 1;  // shared-precision batches: the group pass is not chunked
  else if (b->pipeline > 1) nchunk = b->pipeline;
  else if (b->pipeline < 0) {
    int64_t nmsg = 0, nlaunch = 0;
    for (int t : ids)
      for (int dir = 0; dir < 2; dir++) {
        nmsg += (int64_t)p->trees[t].trav[dir].msgs.size();
        nlaunch += (int64_t)p->trees[t].trav[dir].groups.size();
      }
    const double per_launch = nlaunch ? (double)b->B * (double)nmsg / (double)nlaunch : 1e30;
    // (deep loopy schedules are launch-bound already: more launches would not help them)
    if (per_launch < 1.5e6 && nlaunch * niter <= 512) nchunk = (int)std::min<int64_t>(4, b->B / 8192);
  }
  if (nchunk < 1) nchunk = 1;
#endif
  if (nchunk == 1) {
    b->chunk_begin = 0; b->chunk_end = 0;
    return enqueue();
  }
#ifndef PGBP_HOST_EMUL
  while ((int)b->pipe_streams.size() < nchunk) {
    cudaStream_t s;
    PGBP_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    b->pipe_streams.push_back(s);
  }
  while ((int)b->pipe_events.size() < nchunk + 1) {
    cudaEvent_t ev;
    PGBP_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    b->pipe_events.push_back((void*)ev);
  }
  const int64_t csz = ((b->B + nchunk - 1) / nchunk + 127) / 128 * 128;
  cudaStream_t main_stream = b->stream;
  PGBP_CUDA(cudaEventRecord((cudaEvent_t)b->pipe_events[0], main_stream));
  int rc = 0;
  int used = 0;
  for (int c = 0; c < nchunk && !rc; c++) {
    const int64_t e0 = (int64_t)c * csz, e1 = std::min<int64_t>(b->B, e0 + csz);
    if (e0 >= e1) break;
    b->stream = b->pipe_streams[c];
    b->chunk_begin = e0; b->chunk_end = e1;
    cudaError_t ce = cudaStreamWaitEvent(b->stream, (cudaEvent_t)b->pipe_events[0], 0);
    if (ce != cudaSuccess) { rc = PGBP_ECUDA; set_error("cudaStreamWaitEvent failed"); break; }
    rc = enqueue();
    if (!rc && cudaEventRecord((cudaEvent_t)b->pipe_events[c + 1], b->stream) != cudaSuccess) { rc = PGBP_ECUDA; set_error("cudaEventRecord failed"); }
    used = c + 1;
  }
  b->stream = main_stream;
  b->chunk_begin = 0; b->chunk_end = 0;
  for (int c = 0; c < used; c++)  // join (also on error, so that the main stream stays ordered after the chunks)
    if (cudaStreamWaitEvent(main_stream, (cudaEvent_t)b->pipe_events[c + 1], 0) != cudaSuccess && !rc) { rc = PGBP_ECUDA; set_error("cudaStreamWaitEvent failed"); }
  return rc;
#else
  return enqueue();
#endif
}

extern "C" {

int32_t pgbp_calibrate(pgbp_batch* b, const int32_t* tree_ids, int32_t ntrees, int32_t niter, uint32_t flags,
                       int32_t* succ, int32_t* iscal, int32_t* iter_tree) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  b->want_info = iter_tree != nullptr;
  int rc = pgbp_calibrate_async(b, tree_ids, ntrees, niter, flags);
  b->want_info = false;
  PGBP_TRY(rc);
  const int64_t B = b->B;
  // results go through the batch's pinned bounce buffer when it is available: [status | iscal]
  int32_t* pin = (succ || iscal) ? (int32_t*)batch_pinned(b, sizeof(int32_t) * 2 * (size_t)B) : nullptr;
  std::vector<int32_t> st_v;
  int32_t* st = nullptr;
  const bool want_ic = iscal && b->iscal && (flags & PGBP_CAL_RESIDNORM);
  if (succ || iscal) {
    if (pin) st = pin;
    else { st_v.resize(B); st = st_v.data(); }
    PGBP_TRY(d2h(st, b->status, sizeof(int32_t) * B, b->stream));
  }
  if (iscal) {
    if (want_ic) PGBP_TRY(d2h(pin ? pin + B : iscal, b->iscal, sizeof(int32_t) * B, b->stream));
    else memset(iscal, 0, sizeof(int32_t) * B);
  }
  std::vector<int32_t> itr;
  if (iter_tree) {
    if (b->itertree) {
      itr.resize(2 * b->ld);
      PGBP_TRY(d2h(itr.data(), b->itertree, sizeof(int32_t) * 2 * b->ld, b->stream));
    }
  }
  PGBP_TRY(stream_sync(b->stream));
  if (want_ic && pin) memcpy(iscal, pin + B, sizeof(int32_t) * B);
  if (succ) for (int64_t e = 0; e < B; e++) succ[e] = st[e] == 0;
  if (iscal) for (int64_t e = 0; e < B; e++) if (st[e] != 0) iscal[e] = 0;  // (false,false) on failure
  if (iter_tree) for (int64_t e = 0; e < B; e++) {
    iter_tree[2 * e] = itr.empty() ? 0 : itr[e];
    iter_tree[2 * e + 1] = itr.empty() ? 0 : itr[b->ld + e];
  }
  return 0;
}

int32_t pgbp_batch_set_walk_mode(pgbp_batch* b, int32_t mode) {
  if (!b || mode < -1 || mode > 1) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  b->walk_mode = mode;
  return 0;
}

int32_t pgbp_batch_set_pipeline(pgbp_batch* b, int32_t nchunks) {
  if (!b || nchunks == 0 || nchunks < -1 || nchunks > 64) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  b->pipeline = nchunks;
  return 0;
}

int32_t pgbp_batch_set_tilewalk_mode(pgbp_batch* b, int32_t mode) {
  if (!b || mode < -1 || mode > 1) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  b->tilewalk_mode = mode;
  return 0;
}

int32_t pgbp_batch_set_tilewalk_params(pgbp_batch* b, int32_t lanes, int32_t wide) {
  if (!b || (lanes != 0 && lanes != 4 && lanes != 8 && lanes != 16) || wide < 0) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  if (lanes) b->tw_lanes = lanes;
  if (wide) b->tw_wide = wide;
  return 0;
}

int32_t pgbp_batch_set_graph_mode(pgbp_batch* b, int32_t mode) {
  if (!b || mode < -1 || mode > 1) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  b->graph_mode = mode;
  return 0;
}

int32_t pgbp_batch_set_coop_mode(pgbp_batch* b, int32_t mode) {
  if (!b || (mode != -1 && mode != 0 && mode != 1 && mode != 2 && mode != 4 && mode != 8)) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  b->coop_mode = mode;
  return 0;
}

int32_t pgbp_propagate(pgbp_batch* b, int32_t from_cluster, int32_t sepset, int32_t to_cluster, uint32_t flags) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  const pgbp_plan* p = b->plan;
  if (from_cluster < 0 || from_cluster >= p->nclusters || to_cluster < 0 || to_cluster >= p->nclusters)
    PGBP_FAIL(PGBP_EINVAL, "cluster index out of range");
  const int j = sepset >= p->nclusters ? sepset - p->nclusters : sepset;  // accept belief index or sepset index
  MsgDesc md;
  PGBP_TRY(p->make_msg(from_cluster, j, to_cluster, &md));  // the plan is immutable: no table ever grows here
  PGBP_TRY(set_device(b->device));
  PGBP_TRY(batch_materialize_sepsets(b));
  if (b->jb) return shared_propagate(b, md, flags & PGBP_CAL_RESIDNORM, 0x3ffff0);
  PGBP_TRY(h2d(b->d_one, &md, sizeof md, b->stream));
  PGBP_TRY(stream_sync(b->stream));  // md is a stack object
  LaunchGroup g;
  g.step = 0; g.first = 0; g.count = 1;
  shape_class(md.mF - md.s, md.s, &g.ci, &g.cs, &g.maxm);
  MsgArgs a = make_args(b, flags & (PGBP_CAL_RESIDNORM | PGBP_CAL_REFORDER), 0x3ffff0, false);
  if (!b->calflag) a.opts &= ~PGBP_CAL_RESIDNORM;
  return launch_group(b, a, b->d_one, g);
}

int32_t pgbp_integrate_device(pgbp_batch* b, int32_t belief, double* d_mu_soa, double* d_norm) {
  if (!b || !d_norm) PGBP_FAIL(PGBP_EINVAL, "null argument");
  if (belief < 0 || belief >= b->plan->nbeliefs) PGBP_FAIL(PGBP_EINVAL, "belief index out of range");
  PGBP_TRY(set_device(b->device));
  return integrate_launch(b, belief, d_mu_soa, d_norm, b->ld, nullptr);
}

int32_t pgbp_integrate(pgbp_batch* b, int32_t belief, double* mu, double* norm) {
  if (!b || !norm) PGBP_FAIL(PGBP_EINVAL, "null argument");
  if (belief < 0 || belief >= b->plan->nbeliefs) PGBP_FAIL(PGBP_EINVAL, "belief index out of range");
  PGBP_TRY(set_device(b->device));
  const int M = b->plan->dim[belief];
  const int64_t ld = b->ld;
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (size_t)ld * (size_t)(M + 1) * (mu ? 2 : 1)));
  double* d_norm = b->scratch;
  double* d_mu = mu ? b->scratch + ld : nullptr;
  PGBP_TRY(integrate_launch(b, belief, d_mu, d_norm, ld, nullptr));
  double* pin = (double*)batch_pinned(b, sizeof(double) * (size_t)b->B);  // log-likelihoods through pinned memory
  PGBP_TRY(d2h(pin ? pin : norm, d_norm, sizeof(double) * b->B, b->stream));
  if (mu && M > 0) {
    double* d_aos = b->scratch + ld * (int64_t)(M + 1);
    PGBP_TRY(soa_to_aos(b, d_mu, ld, d_aos, M, nullptr));
    PGBP_TRY(d2h(mu, d_aos, sizeof(double) * b->B * M, b->stream));
  }
  PGBP_TRY(stream_sync(b->stream));
  if (pin) memcpy(norm, pin, sizeof(double) * b->B);
  return 0;
}

int32_t pgbp_integrate_cov(pgbp_batch* b, int32_t belief, double* mu, double* cov, double* norm) {
  if (!b || !norm || !cov) PGBP_FAIL(PGBP_EINVAL, "null argument");
  if (belief < 0 || belief >= b->plan->nbeliefs) PGBP_FAIL(PGBP_EINVAL, "belief index out of range");
  PGBP_TRY(set_device(b->device));
  const int M = b->plan->dim[belief];
  const int64_t ld = b->ld;
  const int SM = tri(M);
  // scratch: norm | mu SoA | cov packed SoA | AoS staging (M*M columns)
  const size_t need = sizeof(double) * (size_t)ld * (size_t)(1 + M + SM + (size_t)M * M + 1);
  PGBP_TRY(batch_need_scratch(b, need));
  double* d_norm = b->scratch;
  double* d_mu = b->scratch + ld;
  double* d_cov = d_mu + ld * (int64_t)M;
  double* d_aos = d_cov + ld * (int64_t)SM;
  PGBP_TRY(integrate_launch(b, belief, d_mu, d_norm, ld, d_cov));
  PGBP_TRY(d2h(norm, d_norm, sizeof(double) * b->B, b->stream));
  if (M > 0) {
    if (mu) {
      PGBP_TRY(soa_to_aos(b, d_mu, ld, d_aos, M, nullptr));
      PGBP_TRY(d2h(mu, d_aos, sizeof(double) * b->B * M, b->stream));
      PGBP_TRY(stream_sync(b->stream));
    }
    std::vector<int32_t> sl((size_t)M * M);  // full square from the packed upper triangle
    for (int c = 0; c < M; c++)
      for (int r = 0; r < M; r++) sl[(size_t)c * M + r] = r <= c ? pk(r, c) : pk(c, r);
    int32_t* d_sl = nullptr;
    void* v = nullptr;
    PGBP_TRY(dev_malloc(&v, sizeof(int32_t) * sl.size()));
    d_sl = (int32_t*)v;
    int rc = h2d(d_sl, sl.data(), sizeof(int32_t) * sl.size(), b->stream);
    if (!rc) rc = soa_to_aos(b, d_cov, ld, d_aos, M * M, d_sl);
    if (!rc) rc = d2h(cov, d_aos, sizeof(double) * b->B * (size_t)M * M, b->stream);
    if (!rc) rc = stream_sync(b->stream);
    dev_free(d_sl);
    PGBP_TRY(rc);
  }
  return stream_sync(b->stream);
}

}  // extern "C"
