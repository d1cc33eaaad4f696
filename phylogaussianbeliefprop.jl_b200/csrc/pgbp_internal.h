// Internal structures of libpgbp_b200: the plan (static index work, host) and
// the batch (device state).  See DESIGN.md for the HBM layout.
#pragma once
#include <map>
#include <string>
#include <memory>
#include <vector>

#include "../../include/pgbp_b200.h"
#include "pgbp_backend.h"

namespace pgbp {

PGBP_HD int tri(int m) { return m * (m + 1) / 2; }
// packed upper, column-major: (r <= c) -> c(c+1)/2 + r
PGBP_HD int pk(int r, int c) { return c * (c + 1) / 2 + r; }

// Where the J rows of an element live.  Ordinary batches: base == nullptr (the element's own column of the state
// array).  Shared-precision batches: the array of the group batch (pgbp_batch::jb), pitch ld, column e / gs.
struct JSide {
  const double* base;
  int64_t ld, gs;
};
PGBP_HD const double* jcolumn(const JSide& j, int64_t e) { return j.base ? j.base + e / j.gs : nullptr; }

// One message F -> T through sepset S (src/beliefupdates.jl:650-665), as index
// data only.  Slots index rows of the batch's SoA arrays.
struct MsgDesc {
  int64_t fJ, fh, fg;  // sender cluster slots (state)
  int64_t sJ, sh, sg;  // sepset slots (state)
  int64_t tJ, th, tg;  // receiver cluster slots (state)
  int64_t rJ, rh;      // residual slots (resid array)
  int32_t dmsg;        // directed-message id = 2*sepset + side (flags / kldiv row)
  int32_t mF, s;       // sender and sepset dimension; i = mF - s is integrated out
  int32_t gat;         // table: S(mF) packed J slots of the sender in [I;K] order, then mF h slots
  int32_t sca;         // table: S(s) packed J slots of the receiver, then s h slots
  int32_t ref;         // position in the reference's sequential order of this traversal
  int32_t wid;         // walk-kernel shape id (pgbp_shapes.h), -1 if outside the family
};

// Tile-walk descriptor: one message of sender dimension <= 4 with every slot index resolved (no
// index-table indirection), 160 bytes = ten 16-byte chunks, staged in shared memory one stage ahead.
#define PGBP_TW_MAXM 4
#define PGBP_TW_STAGE 64  // messages per stage (a stage never crosses a step boundary)
struct alignas(16) TwDesc {
  uint32_t fJ[10];    // sender J slots, packed upper in [I;K] order
  uint32_t fh[4];     // sender h slots in [I;K] order
  uint32_t tJ[10];    // receiver J slots of the sepset scope, packed upper
  uint32_t th[4];     // receiver h slots of the sepset scope
  uint32_t fg, sg, tg;
  uint32_t sJ, sh;    // sepset J / h rows (contiguous)
  uint32_t rJ, rh;    // residual rows (contiguous)
  uint32_t dmsg, ref;
  uint32_t shape;     // I * 8 + S
  uint32_t pad[2];
};
static_assert(sizeof(TwDesc) == 160, "TwDesc must be ten 16-byte chunks");

struct LaunchGroup {
  int32_t step;        // launch step (groups of one step are independent)
  int32_t ci, cs;      // shape class (i, s) if specialised, (-1,-1) generic
  int32_t maxm;        // for the generic kernel: max sender dimension in the group
  int32_t first, count;  // range in Traversal::msgs
};

struct Traversal {
  std::vector<MsgDesc> msgs;          // execution order
  std::vector<int32_t> step_of_msg;   // step of msgs[i]
  std::vector<LaunchGroup> groups;    // launch order
  std::vector<int32_t> step_off;      // [nsteps+1] range of msgs of each step (msgs are sorted by step)
  int32_t max_mF = 0;                 // largest sender dimension
  // tile-walk form (only when max_mF <= PGBP_TW_MAXM): resolved descriptors in execution order, stages of
  // <= PGBP_TW_STAGE messages inside one step, first stage of every step ([nsteps+1])
  std::vector<TwDesc> tw;
  std::vector<int32_t> stage_off, step_stage;
  int32_t nsteps = 0;
  double bytes_noresid = 0, bytes_resid = 0, flops = 0;  // algorithmic, per element
};

struct Tree {
  std::vector<int32_t> parent, child, sepset;
  Traversal trav[2];  // 0 postorder, 1 preorder
  std::vector<MsgDesc> walk;  // postorder then preorder messages in reference order
  bool walkable = false;      // every message is inside the walk family of ntraits
  bool covers_sepsets = false;  // the edges are nsepsets DISTINCT sepsets: one traversal writes every sepset exactly once
                                // (condition of the lazy sepset zero)
};

struct FamilyTable {
  int32_t nnodes = 0, ntips = 0, root_fixed = 0;
  std::vector<int32_t> node_cluster, mem_off, mem_pos, mem_color, node_datarow;
  std::vector<double> mem_length, mem_gamma;
  // derived: nodes of each cluster, ascending (order of the loop at src/beliefs.jl:798)
  std::vector<int32_t> clu_off, clu_node;
  // derived, for the write-once path of K1: clu_flag bit 0 = some scope entry of the cluster is covered
  // by no family (zero-fill first); first_J[v] bit a*8+b / first_h[v] bit a = family v is the first
  // (in node order) to touch block (member a, member b) / member a's h segment of its cluster
  std::vector<uint8_t> clu_flag, first_h;
  std::vector<uint64_t> first_J;
  int32_t ncolors_min = 1;
  // trait-level scopes (missing data): scoped == true routes K1 through the generic scoped body
  bool scoped = false;
  std::vector<int32_t> mem_tpos;     // [#members * p]
  std::vector<uint8_t> tip_missing;  // [ntips * p]
};

}  // namespace pgbp

struct pgbp_plan {
  int32_t nclusters = 0, nsepsets = 0, nbeliefs = 0, ntraits = 0;
  std::vector<int32_t> dim;
  std::vector<int64_t> jslot, hslot, gslot;  // state layout per belief
  int64_t nslots_state = 0, nslots_factor = 0;
  std::vector<int64_t> rjslot, rhslot;       // residual layout per directed message
  int64_t nslots_resid = 0;
  std::vector<int32_t> sep_a, sep_b;
  std::vector<std::vector<int32_t>> up_a, up_b;
  std::map<std::pair<int32_t, int32_t>, int32_t> sep_of;  // (min,max cluster) -> sepset
  std::vector<pgbp::Tree> trees;
  std::vector<int32_t> tab;                  // deduplicated index tables
  std::map<std::vector<int32_t>, int32_t> tab_index;
  // neighbours of each cluster ordered by neighbour code (neighbor_labels order)
  std::vector<std::vector<std::pair<int32_t, int32_t>>> nbrs;  // (neighbour cluster, sepset)
  bool has_families = false;
  pgbp::FamilyTable fam;
  int32_t max_dim = 0;

  int32_t intern_table(const std::vector<int32_t>& t);        // plan creation only
  int32_t find_table(const std::vector<int32_t>& t) const;  // -1 if absent
  // build the descriptor of message from -> to through sepset j (read-only: every table is interned at creation)
  int make_msg(int32_t from, int32_t j, int32_t to, pgbp::MsgDesc* out) const;
};

struct pgbp_batch {
  const pgbp_plan* plan = nullptr;
  int64_t B = 0, ld = 0;
  int32_t device = 0;
  uint32_t flags = 0;
  pgbp_stream_t stream = 0;
  bool own_stream = false;
  double* state = nullptr;
  double* factor = nullptr;
  double* resid = nullptr;
  double* kldiv = nullptr;
  uint8_t* calflag = nullptr;  // [2*nsepsets][ld]
  uint8_t* calflagJ = nullptr; // (unused since the factored shared-precision layout: the J part of the flags lives in jb->calflag)
  int64_t group_size = 0;      // > 1: shared-precision mode, elements [k*gs, (k+1)*gs) share every J
  // ---- shared-precision batches (group_size > 1): factored layout -------------------------------------------
  // The precisions J of a group depend on its parameter vector only (src/beliefupdates.jl:77-81: only h and g see
  // the data), so they are kept ONCE per group, in `jb`: an ordinary batch with one element per group (row pitch
  // jb->ld ~ ngroups) that owns every J row, the J part of the residuals and of the calibration flags.  This batch
  // then holds per ELEMENT only h and g, in a compact row numbering: belief i owns rows eh[i] .. eh[i]+m-1 (h) and
  // eh[i]+m (g) of `state` (clusters first: the first nrows_efactor rows are also the layout of `factor`);
  // directed message d owns rows erh[d] .. erh[d]+s-1 of `resid` (dh).  A message is passed in two kernels:
  // k_jmsg (one warp per (message, group)) factorises J_I, updates the J part and leaves U, 1/diag(U),
  // Z = U^-T J_IK and logdet in `cache`; k_hmsg (one thread per (message, element)) applies them to h and g.
  pgbp_batch* jb = nullptr;
  pgbp_batch* jparent = nullptr;      // set on the group batch: the shared-precision batch it belongs to
  int64_t ngroups = 0;
  double* jucache = nullptr;          // K1: family precision blocks per (node family, group), see AssignFast
  size_t jucache_len = 0;
  std::vector<int64_t> eh, erh;       // compact rows per belief / per directed message
  int64_t nrows_e = 0, nrows_efactor = 0, nrows_eresid = 0;
  std::vector<double*> jcache;        // index 2*tree+dir: [ngroups][jcache_len] factor records of one traversal
  std::vector<int64_t*> d_jcache_off; // index 2*tree+dir: record offset (doubles) of every message, execution order
  std::vector<int64_t> jcache_len;    // index 2*tree+dir: doubles per group
  // The group pass is latency-bound (one warp per (message, group), deep narrow schedules) and does not depend on
  // the element pass: it runs on its own stream `jstream`, one event per step; the element pass of step s waits
  // for event s only.  jcache_free[td]: recorded (main stream) after the element pass of traversal td, so that the
  // next group pass does not overwrite records that are still being read.
  pgbp_stream_t jstream = 0;
  std::vector<void*> jstep_events;    // cudaEvent_t per step (grown on demand)
  std::vector<void*> jcache_free;     // cudaEvent_t per traversal (null until first use)
  std::vector<char> jcache_used;      // traversal already passed during the current calibrate! call
  std::vector<unsigned*> d_walkflags;  // per traversal: [nsteps][ngroups] executions of the group walk per step
  std::vector<unsigned*> d_walkcount;  // per traversal: {executions of the element walk, blocks done in the current one}
  void* jfork_event = nullptr;
  bool jfork_pending = true;          // set at the start of every calibrate! call
  double* jcache_one = nullptr;       // scratch record for single messages (pgbp_propagate, regularize_onschedule)
  int64_t* d_zero64 = nullptr;        // device constant 0 (record offset of a single message)
  uint8_t* done = nullptr;     // [ld] (auto-stop mask)
  int32_t* status = nullptr;   // [ld]
  int32_t* iscal = nullptr;    // [ld]
  int32_t* itertree = nullptr; // [2][ld]
  int32_t* d_tab = nullptr;
  // per-tree, per-direction descriptor arrays on the device
  std::vector<pgbp::MsgDesc*> d_msgs;  // index 2*tree+dir
  std::vector<pgbp::MsgDesc*> d_walk;  // per tree, reference order (walk kernel)
  std::vector<int32_t*> d_step_off;    // index 2*tree+dir
  std::vector<pgbp::TwDesc*> d_tw;     // index 2*tree+dir (tile-walk kernel; null when not applicable)
  std::vector<int32_t*> d_stage_off;   // index 2*tree+dir
  int32_t tilewalk_mode = -1;          // -1 auto, 0 off, 1 on (where applicable)
  int32_t tw_lanes = 8, tw_wide = 512;  // tile-walk tuning: message lanes per block, width of a step launched alone
  pgbp::MsgDesc* d_one = nullptr;      // scratch descriptor for pgbp_propagate
  double* scratch = nullptr;           // staging for host<->device transposes / outputs
  size_t scratch_bytes = 0;
  // K1 device tables
  void* d_fam = nullptr;
  int64_t device_bytes = 0;
  int64_t launches = 0;
  bool want_info = false;
  int32_t walk_mode = -1;  // -1 auto, 0 never, 1 always (when walkable)
  // pipelined calibration: the batch is cut into `pipeline` chunks of elements, each walking the whole
  // schedule on its own stream (elements are independent), so that the ramp-up / tail of one chunk's
  // small launches overlaps the others' work.  chunk_begin / chunk_end: range being enqueued.
  int32_t pipeline = -1;  // -1 auto, 1 off, n > 1 chunks
  // CUDA-graph cache of calibrate! calls, keyed by (schedule, niter, flags, strategy, stream)
  struct GraphEntry { void* exec = nullptr; int64_t launches = 0; bool failed = false; };
  std::map<std::string, GraphEntry> graphs;
  int32_t graph_mode = -1;  // -1 auto (calls with >= 24 launches), 0 off, 1 on
  int64_t chunk_begin = 0, chunk_end = 0;
  std::vector<pgbp_stream_t> pipe_streams;
  std::vector<void*> pipe_events;  // cudaEvent_t: [0] fork, [1..] joins
  // Lazy zero of the sepsets: assignfactors! / reset leave the sepset rows unwritten and set this flag; the
  // first postorder traversal of a tree that covers every sepset treats their old value as 0 and writes
  // them (saves one write and one read of every sepset); anything else that looks at the state calls
  // batch_materialize_sepsets() first.
  bool sepsets_lazy_zero = false;
  // Lazy factor snapshot: assignfactors! copies every cluster belief into its ClusterFactor
  // (src/clustergraphbeliefs.jl:106).  K1 is a pure function of the prepared parameter / tip tables the
  // batch keeps on the device, so instead of copying (one read + one write of every cluster) the batch
  // remembers the call; the factors are produced by running K1 again into the factor array the first time
  // something reads them (factored_energy, get_factor).  Bit-identical by construction.  `valid` = the factors
  // (materialised or not) still equal K1's output for the remembered call: init_beliefs_reset_fromfactors! then
  // re-runs K1 straight into the beliefs (one write of every cluster) instead of copying (one read + one write).
  struct LazyFactors { bool pending = false; bool valid = false; int32_t ncolors = 1; int64_t nparamsets = 0, ndatasets = 0; int32_t pairing = 0; } lazy_factors;
  int32_t coop_mode = -1;  // medium shapes: -1 auto (cooperative), 0 thread-local generic, 4 / 8 lanes for m <= 16
  // pinned host bounce buffer for the small per-call results (status / iscal / log-likelihoods): a device-to-host
  // copy into pageable memory is staged by the driver synchronously; through pinned memory it is a plain DMA
  void* h_pinned = nullptr;
  size_t h_pinned_bytes = 0;
  int32_t* d_slot = nullptr;  // device scratch for transpose slot tables
  size_t d_slot_len = 0;
  void* d_sim = nullptr;  // pgbp_simulate: node descriptors of the last mem_parent table (pgbp_simulate.cu)
};
