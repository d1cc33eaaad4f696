// Cross-file internal entry points.
#pragma once
#include "pgbp_internal.h"

namespace pgbp {
struct MsgArgs;
const std::string& last_error();
int batch_upload_tables(pgbp_batch* b);
int batch_need_scratch(pgbp_batch* b, size_t bytes);
// AoS (host layout: src[e*K + k]) <-> SoA (dst[slot[k]*ld + e]); slot == nullptr
// means identity; slot[k] < 0 skips column k.  d_slot is a DEVICE table.
int aos_to_soa(pgbp_batch* b, const double* d_aos, int K, const int32_t* d_slot, double* d_soa, int64_t ld, int64_t gs = 0);
int soa_to_aos(pgbp_batch* b, const double* d_soa, int64_t ld, double* d_aos, int K, const int32_t* d_slot = nullptr, int64_t gs = 0);
int integrate_launch(pgbp_batch* b, int belief, double* d_mu_soa, double* d_norm, int64_t ld_out, double* d_cov_soa = nullptr);
int launch_group(pgbp_batch* b, MsgArgs a, const MsgDesc* d_msgs, const LaunchGroup& g);
void free_tables(pgbp_batch* b);
void sim_free(pgbp_batch* b);  // pgbp_simulate's cached node descriptors
// write the pending zeros of the sepset rows (no-op unless sepsets_lazy_zero)
int batch_materialize_sepsets(pgbp_batch* b);
// the sepsets become zero: lazily when `lazy`, else with a memset now
int batch_zero_sepsets(pgbp_batch* b, bool lazy);
// run the pending K1 into the factor array (no-op unless lazy_factors.pending)
int batch_materialize_factors(pgbp_batch* b);
// beliefs <- factors by re-running K1 into the state array; returns 1 if done, 0 if the factors are not K1's
// output any more (caller copies), < 0 on error
int batch_reset_by_assign(pgbp_batch* b);
// pinned host staging of at least `bytes` (nullptr when unavailable: host emulation, allocation failure)
void* batch_pinned(pgbp_batch* b, size_t bytes);
MsgArgs make_args(pgbp_batch* b, uint32_t opts, int32_t ref_base, bool use_done);
struct LaunchGroup;
int launch_kldiv(pgbp_batch* b, MsgArgs a, const MsgDesc* d_msgs, const LaunchGroup& g);
int launch_iscal(pgbp_batch* b, int it, int tr, int autostop);
// rows of belief i's h / g in the batch's element array: the plan's slots, or the compact numbering of a
// shared-precision batch (pgbp_batch::eh)
inline int64_t batch_hrow(const pgbp_batch* b, int i) { return b->jb ? b->eh[i] : b->plan->hslot[i]; }
inline int64_t batch_grow(const pgbp_batch* b, int i) { return b->jb ? b->eh[i] + b->plan->dim[i] : b->plan->gslot[i]; }
inline JSide batch_jside(const pgbp_batch* b) { return JSide{b->jb ? b->jb->state : nullptr, b->jb ? b->jb->ld : 0, b->group_size}; }
// shared-precision batches (pgbp_shared.cu)
int shared_create(pgbp_batch* b);    // group batch, compact layout, caches (called by pgbp_batch_create_shared)
void shared_destroy(pgbp_batch* b);
int shared_run_traversal(pgbp_batch* b, int tree, int dir, uint32_t opts, int32_t ref_base);
int shared_propagate(pgbp_batch* b, const MsgDesc& md_plan, uint32_t opts, int32_t ref_base);
// remap the h / g rows of a plan descriptor to the compact element numbering of shared-precision batch b
MsgDesc shared_remap(const pgbp_batch* b, const MsgDesc& m);
}  // namespace pgbp
