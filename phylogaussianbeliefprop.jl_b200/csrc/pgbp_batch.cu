// Batch = device state of B independent replicas of one cluster graph.
// HBM layout (DESIGN.md): structure-of-arrays, batch innermost.  Row k of an
// array is `ld` doubles (ld = B rounded up to 32 elements = 256 bytes), so a
// warp working on 32 consecutive elements reads one aligned 256-byte line per
// slot.  A belief owns S(m) rows of packed-upper J, m rows of h, 1 row of g.
#include <algorithm>

#include "pgbp_launch.h"
#include "pgbp_shapes.h"

using namespace pgbp;

namespace pgbp {

template <class T>
static int alloc(pgbp_batch* b, T** p, size_t n) {
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, n * sizeof(T)));
  *p = (T*)v;
  b->device_bytes += (int64_t)(n * sizeof(T));
  return 0;
}

int batch_need_scratch(pgbp_batch* b, size_t bytes) {
  if (bytes <= b->scratch_bytes) return 0;
  PGBP_TRY(stream_sync(b->stream));
  dev_free(b->scratch);
  b->device_bytes -= (int64_t)b->scratch_bytes;
  b->scratch = nullptr;
  b->scratch_bytes = 0;
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, bytes));
  b->scratch = (double*)v;
  b->scratch_bytes = bytes;
  b->device_bytes += (int64_t)bytes;
  return 0;
}

static int need_slot_table(pgbp_batch* b, size_t n) {
  if (n <= b->d_slot_len) return 0;
  PGBP_TRY(stream_sync(b->stream));
  dev_free(b->d_slot);
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, n * sizeof(int32_t)));
  b->d_slot = (int32_t*)v;
  b->d_slot_len = n;
  return 0;
}

void* batch_pinned(pgbp_batch* b, size_t bytes) {
#ifdef PGBP_HOST_EMUL
  (void)b; (void)bytes;
  return nullptr;
#else
  if (bytes <= b->h_pinned_bytes) return b->h_pinned;
  if (b->h_pinned) { cudaStreamSynchronize(b->stream); cudaFreeHost(b->h_pinned); b->h_pinned = nullptr; b->h_pinned_bytes = 0; }
  void* v = nullptr;
  if (cudaHostAlloc(&v, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  b->h_pinned = v;
  b->h_pinned_bytes = bytes;
  return v;
#endif
}

int batch_zero_sepsets(pgbp_batch* b, bool lazy) {
  const pgbp_plan* p = b->plan;
  if (lazy) { b->sepsets_lazy_zero = true; return 0; }
  if (b->jb) {  // shared-precision batch: J rows of the sepsets in the group batch, h / g rows here
    b->sepsets_lazy_zero = false;
    b->jb->stream = b->stream;
    PGBP_TRY(batch_zero_sepsets(b->jb, false));
    return dev_memset(b->state + (size_t)b->nrows_efactor * (size_t)b->ld, 0,
                      sizeof(double) * (size_t)(b->nrows_e - b->nrows_efactor) * (size_t)b->ld, b->stream);
  }
  b->sepsets_lazy_zero = false;
  return dev_memset(b->state + (size_t)p->nslots_factor * (size_t)b->ld, 0,
                    sizeof(double) * (size_t)(p->nslots_state - p->nslots_factor) * (size_t)b->ld, b->stream);
}
int batch_materialize_sepsets(pgbp_batch* b) {
  if (!b->sepsets_lazy_zero) return 0;
  return batch_zero_sepsets(b, false);
}

int batch_upload_tables(pgbp_batch* b) {
  const pgbp_plan* p = b->plan;
  PGBP_TRY(stream_sync(b->stream));
  dev_free(b->d_tab);
  b->d_tab = nullptr;
  void* v = nullptr;
  PGBP_TRY(dev_malloc(&v, std::max<size_t>(1, p->tab.size()) * sizeof(int32_t)));
  b->d_tab = (int32_t*)v;
  PGBP_TRY(h2d(b->d_tab, p->tab.data(), p->tab.size() * sizeof(int32_t), b->stream));
  return stream_sync(b->stream);
}

// ---- AoS <-> SoA transposes (32 x 32 shared-memory tiles) -----------------
#ifndef PGBP_HOST_EMUL
// gs > 1: the columns are J rows of a shared-precision batch -- they live in the group leader's column:
// the upload keeps the leader's values, the download broadcasts them to the whole group
__global__ void k_aos_to_soa(const double* __restrict__ aos, int K, const int32_t* __restrict__ slot,
                             double* __restrict__ soa, int64_t ld, int64_t B, int64_t gs) {
  __shared__ double tile[32][33];
  const int64_t e0 = (int64_t)blockIdx.x * 32;
  const int k0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t e = e0 + r;
    const int k = k0 + threadIdx.x;
    if (e < B && k < K) tile[r][threadIdx.x] = aos[e * K + k];
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int k = k0 + r;
    const int64_t e = e0 + threadIdx.x;
    if (e < B && k < K) {
      const int sl = slot ? slot[k] : k;
      if (sl >= 0 && (gs <= 1 || e % gs == 0)) soa[(int64_t)sl * ld + e] = tile[threadIdx.x][r];
    }
  }
}
__global__ void k_soa_to_aos(const double* __restrict__ soa, int64_t ld, const int32_t* __restrict__ slot,
                             double* __restrict__ aos, int K, int64_t B, int64_t gs) {
  __shared__ double tile[32][33];
  const int64_t e0 = (int64_t)blockIdx.x * 32;
  const int k0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int k = k0 + r;
    const int64_t e = e0 + threadIdx.x;
    if (e < B && k < K) {
      const int sl = slot ? slot[k] : k;
      tile[r][threadIdx.x] = soa[(int64_t)sl * ld + (gs > 1 ? e - e % gs : e)];
    }
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t e = e0 + r;
    const int k = k0 + threadIdx.x;
    if (e < B && k < K) aos[e * K + k] = tile[threadIdx.x][r];
  }
}
#endif

#ifndef PGBP_HOST_EMUL
__global__ void k_fill(double* p, int64_t n, double v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
#endif
static int fill(pgbp_batch* b, double* p, int64_t n, double v) {
  if (n <= 0) return 0;
#ifdef PGBP_HOST_EMUL
  for (int64_t i = 0; i < n; i++) p[i] = v;
#else
  k_fill<<<(unsigned)((n + 255) / 256), 256, 0, b->stream>>>(p, n, v);
#endif
  b->launches++;
  return check_launch("k_fill");
}

int aos_to_soa(pgbp_batch* b, const double* d_aos, int K, const int32_t* d_slot, double* d_soa, int64_t ld, int64_t gs) {
  if (K <= 0) return 0;
#ifdef PGBP_HOST_EMUL
  for (int64_t e = 0; e < b->B; e++)
    for (int k = 0; k < K; k++) {
      const int sl = d_slot ? d_slot[k] : k;
      if (sl >= 0 && (gs <= 1 || e % gs == 0)) d_soa[(int64_t)sl * ld + e] = d_aos[e * K + k];
    }
#else
  dim3 grid((unsigned)((b->B + 31) / 32), (unsigned)((K + 31) / 32));
  k_aos_to_soa<<<grid, dim3(32, 8), 0, b->stream>>>(d_aos, K, d_slot, d_soa, ld, b->B, gs);
#endif
  b->launches++;
  return check_launch("k_aos_to_soa");
}

int soa_to_aos(pgbp_batch* b, const double* d_soa, int64_t ld, double* d_aos, int K, const int32_t* d_slot, int64_t gs) {
  if (K <= 0) return 0;
#ifdef PGBP_HOST_EMUL
  for (int64_t e = 0; e < b->B; e++)
    for (int k = 0; k < K; k++) d_aos[e * K + k] = d_soa[(int64_t)(d_slot ? d_slot[k] : k) * ld + (gs > 1 ? e - e % gs : e)];
#else
  dim3 grid((unsigned)((b->B + 31) / 32), (unsigned)((K + 31) / 32));
  k_soa_to_aos<<<grid, dim3(32, 8), 0, b->stream>>>(d_soa, ld, d_slot, d_aos, K, b->B, gs);
#endif
  b->launches++;
  return check_launch("k_soa_to_aos");
}

// copy K host columns <-> device rows given by `slots` (host table)
static int put_columns(pgbp_batch* b, const double* host, int K, const std::vector<int32_t>& slots, double* d_soa,
                       int64_t gs = 0) {
  if (K <= 0) return 0;
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (size_t)b->B * K));
  PGBP_TRY(need_slot_table(b, K));
  PGBP_TRY(h2d(b->scratch, host, sizeof(double) * (size_t)b->B * K, b->stream));
  PGBP_TRY(h2d(b->d_slot, slots.data(), sizeof(int32_t) * K, b->stream));
  PGBP_TRY(aos_to_soa(b, b->scratch, K, b->d_slot, d_soa, b->ld, gs));
  return stream_sync(b->stream);  // `slots` may be a temporary
}
static int get_columns(pgbp_batch* b, double* host, int K, const std::vector<int32_t>& slots, const double* d_soa,
                       int64_t gs = 0) {
  if (K <= 0) return 0;
  PGBP_TRY(batch_need_scratch(b, sizeof(double) * (size_t)b->B * K));
  PGBP_TRY(need_slot_table(b, K));
  PGBP_TRY(h2d(b->d_slot, slots.data(), sizeof(int32_t) * K, b->stream));
  PGBP_TRY(soa_to_aos(b, d_soa, b->ld, b->scratch, K, b->d_slot, gs));
  PGBP_TRY(d2h(host, b->scratch, sizeof(double) * (size_t)b->B * K, b->stream));
  return stream_sync(b->stream);
}

static void square_slots(int m, int64_t base, bool upper_only, std::vector<int32_t>* out) {
  out->resize((size_t)m * m);
  for (int c = 0; c < m; c++)
    for (int r = 0; r < m; r++) {
      int32_t v;
      if (r <= c) v = (int32_t)(base + pk(r, c));
      else v = upper_only ? -1 : (int32_t)(base + pk(c, r));
      (*out)[(size_t)c * m + r] = v;
    }
}

static int access_hJg(pgbp_batch* b, bool put, double* d_arr, int m, int64_t js, int64_t hs, int64_t gs,
                      double* J, double* h, double* g) {
  PGBP_TRY(set_device(b->device));
  if (d_arr == b->state) PGBP_TRY(batch_materialize_sepsets(b));
  std::vector<int32_t> sl;
  if (J && m > 0) {
    square_slots(m, js, put, &sl);
    PGBP_TRY(put ? put_columns(b, J, m * m, sl, d_arr) : get_columns(b, J, m * m, sl, d_arr));
  }
  if (h && m > 0) {
    sl.resize(m);
    for (int k = 0; k < m; k++) sl[k] = (int32_t)(hs + k);
    PGBP_TRY(put ? put_columns(b, h, m, sl, d_arr) : get_columns(b, h, m, sl, d_arr));
  }
  if (g && gs >= 0) {
    if (put) PGBP_TRY(h2d(d_arr + gs * b->ld, g, sizeof(double) * b->B, b->stream));
    else PGBP_TRY(d2h(g, d_arr + gs * b->ld, sizeof(double) * b->B, b->stream));
    PGBP_TRY(stream_sync(b->stream));
  }
  return 0;
}

}  // namespace pgbp

extern "C" {

int32_t pgbp_batch_create(const pgbp_plan* plan, int64_t B, int32_t device, uint32_t flags, pgbp_batch** out) {
  return pgbp_batch_create_shared(plan, B, 0, device, flags, out);
}

// ld_align: row pitch granularity in elements (32 = 256-byte rows; the group batch of a shared-precision batch
// uses 4, or 1 below four groups: it is addressed per (message, group), not per warp of elements, and with ONE group
// a pitch of 4 would leave 8 useful bytes in every 32-byte sector -- the group pass of C5 was DRAM-bound on that)
static int batch_create_impl(const pgbp_plan* plan, int64_t B, int64_t group_size, int32_t device, uint32_t flags,
                             int64_t ld_align, pgbp_batch** out) {
  if (!plan || !out || B <= 0) PGBP_FAIL(PGBP_EINVAL, "bad arguments");
  if (group_size < 0 || (group_size > 1 && B % group_size != 0))
    PGBP_FAIL(PGBP_EINVAL, "group size must divide the batch size");
  if (plan->nslots_state >= (int64_t)1 << 31 || plan->nslots_resid >= (int64_t)1 << 31)
    PGBP_FAIL(PGBP_EINVAL, "cluster graph too large for int32 slot tables");
  if ((B + 31) / 32 * 32 * 8 >= (int64_t)1 << 32) PGBP_FAIL(PGBP_EINVAL, "batch too large: row pitch must stay below 4 GiB");
  PGBP_TRY(set_device(device));
  // any failure below releases the stream and every device buffer allocated so far
  struct Destroy { void operator()(pgbp_batch* x) const { pgbp_batch_destroy(x); } };
  std::unique_ptr<pgbp_batch, Destroy> b(new pgbp_batch);
  b->plan = plan;
  b->B = B;
  b->ld = (B + ld_align - 1) / ld_align * ld_align;
  b->device = device;
  b->flags = flags;
  b->group_size = group_size > 1 ? group_size : 0;
#ifndef PGBP_HOST_EMUL
  PGBP_CUDA(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
  b->own_stream = true;
#endif
  if (b->group_size > 1) {
    // shared-precision batch: h, g per element here (compact rows), every J row once per group in `jb`
    PGBP_TRY(shared_create(b.get()));
    pgbp_batch* jb = nullptr;
    PGBP_TRY(batch_create_impl(plan, B / group_size, 0, device, flags, B / group_size >= 4 ? 4 : 1, &jb));
    b->jb = jb;
    PGBP_TRY(pgbp_batch_set_stream(jb, (void*)b->stream));  // one stream, program order
    b->device_bytes += jb->device_bytes;
    if (flags & PGBP_BATCH_RESIDUALS) PGBP_TRY(pgbp_reset_calibration_flags(b.get(), 1));
    *out = b.release();
    return 0;
  }
  const size_t ld = (size_t)b->ld;
  PGBP_TRY(alloc(b.get(), &b->state, (size_t)plan->nslots_state * ld));
  PGBP_TRY(dev_memset(b->state, 0, sizeof(double) * (size_t)plan->nslots_state * ld, b->stream));
  if (flags & PGBP_BATCH_FACTORS) {
    PGBP_TRY(alloc(b.get(), &b->factor, (size_t)plan->nslots_factor * ld));
    PGBP_TRY(dev_memset(b->factor, 0, sizeof(double) * (size_t)plan->nslots_factor * ld, b->stream));
  }
  if (flags & PGBP_BATCH_RESIDUALS) {
    const size_t nd = 2 * (size_t)plan->nsepsets;
    PGBP_TRY(alloc(b.get(), &b->resid, std::max<size_t>(1, (size_t)plan->nslots_resid) * ld));
    PGBP_TRY(dev_memset(b->resid, 0, sizeof(double) * std::max<size_t>(1, (size_t)plan->nslots_resid) * ld, b->stream));
    PGBP_TRY(alloc(b.get(), &b->kldiv, std::max<size_t>(1, nd) * ld));
    PGBP_TRY(alloc(b.get(), &b->calflag, std::max<size_t>(1, nd) * ld));
    PGBP_TRY(alloc(b.get(), &b->done, ld));
    PGBP_TRY(alloc(b.get(), &b->iscal, ld));
    PGBP_TRY(alloc(b.get(), &b->itertree, 2 * ld));
    PGBP_TRY(dev_memset(b->done, 0, ld, b->stream));
    PGBP_TRY(dev_memset(b->iscal, 0, sizeof(int32_t) * ld, b->stream));
    PGBP_TRY(dev_memset(b->itertree, 0, sizeof(int32_t) * 2 * ld, b->stream));
  }
  PGBP_TRY(alloc(b.get(), &b->status, ld));
  PGBP_TRY(dev_memset(b->status, 0, sizeof(int32_t) * ld, b->stream));
  PGBP_TRY(alloc(b.get(), &b->d_one, 1));
  PGBP_TRY(batch_upload_tables(b.get()));
  b->device_bytes += (int64_t)(plan->tab.size() * sizeof(int32_t));
  b->d_msgs.assign(2 * plan->trees.size(), nullptr);
  for (size_t t = 0; t < plan->trees.size(); t++)
    for (int dir = 0; dir < 2; dir++) {
      const Traversal& tv = plan->trees[t].trav[dir];
      PGBP_TRY(alloc(b.get(), &b->d_msgs[2 * t + dir], std::max<size_t>(1, tv.msgs.size())));
      PGBP_TRY(h2d(b->d_msgs[2 * t + dir], tv.msgs.data(), tv.msgs.size() * sizeof(MsgDesc), b->stream));
    }
  b->d_step_off.assign(2 * plan->trees.size(), nullptr);
  for (size_t t = 0; t < plan->trees.size(); t++)
    for (int dir = 0; dir < 2; dir++) {
      const auto& so = plan->trees[t].trav[dir].step_off;
      PGBP_TRY(alloc(b.get(), &b->d_step_off[2 * t + dir], std::max<size_t>(1, so.size())));
      PGBP_TRY(h2d(b->d_step_off[2 * t + dir], so.data(), so.size() * sizeof(int32_t), b->stream));
    }
  b->d_tw.assign(2 * plan->trees.size(), nullptr);
  b->d_stage_off.assign(2 * plan->trees.size(), nullptr);
  for (size_t t = 0; t < plan->trees.size(); t++)
    for (int dir = 0; dir < 2; dir++) {
      const Traversal& tv = plan->trees[t].trav[dir];
      if (tv.tw.empty()) continue;
      PGBP_TRY(alloc(b.get(), &b->d_tw[2 * t + dir], tv.tw.size()));
      PGBP_TRY(h2d(b->d_tw[2 * t + dir], tv.tw.data(), tv.tw.size() * sizeof(TwDesc), b->stream));
      PGBP_TRY(alloc(b.get(), &b->d_stage_off[2 * t + dir], tv.stage_off.size()));
      PGBP_TRY(h2d(b->d_stage_off[2 * t + dir], tv.stage_off.data(), tv.stage_off.size() * sizeof(int32_t), b->stream));
    }
  b->d_walk.assign(plan->trees.size(), nullptr);
  for (size_t t = 0; t < plan->trees.size(); t++) {
    const auto& w = plan->trees[t].walk;
    PGBP_TRY(alloc(b.get(), &b->d_walk[t], std::max<size_t>(1, w.size())));
    PGBP_TRY(h2d(b->d_walk[t], w.data(), w.size() * sizeof(MsgDesc), b->stream));
  }
  PGBP_TRY(stream_sync(b->stream));
  if (flags & PGBP_BATCH_RESIDUALS) PGBP_TRY(pgbp_reset_calibration_flags(b.get(), 1));
  *out = b.release();  // only after the last fallible step
  return 0;
}

int32_t pgbp_batch_create_shared(const pgbp_plan* plan, int64_t B, int64_t group_size, int32_t device, uint32_t flags,
                                 pgbp_batch** out) {
  return batch_create_impl(plan, B, group_size, device, flags, 32, out);
}

int32_t pgbp_batch_destroy(pgbp_batch* b) {
  if (!b) return 0;
  set_device(b->device);
  stream_sync(b->stream);
  dev_free(b->state); dev_free(b->factor); dev_free(b->resid); dev_free(b->kldiv);
  dev_free(b->calflag); dev_free(b->calflagJ); dev_free(b->done); dev_free(b->status); dev_free(b->iscal); dev_free(b->itertree);
  dev_free(b->d_tab); dev_free(b->d_one); dev_free(b->scratch); dev_free(b->d_slot); free_tables(b); sim_free(b);
  shared_destroy(b);
  for (auto* p : b->d_msgs) dev_free(p);
  for (auto* p : b->d_walk) dev_free(p);
  for (auto* p : b->d_step_off) dev_free(p);
  for (auto* p : b->d_tw) dev_free(p);
  for (auto* p : b->d_stage_off) dev_free(p);
#ifndef PGBP_HOST_EMUL
  for (auto& kv : b->graphs) if (kv.second.exec) cudaGraphExecDestroy((cudaGraphExec_t)kv.second.exec);
  for (auto s : b->pipe_streams) cudaStreamDestroy(s);
  for (auto ev : b->pipe_events) cudaEventDestroy((cudaEvent_t)ev);
  if (b->own_stream) cudaStreamDestroy(b->stream);
  if (b->h_pinned) cudaFreeHost(b->h_pinned);
#endif
  delete b;
  return 0;
}

int32_t pgbp_batch_set_stream(pgbp_batch* b, void* s) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  PGBP_TRY(stream_sync(b->stream));
#ifndef PGBP_HOST_EMUL
  if (b->own_stream) cudaStreamDestroy(b->stream);
  b->stream = (cudaStream_t)s;
#endif
  b->own_stream = false;
  if (b->jb) b->jb->stream = b->stream;
  return 0;
}

int32_t pgbp_batch_synchronize(pgbp_batch* b) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  return stream_sync(b->stream);
}
int64_t pgbp_batch_size(const pgbp_batch* b) { return b ? b->B : 0; }
int64_t pgbp_batch_device_bytes(const pgbp_batch* b) { return b ? b->device_bytes : 0; }
int64_t pgbp_batch_launch_count(pgbp_batch* b, int32_t reset) {
  if (!b) return 0;
  const int64_t n = b->launches;
  if (reset) b->launches = 0;
  return n;
}

// shared-precision batches: J of a belief / factor / residual lives once per group in the group batch.  Host side:
// set takes each group's FIRST element, get broadcasts the group's matrix to its elements.
static int shared_put_J(pgbp_batch* b, int m, const double* J, int (*put)(pgbp_batch*, int32_t, const double*), int32_t idx) {
  const size_t mm = (size_t)m * m;
  std::vector<double> Jg((size_t)b->ngroups * mm);
  for (int64_t g = 0; g < b->ngroups; g++) memcpy(Jg.data() + g * mm, J + (size_t)(g * b->group_size) * mm, sizeof(double) * mm);
  return put(b->jb, idx, Jg.data());
}
static void shared_broadcast_J(const pgbp_batch* b, int m, const std::vector<double>& Jg, double* J) {
  const size_t mm = (size_t)m * m;
  for (int64_t e = 0; e < b->B; e++) memcpy(J + (size_t)e * mm, Jg.data() + (size_t)(e / b->group_size) * mm, sizeof(double) * mm);
}

int32_t pgbp_set_belief(pgbp_batch* b, int32_t i, const double* J, const double* h, const double* g) {
  if (!b || i < 0 || i >= b->plan->nbeliefs) PGBP_FAIL(PGBP_EINVAL, "bad batch / belief index");
  const pgbp_plan* p = b->plan;
  if (b->jb) {
    b->jb->stream = b->stream;
    PGBP_TRY(set_device(b->device));
    PGBP_TRY(batch_materialize_sepsets(b));
    if (J && p->dim[i] > 0)
      PGBP_TRY(shared_put_J(b, p->dim[i], J, [](pgbp_batch* jb, int32_t k, const double* Jg) { return (int)pgbp_set_belief(jb, k, Jg, nullptr, nullptr); }, i));
    return access_hJg(b, true, b->state, p->dim[i], 0, batch_hrow(b, i), batch_grow(b, i), nullptr, (double*)h, (double*)g);
  }
  return access_hJg(b, true, b->state, p->dim[i], p->jslot[i], p->hslot[i], p->gslot[i], (double*)J, (double*)h, (double*)g);
}
int32_t pgbp_get_belief(pgbp_batch* b, int32_t i, double* J, double* h, double* g) {
  if (!b || i < 0 || i >= b->plan->nbeliefs) PGBP_FAIL(PGBP_EINVAL, "bad batch / belief index");
  const pgbp_plan* p = b->plan;
  if (b->jb) {
    b->jb->stream = b->stream;
    PGBP_TRY(set_device(b->device));
    PGBP_TRY(batch_materialize_sepsets(b));
    if (J && p->dim[i] > 0) {
      std::vector<double> Jg((size_t)b->ngroups * p->dim[i] * p->dim[i]);
      PGBP_TRY(pgbp_get_belief(b->jb, i, Jg.data(), nullptr, nullptr));
      shared_broadcast_J(b, p->dim[i], Jg, J);
    }
    return access_hJg(b, false, b->state, p->dim[i], 0, batch_hrow(b, i), batch_grow(b, i), nullptr, h, g);
  }
  return access_hJg(b, false, b->state, p->dim[i], p->jslot[i], p->hslot[i], p->gslot[i], J, h, g);
}
int32_t pgbp_get_factor(pgbp_batch* b, int32_t i, double* J, double* h, double* g) {
  if (!b || i < 0 || i >= b->plan->nclusters) PGBP_FAIL(PGBP_EINVAL, "bad batch / cluster index");
  if (!b->factor) PGBP_FAIL(PGBP_ESTATE, "batch was created without PGBP_BATCH_FACTORS");
  const pgbp_plan* p = b->plan;
  PGBP_TRY(set_device(b->device));
  if (b->jb) {
    b->jb->stream = b->stream;
    if (J && p->dim[i] > 0) {
      std::vector<double> Jg((size_t)b->ngroups * p->dim[i] * p->dim[i]);
      PGBP_TRY(pgbp_get_factor(b->jb, i, Jg.data(), nullptr, nullptr));
      shared_broadcast_J(b, p->dim[i], Jg, J);
    }
    return access_hJg(b, false, b->factor, p->dim[i], 0, batch_hrow(b, i), batch_grow(b, i), nullptr, h, g);
  }
  PGBP_TRY(batch_materialize_factors(b));
  return access_hJg(b, false, b->factor, p->dim[i], p->jslot[i], p->hslot[i], p->gslot[i], J, h, g);
}
int32_t pgbp_get_residual(pgbp_batch* b, int32_t j, int32_t to_cluster, double* dJ, double* dh, uint8_t* iscal_resid,
                          double* kldiv) {
  if (!b || j < 0 || j >= b->plan->nsepsets) PGBP_FAIL(PGBP_EINVAL, "bad batch / sepset index");
  if (!b->resid) PGBP_FAIL(PGBP_ESTATE, "batch was created without PGBP_BATCH_RESIDUALS");
  const pgbp_plan* p = b->plan;
  int side;
  if (to_cluster == p->sep_a[j]) side = 0;
  else if (to_cluster == p->sep_b[j]) side = 1;
  else PGBP_FAIL(PGBP_EINVAL, "cluster %d is not an end of sepset %d", to_cluster, j);
  const int d = 2 * j + side;
  const int s = p->dim[p->nclusters + j];
  if (b->jb) {
    b->jb->stream = b->stream;
    std::vector<uint8_t> fJ((size_t)b->ngroups);
    if (dJ && s > 0) {
      std::vector<double> Jg((size_t)b->ngroups * s * s);
      PGBP_TRY(pgbp_get_residual(b->jb, j, to_cluster, Jg.data(), nullptr, nullptr, nullptr));
      shared_broadcast_J(b, s, Jg, dJ);
    }
    PGBP_TRY(access_hJg(b, false, b->resid, s, 0, b->erh[d], -1, nullptr, dh, nullptr));
    if (iscal_resid) {  // flag of the message = h part (element) AND J part (group)
      PGBP_TRY(d2h(iscal_resid, b->calflag + (int64_t)d * b->ld, (size_t)b->B, b->stream));
      PGBP_TRY(d2h(fJ.data(), b->jb->calflag + (int64_t)d * b->jb->ld, (size_t)b->ngroups, b->stream));
    }
    if (kldiv) PGBP_TRY(d2h(kldiv, b->kldiv + (int64_t)d * b->ld, sizeof(double) * (size_t)b->B, b->stream));
    PGBP_TRY(stream_sync(b->stream));
    if (iscal_resid) for (int64_t e = 0; e < b->B; e++) iscal_resid[e] = iscal_resid[e] && fJ[e / b->group_size];
    return 0;
  }
  PGBP_TRY(access_hJg(b, false, b->resid, s, p->rjslot[d], p->rhslot[d], -1, dJ, dh, nullptr));
  if (iscal_resid) PGBP_TRY(d2h(iscal_resid, b->calflag + (int64_t)d * b->ld, (size_t)b->B, b->stream));
  if (kldiv) PGBP_TRY(d2h(kldiv, b->kldiv + (int64_t)d * b->ld, sizeof(double) * (size_t)b->B, b->stream));
  return stream_sync(b->stream);
}
int32_t pgbp_get_status(pgbp_batch* b, int32_t* status) {
  if (!b || !status) PGBP_FAIL(PGBP_EINVAL, "null argument");
  PGBP_TRY(set_device(b->device));
  int32_t* pin = (int32_t*)batch_pinned(b, sizeof(int32_t) * (size_t)b->B);
  PGBP_TRY(d2h(pin ? pin : status, b->status, sizeof(int32_t) * (size_t)b->B, b->stream));
  PGBP_TRY(stream_sync(b->stream));
  if (pin) memcpy(status, pin, sizeof(int32_t) * (size_t)b->B);
  return 0;
}
int32_t pgbp_clear_status(pgbp_batch* b) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  PGBP_TRY(set_device(b->device));
  return dev_memset(b->status, 0, sizeof(int32_t) * (size_t)b->ld, b->stream);
}

int32_t pgbp_reset_beliefs(pgbp_batch* b) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  PGBP_TRY(set_device(b->device));
  b->sepsets_lazy_zero = false;
  if (b->jb) {
    b->jb->stream = b->stream;
    PGBP_TRY(pgbp_reset_beliefs(b->jb));
    return dev_memset(b->state, 0, sizeof(double) * (size_t)b->nrows_e * (size_t)b->ld, b->stream);
  }
  return dev_memset(b->state, 0, sizeof(double) * (size_t)b->plan->nslots_state * (size_t)b->ld, b->stream);
}
int32_t pgbp_factors_from_beliefs(pgbp_batch* b) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  if (!b->factor) PGBP_FAIL(PGBP_ESTATE, "batch was created without PGBP_BATCH_FACTORS");
  PGBP_TRY(set_device(b->device));
  b->lazy_factors.pending = false;
  b->lazy_factors.valid = false;
  if (b->jb) {
    b->jb->stream = b->stream;
    PGBP_TRY(pgbp_factors_from_beliefs(b->jb));
    return d2d(b->factor, b->state, sizeof(double) * (size_t)b->nrows_efactor * (size_t)b->ld, b->stream);
  }
  return d2d(b->factor, b->state, sizeof(double) * (size_t)b->plan->nslots_factor * (size_t)b->ld, b->stream);
}
int32_t pgbp_reset_from_factors(pgbp_batch* b) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  if (!b->factor) PGBP_FAIL(PGBP_ESTATE, "batch was created without PGBP_BATCH_FACTORS");
  PGBP_TRY(set_device(b->device));
  const pgbp_plan* p = b->plan;
  const size_t ld = (size_t)b->ld;
  if (b->jb) {
    b->jb->stream = b->stream;
    PGBP_TRY(pgbp_reset_from_factors(b->jb));
    PGBP_TRY(batch_materialize_sepsets(b->jb));  // (the group batch's own laziness is not used: one flag, this batch's)
    PGBP_TRY(d2d(b->state, b->factor, sizeof(double) * (size_t)b->nrows_efactor * ld, b->stream));
    return batch_zero_sepsets(b, true);
  }
  {  // factors that are still K1's output: re-run K1 into the beliefs (write only) instead of copying
    const int r = batch_reset_by_assign(b);
    if (r < 0) return r;
    if (r == 1) return batch_zero_sepsets(b, true);
  }
  PGBP_TRY(batch_materialize_factors(b));
  PGBP_TRY(d2d(b->state, b->factor, sizeof(double) * (size_t)p->nslots_factor * ld, b->stream));
  return batch_zero_sepsets(b, true);
}
int32_t pgbp_reset_calibration_flags(pgbp_batch* b, int32_t reset_kl) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  if (!b->calflag) PGBP_FAIL(PGBP_ESTATE, "batch was created without PGBP_BATCH_RESIDUALS");
  PGBP_TRY(set_device(b->device));
  // empty messages are born calibrated and are never reset (src/beliefs.jl:919-922, 973-974)
  const pgbp_plan* p = b->plan;
  if (b->jb) {
    b->jb->stream = b->stream;
    PGBP_TRY(pgbp_reset_calibration_flags(b->jb, 0));
  }
  PGBP_TRY(dev_memset(b->calflag, 0, 2 * (size_t)p->nsepsets * (size_t)b->ld, b->stream));
  if (b->calflagJ) PGBP_TRY(dev_memset(b->calflagJ, 0, 2 * (size_t)p->nsepsets * (size_t)b->ld, b->stream));
  for (int j = 0; j < p->nsepsets; j++)
    if (p->dim[p->nclusters + j] == 0) {
      PGBP_TRY(dev_memset(b->calflag + (int64_t)2 * j * b->ld, 1, 2 * (size_t)b->ld, b->stream));
      if (b->calflagJ) PGBP_TRY(dev_memset(b->calflagJ + (int64_t)2 * j * b->ld, 1, 2 * (size_t)b->ld, b->stream));
    }
  if (reset_kl && b->kldiv) {  // kldiv <- -1, 0 for empty messages (src/beliefs.jl:908-922, 975)
    PGBP_TRY(fill(b, b->kldiv, (int64_t)2 * p->nsepsets * b->ld, -1.0));
    for (int j = 0; j < p->nsepsets; j++)
      if (p->dim[p->nclusters + j] == 0) PGBP_TRY(fill(b, b->kldiv + (int64_t)2 * j * b->ld, 2 * b->ld, 0.0));
  }
  return 0;
}

int32_t pgbp_batch_belief_rows(const pgbp_batch* b, int32_t belief, int64_t* hrow, int64_t* grow) {
  if (!b || belief < 0 || belief >= b->plan->nbeliefs) PGBP_FAIL(PGBP_EINVAL, "bad batch / belief index");
  if (hrow) *hrow = batch_hrow(b, belief);
  if (grow) *grow = batch_grow(b, belief);
  return 0;
}

int32_t pgbp_device_view(pgbp_batch* b, double** base, int64_t* ld, int64_t* nslots) {
  if (!b) PGBP_FAIL(PGBP_EINVAL, "null batch");
  PGBP_TRY(set_device(b->device));
  PGBP_TRY(batch_materialize_sepsets(b));  // the caller may read any row
  if (base) *base = b->state;
  if (ld) *ld = b->ld;
  // (shared-precision batches: the element array holds h and g only, in compact rows -- pgbp_batch_belief_rows)
  if (nslots) *nslots = b->jb ? b->nrows_e : b->plan->nslots_state;
  return 0;
}

}  // extern "C"
