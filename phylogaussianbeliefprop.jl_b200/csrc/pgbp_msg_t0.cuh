// K2 register-class ("T0", operands staged in shared memory) and thread-local generic ("T1") message kernels + their
// launchers.
// Included by several translation units (the 78 T0 shapes are split over three of them so that the
// library builds in about a minute instead of three).
#pragma once
#include "pgbp_bulk.cuh"
#include "pgbp_kernels.cuh"
#include "pgbp_launch.h"
#include "pgbp_shapes.h"

namespace pgbp {

#define PGBP_MSG_THREADS 128
#ifndef PGBP_STAGE_TILE
// elements per block of k_message_staged.  Measured on C2 (one B200, 1000 W): 64 -> 93.0 M calibrations/s, 32 -> 81.9 M
// (4 one-warp blocks per SM), the register kernel it replaced 89.9 M (DESIGN.md section 7)
#define PGBP_STAGE_TILE 64
#endif

#ifndef PGBP_HOST_EMUL
template <int MAXM>
__global__ void __launch_bounds__(PGBP_MSG_THREADS) k_message(MsgArgs a) {
  const int64_t e = a.e0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.B) return;
  message_thread_rt<MAXM>(a, blockIdx.y, e);
}

// Operand source of message_body_t0 in k_message_staged: row n of this element at tile[n * TILE].
template <int TILE>
struct T0Staged {
  const double* tile;
  const uint32_t* sslot;  // slot of every staged row
  PGBP_D uint32_t slot(int n) const { return sslot[n]; }
  PGBP_D double at(int n, uint32_t) const { return tile[n * TILE]; }
};

// Register class (i >= 1, i + s <= 12) with its operands staged in shared memory.  One thread per element
// keeps too few loads in flight: the register body needs 170-250 registers, so only 8 warps fit on an SM, each
// with 24 loads outstanding (long-scoreboard stalls, 1.2-2.3 TB/s per launch).  Here a block of TILE threads owns
// TILE consecutive elements of ONE message.  With the batch-innermost layout every row the message reads (T0Rows:
// sender J, h, g, receiver rows at the sepset's positions, old sepset) is one contiguous segment of 8 TILE bytes,
// so thread n issues one cp.async.bulk per row n, n + TILE, ..., all complete on one mbarrier, and the whole tile
// (201 rows = 103 KB for (i,s) = (3,9) at 64 elements) is in flight at once without holding a register.  The
// arithmetic is then message_body_t0 with operands read from shared memory (conflict-free: lane = element):
// bit-identical results.
// Outputs are plain coalesced per-thread stores.  Elements in [B, ld), failed or done elements are staged but
// never written.
template <int CI, int CS>
__global__ void __launch_bounds__(PGBP_STAGE_TILE) k_message_staged(MsgArgs a) {
  constexpr int TILE = PGBP_STAGE_TILE;
  using R = T0Rows<CI, CS>;
  extern __shared__ __align__(128) double sm[];
  __shared__ uint32_t sslot[R::N];
  __shared__ __align__(8) unsigned long long mbar;
  const int tid = threadIdx.x;
  const MsgDesc md = a.msgs[blockIdx.y];
  const int nrows = (a.opts & PGBP_OPT_SEPZERO) ? R::SG : R::N;
  const int64_t e0 = a.e0 + (int64_t)blockIdx.x * TILE, e = e0 + tid;
  const int64_t left = a.ld - e0;  // rows are cut at the pitch
  const uint32_t rowbytes = (uint32_t)(left < TILE ? left : TILE) * 8u;
  const uint32_t ld8 = (uint32_t)(a.ld * 8);
  if (tid == 0) {
    mbar_init(&mbar, 1);
    mbar_expect_tx(&mbar, (unsigned)nrows * rowbytes);
  }
  __syncthreads();
  const char* tileb = (const char*)(a.state + e0);
  const int32_t* __restrict__ gat = a.tab + md.gat;
  const int32_t* __restrict__ sca = a.tab + md.sca;
  for (int n = tid; n < nrows; n += TILE) {
    const uint32_t slot = R::slot(md, gat, sca, n);
    sslot[n] = slot;
    bulk_g2s(sm + (size_t)n * TILE, tileb + (uint64_t)slot * (uint64_t)ld8, rowbytes, &mbar);
  }
  const bool active = e < a.B && a.status[e] == 0 && !(a.done && a.done[e]);
  __syncthreads();      // sslot
  mbar_wait(&mbar, 0);  // every row has landed (no thread leaves the block before that)
  if (!active) return;
  message_body_t0<CI, CS>(a, md, e, T0Staged<TILE>{sm + tid, sslot});
}
#endif

// generic runtime-shape kernel (message_thread_rt), sender dimension <= MAXM
template <int MAXM>
static inline int launch_message(pgbp_batch* b, const MsgArgs& a, int nmsg) {
#ifdef PGBP_HOST_EMUL
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_rt<MAXM>(a, m, e);
#else
  dim3 grid((unsigned)((a.B - a.e0 + PGBP_MSG_THREADS - 1) / PGBP_MSG_THREADS), (unsigned)nmsg);
  k_message<MAXM><<<grid, PGBP_MSG_THREADS, 0, b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message");
}

// register class, shape (CI, CS): k_message_staged on the device, message_thread_t0 in the host emulation
template <int CI, int CS>
static inline int launch_message_staged(pgbp_batch* b, const MsgArgs& a, int nmsg) {
#ifdef PGBP_HOST_EMUL
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_t0<CI, CS>(a, m, e);
#else
  constexpr int TILE = PGBP_STAGE_TILE;
  using R = T0Rows<CI, CS>;
  // bulk copies move 16-byte aligned multiples of 16 bytes: even pitch (batches use multiples of 32), tiles that
  // start at multiples of TILE (element chunks start at multiples of 128)
  if (a.ld % 2 != 0 || a.e0 % TILE != 0) PGBP_FAIL(PGBP_ESTATE, "k_message_staged: rows not 16-byte aligned");
  const int nrows = (a.opts & PGBP_OPT_SEPZERO) ? R::SG : R::N;
  static AttrOnce attr;  // per instantiation and device
  if (attr.first())
    PGBP_CUDA(cudaFuncSetAttribute(k_message_staged<CI, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(sizeof(double) * R::N * TILE)));
  dim3 grid((unsigned)((a.B - a.e0 + TILE - 1) / TILE), (unsigned)nmsg);
  k_message_staged<CI, CS><<<grid, TILE, sizeof(double) * (size_t)nrows * TILE, b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message_staged");
}

// parts of the T0 shape table (pgbp_message_t0.cu compiled with -DPGBP_T0_PART=0,1,2): return
// PGBP_NOT_MINE when (ci, cs) belongs to another part
#define PGBP_NOT_MINE 12345
int launch_t0_part0(pgbp_batch* b, const MsgArgs& a, int nmsg, int ci, int cs);
int launch_t0_part1(pgbp_batch* b, const MsgArgs& a, int nmsg, int ci, int cs);
int launch_t0_part2(pgbp_batch* b, const MsgArgs& a, int nmsg, int ci, int cs);
// medium / large shapes (pgbp_message_medium.cu): shared-memory, cooperative or generic kernel
int launch_medium(pgbp_batch* b, const MsgArgs& a, int nmsg, int I, int S);

}  // namespace pgbp
