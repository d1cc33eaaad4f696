// K2 for medium / large message shapes (sender dimension > 12): shared-memory kernel, cooperative
// kernel, thread-local generic kernel -- and the choice between them.
#include "pgbp_coop.cuh"
#include "pgbp_msg_t0.cuh"

namespace pgbp {

template <int MAXM, int G>
static int launch_coop(pgbp_batch* b, const MsgArgs& a, int nmsg) {
#ifdef PGBP_HOST_EMUL
  // host emulation: the generic body gives bit-identical results (same per-entry update order)
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_rt<MAXM>(a, m, e);
#else
  constexpr int RPB = 128 / G;
  dim3 grid((unsigned)((a.B - a.e0 + RPB - 1) / RPB), (unsigned)nmsg);
  k_message_coop<MAXM, G><<<grid, 128, 0, b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message_coop");
}

#define PGBP_SMEM_LIMIT (200 * 1024)
// EXACT: I is the compile-time integrated dimension (k_message_smem<I>), else an upper bound
// (k_message_smem_rt<MAXI>)
template <int MAXI, bool EXACT>
static int launch_smem(pgbp_batch* b, const MsgArgs& a, int nmsg, int I, int S) {
#ifdef PGBP_HOST_EMUL
  (void)I; (void)S;
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_rt<PGBP_MAX_DIM>(a, m, e);
#else
  static AttrOnce attr_done, attr8_done;  // per instantiation and device
  const bool s8 = EXACT && S <= 8 && MAXI <= 10;  // fully unrolled kept-block loops (register budget: I <= 10)
  const void* fn;
  if constexpr (EXACT) fn = s8 ? (const void*)k_message_smem<MAXI, 8> : (const void*)k_message_smem<MAXI, 0>;
  else fn = (const void*)k_message_smem_rt<MAXI>;
  if (s8 ? attr8_done.first() : attr_done.first())
    PGBP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, PGBP_SMEM_LIMIT));
  if (a.ld * 8 >= ((int64_t)1 << 32)) PGBP_FAIL(PGBP_ESTATE, "batch too large for 32-bit row pitch");
  const size_t bytes = smem_block_bytes(I, S);
  dim3 grid((unsigned)((a.B - a.e0 + 31) / 32), (unsigned)nmsg);
  if constexpr (EXACT) {
    if (s8) k_message_smem<MAXI, 8><<<grid, 32, bytes, b->stream>>>(a);
    else k_message_smem<MAXI, 0><<<grid, 32, bytes, b->stream>>>(a);
  } else {
    k_message_smem_rt<MAXI><<<grid, 32, bytes, b->stream>>>(a);
  }
#endif
  b->launches++;
  return check_launch("k_message_smem");
}


// multi-warp shared-memory kernel (large I): NW warps per tile of 32 elements
#define PGBP_SMEM_MW_LIMIT (225 * 1024)
static size_t mw_bytes(int I, int S, int NW) {  // == smem_mw_block_bytes (pgbp_coop.cuh, device build only)
  const int M = I + S;
  return sizeof(double) * 32 * (size_t)(I * (I + 1) / 2 + I * S + I + 2) + sizeof(int32_t) * 32 * (size_t)(2 + NW) +
         sizeof(uint16_t) * (size_t)(M * (M + 1) / 2 + M + S * (S + 1) / 2 + S + 4);
}
template <int I, int NW, int MINB = (NW <= 4 ? 2 : 1)>
static int launch_smem_mw(pgbp_batch* b, const MsgArgs& a, int nmsg, int S) {
#ifdef PGBP_HOST_EMUL
  (void)S;
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_rt<PGBP_MAX_DIM>(a, m, e);
#else
  static AttrOnce attr_done;  // per instantiation and device
  if (attr_done.first()) {
    PGBP_CUDA(cudaFuncSetAttribute((const void*)k_message_smem_mw<I, NW, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, PGBP_SMEM_MW_LIMIT));
  }
  if (a.ld * 8 >= ((int64_t)1 << 32)) PGBP_FAIL(PGBP_ESTATE, "batch too large for 32-bit row pitch");
  dim3 grid((unsigned)((a.B - a.e0 + 31) / 32), (unsigned)nmsg), block(32, NW);
  k_message_smem_mw<I, NW, MINB><<<grid, block, mw_bytes(I, S, NW), b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message_smem_mw");
}

// multi-warp kernel with the column-parallel Cholesky, tiles of TILE <= 32 elements (C5's (32,16) messages)
static size_t mwp_bytes(int I, int S, int NW, int TILE) {
  const int M = I + S;
  return sizeof(double) * TILE * (size_t)(I * (I + 1) / 2 + I * S + I + 2) + sizeof(int32_t) * TILE * (size_t)(2 + NW) +
         sizeof(uint16_t) * (size_t)(M * (M + 1) / 2 + M + S * (S + 1) / 2 + S + 4) + 16;
}
template <int I, int NW, int TILE>
static int launch_smem_mwp(pgbp_batch* b, const MsgArgs& a, int nmsg, int S) {
#ifdef PGBP_HOST_EMUL
  (void)S;
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_rt<PGBP_MAX_DIM>(a, m, e);
#else
  static AttrOnce attr_done;
  if (attr_done.first()) {
    PGBP_CUDA(cudaFuncSetAttribute((const void*)k_message_smem_mwp<I, NW, TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, PGBP_SMEM_MW_LIMIT));
  }
  if (a.ld * 8 >= ((int64_t)1 << 32)) PGBP_FAIL(PGBP_ESTATE, "batch too large for 32-bit row pitch");
  dim3 grid((unsigned)((a.B - a.e0 + TILE - 1) / TILE), (unsigned)nmsg), block(32, NW);
  k_message_smem_mwp<I, NW, TILE><<<grid, block, mwp_bytes(I, S, NW, TILE), b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message_smem_mwp");
}

// narrow tiles (TILE = 24 or 16 elements per single-warp block) for I <= 32 when the 32-lane factor does not fit
template <int TILE>
static int launch_smem_tile(pgbp_batch* b, const MsgArgs& a, int nmsg, int I, int S) {
#ifdef PGBP_HOST_EMUL
  (void)I; (void)S;
  for (int m = 0; m < nmsg; m++)
    for (int64_t e = a.e0; e < a.B; e++) message_thread_rt<PGBP_MAX_DIM>(a, m, e);
#else
  static AttrOnce attr_done;
  if (attr_done.first()) {
    PGBP_CUDA(cudaFuncSetAttribute((const void*)k_message_smem_rt<32, TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, PGBP_SMEM_MW_LIMIT));
  }
  const size_t bytes = sizeof(double) * TILE * (size_t)(I * (I + 1) / 2 + I * S + I);
  dim3 grid((unsigned)((a.B - a.e0 + TILE - 1) / TILE), (unsigned)nmsg);
  k_message_smem_rt<32, TILE><<<grid, 32, bytes, b->stream>>>(a);
#endif
  b->launches++;
  return check_launch("k_message_smem_rt");
}

int launch_medium(pgbp_batch* b, const MsgArgs& a, int n, int I, int S) {
  const int M = I + S;
  int rc = 0;
  const int mode = b->coop_mode;
  const bool fits = I <= 32 && sizeof(double) * 32 * (size_t)(I * (I + 1) / 2 + I * S + I) + 4 * (size_t)(M * (M + 3) / 2 + S * (S + 3) / 2 + 2) <= PGBP_SMEM_LIMIT;
  // large I (C5: p = 16): one or two single-warp tiles per SM are latency-bound; share the tile among warps
  const bool fits_mw = I >= 12 && I <= 16 && mw_bytes(I, S, 8) <= PGBP_SMEM_MW_LIMIT;
  // (measured on C4: the multi-warp form for I = 8 -- 4 warps x 4 tiles or 2 warps x 8 tiles per SM at 128
  // registers -- is SLOWER than the single-warp kernel with its unrolled S <= 8 variant: 70.6 / 68.5 ms per
  // step against 60.3 ms; it stays reserved for I >= 12.)
  if ((mode == -1 || mode == 2) && fits_mw) {
    switch (I) {
    // two tiles per SM with 4 warps each when they fit (233,472 bytes per SM, 1 KB reserved per block), else
    // one tile with 8 warps
#define PGBP_MW_CASE(I_) case I_: rc = (mode == 2 || 2 * (mw_bytes(I, S, 4) + 1024) <= 233472) ? launch_smem_mw<I_, 4>(b, a, n, S) : launch_smem_mw<I_, 8>(b, a, n, S); break;
      PGBP_MW_CASE(12) PGBP_MW_CASE(13) PGBP_MW_CASE(14) PGBP_MW_CASE(15) PGBP_MW_CASE(16)
#undef PGBP_MW_CASE
    }
  } else if ((mode == -1 || mode == 1 || mode == 2) && fits) {
    switch (I) {
#define PGBP_SMEM_CASE(I_) case I_: rc = launch_smem<I_, true>(b, a, n, I, S); break;
      PGBP_SMEM_CASE(1) PGBP_SMEM_CASE(2) PGBP_SMEM_CASE(3) PGBP_SMEM_CASE(4) PGBP_SMEM_CASE(5) PGBP_SMEM_CASE(6)
      PGBP_SMEM_CASE(7) PGBP_SMEM_CASE(8) PGBP_SMEM_CASE(9) PGBP_SMEM_CASE(10) PGBP_SMEM_CASE(11)
      PGBP_SMEM_CASE(12) PGBP_SMEM_CASE(13) PGBP_SMEM_CASE(14) PGBP_SMEM_CASE(15) PGBP_SMEM_CASE(16)
#undef PGBP_SMEM_CASE
      default: rc = (I <= 24) ? launch_smem<24, false>(b, a, n, I, S) : launch_smem<32, false>(b, a, n, I, S);
    }
  } else if ((mode == -1 || mode == 1 || mode == 2) && I <= 32 &&
             sizeof(double) * 16 * (size_t)(I * (I + 1) / 2 + I * S + I) <= PGBP_SMEM_MW_LIMIT) {
    // the 32-element factor does not fit the SM (C5's (32,16) messages: 274 KB): I = 32 goes to the multi-warp
    // kernel on 24-element tiles (on par with the 16-lane cooperative kernel on C5: 345 vs 355 ms per step),
    // anything else to the cooperative / generic kernels as before
    if (mode == 1) {  // single-warp narrow tiles: measured 880 ms per C5 step (one warp per SM), kept for comparison
      if (sizeof(double) * 24 * (size_t)(I * (I + 1) / 2 + I * S + I) <= PGBP_SMEM_MW_LIMIT) rc = launch_smem_tile<24>(b, a, n, I, S);
      else rc = launch_smem_tile<16>(b, a, n, I, S);
    } else if (I == 32 && mwp_bytes(I, S, 8, 24) <= PGBP_SMEM_MW_LIMIT) {
      rc = launch_smem_mwp<32, 8, 24>(b, a, n, S);
    } else if (M <= PGBP_COOP_MAX) {
      rc = launch_coop<48, 16>(b, a, n);
    } else {
      rc = launch_message<64>(b, a, n);
    }
  } else if (mode != 0 && M <= PGBP_COOP_MAX) {
    if (M <= 16) rc = (mode == 4) ? launch_coop<16, 4>(b, a, n) : launch_coop<16, 8>(b, a, n);
    else if (M <= 24) rc = launch_coop<24, 8>(b, a, n);
    else if (M <= 32) rc = launch_coop<32, 8>(b, a, n);
    else rc = launch_coop<48, 16>(b, a, n);  // 16 lanes per element: 2 elements per warp (half sectors)
  } else if (M <= 32) {
    rc = launch_message<32>(b, a, n);
  } else {
    rc = launch_message<64>(b, a, n);
  }
  return rc;
}

}  // namespace pgbp
