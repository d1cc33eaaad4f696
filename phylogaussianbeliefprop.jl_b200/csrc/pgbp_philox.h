// Counter-based normal draws shared by the CUDA and host-emulation builds (curand is device-only).
// Philox4x32-10 (Salmon et al., SC'11; the round function and constants of Random123) and a Box-Muller pair:
//   key (seed lo, seed hi), counter (c0, c1, c2, c3) -> x0..x3;
//   u1 = ((x0 >> 5) 2^26 + (x1 >> 6) + 1) 2^-53 in (0, 1],  u2 = ((x2 >> 5) 2^26 + (x3 >> 6)) 2^-53 in [0, 1),
//   rho = sqrt(-2 log u1),  z0 = rho cos(2 pi u2),  z1 = rho sin(2 pi u2).
// A draw depends on its counter and key only, so any launch shape or chunking gives the same values.
#pragma once
#include "pgbp_backend.h"

namespace pgbp {

PGBP_HD void philox4x32_10(const uint32_t ctr[4], uint32_t k0, uint32_t k1, uint32_t out[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// The two standard normals of counter (c0, c1, c2, c3) under `seed` (read as unsigned 64-bit).
PGBP_HD void normal_pair(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, double* z0, double* z1) {
  const uint32_t ctr[4] = {c0, c1, c2, c3};
  uint32_t x[4];
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32), x);
  const double u1 = (double)((((uint64_t)(x[0] >> 5)) << 26) + (x[1] >> 6) + 1) * 0x1p-53;
  const double u2 = (double)((((uint64_t)(x[2] >> 5)) << 26) + (x[3] >> 6)) * 0x1p-53;
  const double rho = sqrt(-2.0 * log(u1)), a = 6.283185307179586 * u2;
  *z0 = rho * cos(a);
  *z1 = rho * sin(a);
}

}  // namespace pgbp
