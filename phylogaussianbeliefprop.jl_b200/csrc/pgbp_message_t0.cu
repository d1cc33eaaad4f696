// One third of the register-class message kernels (see pgbp_msg_t0.cuh).  -DPGBP_T0_PART=0: i in 1..3,
// 1: i in 4..6, 2: i in 7..12.
#include "pgbp_msg_t0.cuh"

#ifndef PGBP_T0_PART
#error "compile with -DPGBP_T0_PART=0|1|2"
#endif
#define PGBP_FN(n) launch_t0_part##n
#if PGBP_T0_PART == 0
#define PGBP_PART_LO 1
#define PGBP_PART_HI 3
#define PGBP_PART_FN PGBP_FN(0)
#elif PGBP_T0_PART == 1
#define PGBP_PART_LO 4
#define PGBP_PART_HI 6
#define PGBP_PART_FN PGBP_FN(1)
#else
#define PGBP_PART_LO 7
#define PGBP_PART_HI 12
#define PGBP_PART_FN PGBP_FN(2)
#endif

namespace pgbp {

template <int I_, int S_>
static int try_shape(pgbp_batch* b, const MsgArgs& a, int nmsg, int ci, int cs) {
  if constexpr (I_ >= PGBP_PART_LO && I_ <= PGBP_PART_HI) {
    if (ci == I_ && cs == S_) return launch_message_staged<I_, S_>(b, a, nmsg);
  }
  return PGBP_NOT_MINE;
}

int PGBP_PART_FN(pgbp_batch* b, const MsgArgs& a, int nmsg, int ci, int cs) {
  if (ci < PGBP_PART_LO || ci > PGBP_PART_HI) return PGBP_NOT_MINE;
  int rc = PGBP_NOT_MINE;
#define X(I_, S_) if (rc == PGBP_NOT_MINE) rc = try_shape<I_, S_>(b, a, nmsg, ci, cs);
  PGBP_T0_SHAPES(X)
#undef X
  return rc;
}

}  // namespace pgbp
