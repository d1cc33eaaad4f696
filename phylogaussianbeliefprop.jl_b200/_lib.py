"""ctypes binding of libpgbp_b200.so (include/pgbp_b200.h).

There is NO CPU fallback: if the CUDA library is missing or no CUDA device is
usable, every entry point raises.  (`Library(path)` lets the CPU test-suite
bind the host-emulation build explicitly; the package itself never does.)
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PGBP_B200_LIB selects another build of the SAME CUDA library (kernel-tuning variants); never a CPU path
DEFAULT_LIB = os.environ.get("PGBP_B200_LIB") or os.path.join(HERE, "lib", "libpgbp_b200.so")

i32, i64, u32, u8, f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_uint8, C.c_double
P = C.POINTER


class PgbpError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libpgbp_b200 error {code}: {msg}")
        self.code = code


class FamilyTable(C.Structure):
    _fields_ = [("nnodes", i32), ("ntips", i32), ("node_cluster", P(i32)), ("mem_off", P(i32)),
                ("mem_pos", P(i32)), ("mem_length", P(f64)), ("mem_gamma", P(f64)), ("mem_color", P(i32)),
                ("node_datarow", P(i32)), ("root_fixed", i32), ("mem_tpos", P(i32)), ("tip_missing", P(u8))]


class PlanDesc(C.Structure):
    _fields_ = [("nclusters", i32), ("nsepsets", i32), ("ntraits", i32), ("belief_dim", P(i32)),
                ("sepset_clusters", P(i32)), ("upind_off", P(i32)), ("upind", P(i32)), ("ntrees", i32),
                ("tree_off", P(i32)), ("tree_parent", P(i32)), ("tree_child", P(i32)),
                ("families", P(FamilyTable))]


# name -> (restype, argtypes); must list every symbol declared in include/pgbp_b200.h
vp = C.c_void_p
SIGNATURES = {
    "pgbp_abi_version": (i32, []),
    "pgbp_last_error": (i32, [C.c_char_p, C.c_size_t]),
    "pgbp_plan_create": (i32, [P(PlanDesc), P(vp)]),
    "pgbp_plan_destroy": (i32, [vp]),
    "pgbp_plan_get_levels": (i32, [vp, i32, i32, P(i32), P(i32), P(i32), P(i32), P(i32), P(i32), P(i32)]),
    "pgbp_plan_traversal_cost": (i32, [vp, i32, i32, i32, P(f64), P(f64)]),
    "pgbp_batch_create": (i32, [vp, i64, i32, u32, P(vp)]),
    "pgbp_batch_create_shared": (i32, [vp, i64, i64, i32, u32, P(vp)]),
    "pgbp_batch_destroy": (i32, [vp]),
    "pgbp_batch_set_stream": (i32, [vp, vp]),
    "pgbp_batch_synchronize": (i32, [vp]),
    "pgbp_batch_size": (i64, [vp]),
    "pgbp_batch_device_bytes": (i64, [vp]),
    "pgbp_batch_launch_count": (i64, [vp, i32]),
    "pgbp_batch_set_walk_mode": (i32, [vp, i32]),
    "pgbp_batch_set_coop_mode": (i32, [vp, i32]),
    "pgbp_batch_set_pipeline": (i32, [vp, i32]),
    "pgbp_batch_set_graph_mode": (i32, [vp, i32]),
    "pgbp_batch_set_tilewalk_mode": (i32, [vp, i32]),
    "pgbp_batch_set_tilewalk_params": (i32, [vp, i32, i32]),
    "pgbp_set_belief": (i32, [vp, i32, P(f64), P(f64), P(f64)]),
    "pgbp_get_belief": (i32, [vp, i32, P(f64), P(f64), P(f64)]),
    "pgbp_get_factor": (i32, [vp, i32, P(f64), P(f64), P(f64)]),
    "pgbp_get_residual": (i32, [vp, i32, i32, P(f64), P(f64), P(u8), P(f64)]),
    "pgbp_get_status": (i32, [vp, P(i32)]),
    "pgbp_clear_status": (i32, [vp]),
    "pgbp_reset_beliefs": (i32, [vp]),
    "pgbp_factors_from_beliefs": (i32, [vp]),
    "pgbp_reset_from_factors": (i32, [vp]),
    "pgbp_reset_calibration_flags": (i32, [vp, i32]),
    "pgbp_assign_factors": (i32, [vp, i32, P(f64), i64, P(f64), i64, i32]),
    "pgbp_assign_factors_ou": (i32, [vp, P(f64), i64, P(f64), i64, i32]),
    "pgbp_assign_factors_device": (i32, [vp, i32, vp, i64, vp, i64, i32]),
    "pgbp_calibrate": (i32, [vp, P(i32), i32, i32, u32, P(i32), P(i32), P(i32)]),
    "pgbp_calibrate_async": (i32, [vp, P(i32), i32, i32, u32]),
    "pgbp_propagate": (i32, [vp, i32, i32, i32, u32]),
    "pgbp_integrate": (i32, [vp, i32, P(f64), P(f64)]),
    "pgbp_integrate_device": (i32, [vp, i32, vp, vp]),
    "pgbp_integrate_cov": (i32, [vp, i32, P(f64), P(f64), P(f64)]),
    "pgbp_marginal_moments": (i32, [vp, i32, P(i32), P(i32), P(i32), P(f64), P(f64)]),
    "pgbp_marginal_moments_device": (i32, [vp, i32, P(i32), P(i32), P(i32), vp, vp]),
    "pgbp_factored_energy": (i32, [vp, P(f64)]),
    "pgbp_factored_energy_device": (i32, [vp, vp]),
    "pgbp_regularize_bycluster": (i32, [vp]),
    "pgbp_regularize_onschedule": (i32, [vp]),
    "pgbp_regularize_bynodesubtree": (i32, [vp, i32] + [P(i32)] * 8),
    "pgbp_device_view": (i32, [vp, P(vp), P(i64), P(i64)]),
    "pgbp_belief_slot": (i32, [vp, i32, P(i64), P(i64), P(i64)]),
    "pgbp_batch_belief_rows": (i32, [vp, i32, P(i64), P(i64)]),
    "pgbp_comm_create": (i32, [i32, i32, i32, i64, i32, P(vp)]),
    "pgbp_comm_handle": (i32, [vp, P(u8)]),
    "pgbp_comm_connect": (i32, [vp, P(u8)]),
    "pgbp_comm_disconnect": (i32, [vp]),
    "pgbp_comm_destroy": (i32, [vp]),
    "pgbp_comm_window": (i32, [vp, i32, P(vp), P(i64)]),
    "pgbp_integrate_gather": (i32, [vp, i32, vp, i32]),
    "pgbp_comm_put": (i32, [vp, vp, i32, vp]),
    "pgbp_comm_wait": (i32, [vp, vp, i32, i32]),
    "pgbp_comm_read": (i32, [vp, vp, i32, P(f64)]),
    "pgbp_comm_check": (i32, [vp, vp]),
}

# flags (mirror the header)
BATCH_FACTORS, BATCH_RESIDUALS = 1, 2
CAL_POSTORDER, CAL_PREORDER, CAL_BOTH, CAL_RESIDNORM, CAL_RESIDKLDIV, CAL_AUTO, CAL_REFORDER = 1, 2, 3, 4, 8, 16, 32
PAIR_ZIP, PAIR_PRODUCT = 0, 1


class Library:
    def __init__(self, path=None):
        path = path or DEFAULT_LIB
        if not os.path.exists(path):
            raise ImportError(
                f"{path} not found: build it with `python phylogaussianbeliefprop.jl_b200/build.py` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        self.path = path
        self.dll = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(self.dll, name)
            fn.restype, fn.argtypes = res, args
        if self.dll.pgbp_abi_version() != 2:
            raise ImportError("libpgbp_b200 ABI version mismatch")

    def check(self, rc):
        if rc != 0:
            buf = C.create_string_buffer(512)
            self.dll.pgbp_last_error(buf, 512)
            raise PgbpError(rc, buf.value.decode(errors="replace"))

    def __getattr__(self, name):
        return getattr(self.dll, name)


_default = None


def default_library() -> Library:
    global _default
    if _default is None:
        _default = Library()
    return _default
