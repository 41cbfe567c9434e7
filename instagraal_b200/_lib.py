"""ctypes binding of libinstagraal_b200.so (C ABI declared in include/instagraal_b200.h).

No PyTorch, no pycuda, no CPU fallback: if the shared library (or a CUDA device) is missing the
import / ig_create fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IG_B200_LIB", os.path.join(_HERE, "libinstagraal_b200.so"))

IG_MAX_CANDS = 8         # candidates of one scoring pass
IG_MAX_NEIGHBOURS = 64   # candidates of one step (ig_step_wide, ig_run_cycle_wide, ig_run_cycle_device)
IG_N_OPS = 24
IG_N_FIELDS = 13
FIELDS13 = ("pos", "sub_pos", "id_c", "start_bp", "len_bp", "sub_len", "circ", "prev", "next",
            "l_cont", "sub_l_cont", "l_cont_bp", "ori")

EXPORTS = (
    "ig_create", "ig_destroy", "ig_last_error", "ig_device_count", "ig_set_params", "ig_get_state",
    "ig_set_state", "ig_get_valid_insert", "ig_set_valid_insert", "ig_bomb", "ig_step", "ig_eval_scores",
    "ig_apply", "ig_full_likelihood", "ig_distance_histogram", "ig_set_sym_diag", "ig_device_state_ptr",
    "ig_set_profiling", "ig_get_stats", "ig_set_options", "ig_set_gpu_share", "ig_get_full_refresh_count", "ig_get_kernel_times", "ig_run_cycle", "ig_contact_thumbnail", "ig_set_neighbour_weights",
           "ig_run_cycle_device", "ig_get_cycle_plan", "ig_timeline_reset", "ig_timeline_get", "ig_timeline_blocks", "ig_timeline_phases",
    "ig_selftest_math", "ig_get_nuisance_stats", "ig_clone", "ig_run_cycles_device_multi", "ig_run_cycle_device_async", "ig_cycle_wait",
    "ig_bin_contacts", "ig_nccl_unique_id", "ig_nccl_init", "ig_allgather_best", "ig_get_gathered_state", "ig_nccl_finalize",
    "ig_set_device_nuisance", "ig_get_nuisance_records", "ig_step_wide", "ig_run_cycle_wide", "ig_get_cycle_plan_wide",
    "ig_adopt_gathered", "ig_set_temperature", "ig_get_tempered_records", "ig_get_gathered_live_likelihood",
)


class ig_config(C.Structure):
    _fields_ = [("device", C.c_int32), ("n_frags", C.c_int32), ("n_sub_frags", C.c_int32), ("nnz", C.c_int64),
                ("max_bounds_insert", C.c_int32), ("mean_sub_len_kb", C.c_float), ("n_pix", C.c_double),
                ("compat_last_block", C.c_int32), ("rigid_pruning", C.c_int32)]


class ig_level_data(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("frags13", "sub_parent", "sub_watson", "sub_crick", "sub_j", "row_ptr",
                                         "col", "val", "init_prev", "init_next", "orientable")]


class ig_step_result(C.Structure):
    _fields_ = [("scores", C.c_double * (IG_MAX_CANDS * IG_N_OPS)), ("likelihood", C.c_double),
                ("lnz_full", C.c_double), ("dist", C.c_double), ("sum_l_cont", C.c_int64), ("n_contigs", C.c_int32),
                ("op_sampled", C.c_int32), ("id_f_sampled", C.c_int32), ("cand_index", C.c_int32),
                ("n_uniq", C.c_int32 * IG_MAX_CANDS), ("n_sub", C.c_int32 * IG_MAX_CANDS), ("q4_hits", C.c_int32),
                ("reserved", C.c_int32)]


class ig_cycle_step(C.Structure):
    _fields_ = [("likelihood", C.c_double), ("lnz_full", C.c_double), ("dist", C.c_double), ("sum_l_cont", C.c_int64),
                ("n_contigs", C.c_int32), ("op_sampled", C.c_int32), ("id_f_sampled", C.c_int32), ("cand_index", C.c_int32),
                ("n_proposals", C.c_int32), ("q4_hits", C.c_int32)]


CYCLE_DTYPE = [("likelihood", "<f8"), ("lnz_full", "<f8"), ("dist", "<f8"), ("sum_l_cont", "<i8"), ("n_contigs", "<i4"),
               ("op_sampled", "<i4"), ("id_f_sampled", "<i4"), ("cand_index", "<i4"), ("n_proposals", "<i4"), ("q4_hits", "<i4")]

# ig_nuisance_step (80 B): one device nuisance step of a production-mode cycle
NUIS_DTYPE = [("likelihood_nuis", "<f8"), ("likelihood_t_after", "<f8"), ("u", "<f8"), ("draw", "<f8"), ("p_test", "<f4", (8,)),
              ("id_modif", "<i4"), ("accepted", "<i4"), ("valid", "<i4"), ("pad", "<i4")]

# ig_tempered_step (48 B): the move draw of one production-mode step at a chain temperature T > 0
TEMPERED_DTYPE = [("s_max", "<f8"), ("log_w", "<f8"), ("u", "<f8"), ("u_batch", "<f8"), ("n_scored", "<i4"), ("batch", "<i4"),
                  ("index", "<i4"), ("pad", "<i4")]

_lib = None


def lib():
    """Load the CUDA library; raises OSError when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OSError("instagraal_b200: %s not built -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
        L.ig_create.argtypes = [C.POINTER(ig_config), C.POINTER(ig_level_data), C.POINTER(vp)]
        L.ig_destroy.argtypes = [vp]
        L.ig_destroy.restype = None
        L.ig_last_error.argtypes = [vp]
        L.ig_last_error.restype = C.c_char_p
        L.ig_device_count.argtypes = []
        L.ig_set_params.argtypes = [vp, vp]
        L.ig_get_state.argtypes = [vp, vp]
        L.ig_set_state.argtypes = [vp, vp]
        L.ig_get_valid_insert.argtypes = [vp, vp]
        L.ig_set_valid_insert.argtypes = [vp, vp]
        L.ig_bomb.argtypes = [vp, vp]
        L.ig_step.argtypes = [vp, i32, vp, i32, C.POINTER(ig_step_result)]
        L.ig_eval_scores.argtypes = [vp, i32, i32, i32, vp, C.POINTER(i32), C.POINTER(i32)]
        L.ig_apply.argtypes = [vp, i32, i32, i32, C.POINTER(ig_step_result)]
        L.ig_full_likelihood.argtypes = [vp, vp, i32, vp]
        L.ig_distance_histogram.argtypes = [vp, dbl, dbl, i32, i32, vp, C.POINTER(i64)]
        L.ig_set_sym_diag.argtypes = [vp, vp]
        L.ig_device_state_ptr.argtypes = [vp, C.POINTER(vp), C.POINTER(i64)]
        L.ig_set_profiling.argtypes = [vp, i32]
        L.ig_get_stats.argtypes = [vp, vp, i32]
        L.ig_set_options.argtypes = [vp, i32, i32]
        L.ig_set_gpu_share.argtypes = [vp, i32]
        L.ig_bin_contacts.argtypes = [i32, i64, vp, vp, vp, vp, i32, i32, vp, vp, vp, C.POINTER(i64)]
        L.ig_get_kernel_times.argtypes = [vp, vp, i32]
        L.ig_run_cycle.argtypes = [vp, i32, vp, vp, vp, vp]
        L.ig_contact_thumbnail.argtypes = [vp, vp, i32, vp]
        L.ig_set_neighbour_weights.argtypes = [vp, vp, vp, vp, vp]
        L.ig_run_cycle_device.argtypes = [vp, i32, vp, i32, C.c_uint64, C.c_uint32, vp]
        L.ig_get_cycle_plan.argtypes = [vp, i32, vp]
        L.ig_timeline_reset.argtypes = [vp]
        L.ig_timeline_get.argtypes = [vp, i32, vp]
        L.ig_timeline_blocks.argtypes = [vp, i32, vp]
        L.ig_timeline_phases.argtypes = [vp, vp, i32]
        L.ig_get_full_refresh_count.argtypes = [vp, C.POINTER(i64)]
        L.ig_get_nuisance_stats.argtypes = [vp, vp, i32]
        L.ig_clone.argtypes = [vp, C.POINTER(vp)]
        L.ig_run_cycles_device_multi.argtypes = [vp, i32, i32, vp, i32, vp, C.c_uint32, vp]
        L.ig_run_cycle_device_async.argtypes = [vp, i32, vp, i32, C.c_uint64, C.c_uint32]
        L.ig_cycle_wait.argtypes = [vp, i32, vp]
        L.ig_nccl_unique_id.argtypes = [vp]
        L.ig_nccl_init.argtypes = [vp, i32, i32, i32, vp]
        L.ig_allgather_best.argtypes = [vp, vp, i32, vp, vp, C.POINTER(i32), C.POINTER(C.c_float)]
        L.ig_get_gathered_state.argtypes = [vp, i32, vp]
        L.ig_adopt_gathered.argtypes = [vp, vp, i32, i32, vp, vp, C.POINTER(dbl)]
        L.ig_nccl_finalize.argtypes = [vp]
        L.ig_selftest_math.argtypes = [vp, i32, C.c_float, C.c_float, C.c_float, vp]
        L.ig_set_device_nuisance.argtypes = [vp, i32]
        L.ig_get_nuisance_records.argtypes = [vp, i32, vp]
        L.ig_step_wide.argtypes = [vp, i32, vp, i32, C.POINTER(ig_step_result), vp, vp, vp]
        L.ig_run_cycle_wide.argtypes = [vp, i32, vp, vp, i32, vp, vp]
        L.ig_get_cycle_plan_wide.argtypes = [vp, i32, i32, vp]
        L.ig_set_temperature.argtypes = [vp, dbl]
        L.ig_get_tempered_records.argtypes = [vp, i32, vp]
        L.ig_get_gathered_live_likelihood.argtypes = [vp, vp]
        for name in EXPORTS:
            if name not in ("ig_destroy", "ig_last_error"):
                getattr(L, name).restype = C.c_int
        _lib = L
    return _lib


def check(h, rc, what):
    if rc != 0:
        msg = lib().ig_last_error(h)
        raise RuntimeError("%s failed (rc=%d): %s" % (what, rc, msg.decode() if msg else "?"))
