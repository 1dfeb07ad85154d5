"""ctypes binding of ``libcoevonet_b200.so`` (``include/coevonet_b200.h``).

The library is the product: there is NO CPU fallback.  Importing this module
without the built ``.so`` raises, and every compute call raises on a non-zero
return code with the library's error text.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32,
                    c_int64, c_uint8, c_uint32, c_uint64, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
#: COEVONET_LIB selects another build of the same library (development experiments only)
LIB_PATH = os.environ.get("COEVONET_LIB") or os.path.join(_HERE, "csrc", "libcoevonet_b200.so")

CEV_OK = 0
STATUS_NONFINITE = 1
SEAT = {"adversary_0": 0, "agent_0": 1, "agent_1": 2}
KIND_ES, KIND_GA, KIND_ENV, KIND_FRAMES, KIND_INIT, KIND_XOVER, KIND_ES_MIRROR, KIND_HOF = 0, 1, 2, 3, 4, 5, 6, 7
KIND_ES_SUBSPACE = 8
SUBSPACE_MAX_DIM = 32
ES_SGD, ES_ADAM = 0, 1
INIT_STATE_DIM = 11
ROLLOUT_OUT_DIM = 4
ORDER_STABLE_DESC, ORDER_REFERENCE = 0, 1
#: slots of the device generation state (CEV_GS_* in include/coevonet_b200.h)
GS_GEN, GS_SIGMA, GS_BEST, GS_STALE, GS_STOP, GS_STOP_GEN, GS_LAST_EVAL, GS_HIST = 0, 1, 4, 7, 10, 11, 12, 16


class RolloutCfg(Structure):
    _fields_ = [("n_cycles", c_int32), ("integrate_pos_first", c_int32),
                ("variant", c_int32), ("reserved", c_int32)]


class RolloutRole(Structure):
    """cev_rollout_role (include/coevonet_b200.h): one role of cev_mpe_rollout_roles_f32."""
    _fields_ = [("member_seat", c_int32), ("reserved", c_int32),
                ("members", c_void_p), ("member_pitch", c_int64),
                ("opp_a", c_void_p), ("opp_a_pitch", c_int64),
                ("opp_b", c_void_p), ("opp_b_pitch", c_int64),
                ("init", c_void_p), ("out", c_void_p)]


class CevError(RuntimeError):
    pass


_SIGNATURES = {
    "cev_version": (c_int, []),
    "cev_last_error": (c_char_p, []),
    "cev_create": (c_int, [c_int, POINTER(c_void_p)]),
    "cev_destroy": (c_int, [c_void_p]),
    "cev_device_info": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int)]),
    "cev_fc_dim": (c_int, [c_int]),
    "cev_fc_pitch": (c_int, [c_int]),
    "cev_dqn_dim": (c_int, [c_int, c_int]),
    "cev_dqn_pitch": (c_int, [c_int, c_int]),
    "cev_mpe_rollout_f32": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64,
                                    c_void_p, c_int64, c_void_p, c_int64, c_int,
                                    c_void_p, c_int, c_int, POINTER(RolloutCfg),
                                    c_void_p, c_void_p, c_void_p]),
    "cev_mpe_rollout_roles_f32": (c_int, [c_void_p, c_int, POINTER(RolloutRole), c_int, c_int, c_int, c_int,
                                          POINTER(RolloutCfg), c_void_p, c_void_p]),
    "cev_mpe_rollout_trace_f32": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64,
                                          c_void_p, c_int64, c_void_p, c_int64, c_int,
                                          c_void_p, c_int, c_int, POINTER(RolloutCfg),
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "cev_mpe_rollout_plan": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int)]),
    "cev_kernel_timing_enable": (c_int, [c_void_p, c_int]),
    "cev_kernel_timing_read": (c_int, [c_void_p, c_int, POINTER(c_double), POINTER(c_int)]),
    "cev_mpe_rollout_indexed_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                            c_void_p, c_int64, c_void_p, c_void_p, c_int,
                                            POINTER(RolloutCfg), c_void_p, c_void_p, c_void_p]),
    "cev_fc_forward_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64,
                                   c_void_p, c_void_p, c_void_p, c_void_p]),
    "cev_ga_repopulate_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_float, c_void_p, c_float,
                                      c_uint64, c_int, c_uint32, c_int64, c_int64,
                                      c_void_p, c_void_p, c_void_p]),
    "cev_gather_rows_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int64, c_int64, c_void_p,
                                    c_void_p]),
    "cev_select_topk_f64": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "cev_es_perturb_f32": (c_int, [c_void_p, c_void_p, c_int, c_float, c_void_p, c_uint64, c_int, c_uint32,
                                   c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "cev_es_perturb_prefix_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_float, c_void_p, c_uint64, c_int,
                                          c_uint32, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_es_update_f32": (c_int, [c_void_p, c_void_p, c_int, c_float, c_void_p, c_float, c_int64,
                                  c_uint64, c_int, c_uint32, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_es_update_members_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_float, c_void_p,
                                          c_float, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_weight_stats_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "cev_generation_state_doubles": (c_int, [c_int]),
    "cev_generation_end_f64": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_double,
                                       c_double, c_int, c_double, c_int, c_void_p]),
    "cev_axpy_f32": (c_int, [c_void_p, c_float, c_void_p, c_void_p, c_int64, c_void_p]),
    "cev_es_perturb_mirrored_f32": (c_int, [c_void_p, c_void_p, c_int, c_float, c_void_p, c_uint64, c_int, c_uint32,
                                            c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "cev_es_update_mirrored_f32": (c_int, [c_void_p, c_void_p, c_int, c_float, c_void_p, c_float, c_int64,
                                           c_uint64, c_int, c_uint32, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_centered_ranks_f64": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_es_apply_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, POINTER(c_int), c_int,
                                 c_double, c_float, c_int, c_void_p]),
    "cev_es_perturb_diag_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_uint64, c_int, c_uint32,
                                        c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "cev_es_update_diag_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_uint64, c_int, c_uint32, c_int64,
                                       c_int64, c_void_p, c_void_p, c_void_p]),
    "cev_es_apply_diag_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, POINTER(c_int),
                                      c_float, POINTER(c_double), c_float, c_float, c_void_p]),
    "cev_es_hof_opponents_i64": (c_int, [c_void_p, c_uint64, c_uint32, c_int, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_es_perturb_subspace_f32": (c_int, [c_void_p, c_void_p, c_int, c_float, c_void_p, c_void_p, c_int64, c_int,
                                            c_void_p, c_double, c_int, c_uint64, c_int, c_uint32, c_int64, c_int64,
                                            c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "cev_es_subspace_basis_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_int), c_void_p,
                                          c_void_p, c_void_p]),
    "cev_diversity_dist_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int,
                                       c_void_p, c_void_p]),
    "cev_deepqn_forward": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_int, c_int,
                                   c_int, c_void_p, c_void_p, c_void_p]),
    "cev_atari_synth_step_u8": (c_int, [c_void_p, c_uint64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p]),
    "cev_atari_observe_u8": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "cev_fc_init_f32": (c_int, [c_void_p, c_int, c_uint64, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_init_states_f64": (c_int, [c_void_p, c_uint64, c_uint32, c_int64, c_int64, c_void_p, c_void_p]),
    "cev_random_frames_u8": (c_int, [c_void_p, c_uint64, c_int64, c_void_p, c_void_p]),
    "cev_philox_words": (c_int, [c_void_p, c_uint64, c_int, c_int, c_uint32, c_int64, c_int64,
                                 c_int64, c_void_p, c_void_p]),
    "cev_fp32_peak": (c_int, [c_void_p, c_int, POINTER(c_double), c_void_p]),
}

#: every symbol ``include/coevonet_b200.h`` declares
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load the shared library (once) and bind the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise CevError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C coevonet_b200/csrc`).  coevonet_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != CEV_OK:
        msg = load().cev_last_error()
        raise CevError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


_handles = {}


def handle(device_index, stream=0):
    """Library handle of (device, stream), created on first use.  A handle owns the scratch
    workspaces of the rollout kernels, so work issued concurrently on several CUDA streams needs
    one handle per stream (``stream`` = the raw ``cudaStream_t`` value; 0 = the default handle)."""
    key = (int(device_index), int(stream or 0))
    h = _handles.get(key)
    if h is None:
        lib = load()
        hp = c_void_p()
        check(lib.cev_create(int(device_index), ctypes.byref(hp)), "cev_create")
        h = _handles[key] = hp
    return h


def device_info(device_index):
    n_sm, n_cl = c_int(), c_int()
    check(load().cev_device_info(handle(device_index), ctypes.byref(n_sm), ctypes.byref(n_cl)),
          "cev_device_info")
    return n_sm.value, n_cl.value
