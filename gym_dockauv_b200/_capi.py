"""ctypes binding of libdockauv_b200.so (include/dockauv.h).  There is no fallback: if the library is missing
or was built against another ABI this module raises, and so does every env constructor."""
import ctypes as C
import os

from .params import (ABI_VERSION, DockauvBuffers, DockauvDebugOut, DockauvParams, DockauvPolicy, DockauvPolicyOut,
                     DockauvReplayRing, DockauvReplaySample, DockauvRolloutOut, DockauvScenarioBank,
                     DockauvSquashedActor, DockauvStepOut, DockauvTapBuffers)

LIB_PATH = os.environ.get("DOCKAUV_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib",
                                                        "libdockauv_b200.so")   # DOCKAUV_LIB: tuning builds only

# every symbol include/dockauv.h declares: (restype, argtypes)
_vp, _i, _i64 = C.c_void_p, C.c_int, C.c_int64
SYMBOLS = {
    "dockauv_abi_version": (_i, []),
    "dockauv_last_error": (C.c_char_p, []),
    "dockauv_sizeof_params": (C.c_size_t, []),
    "dockauv_n_obs": (_i, [C.POINTER(DockauvParams)]),
    "dockauv_create": (_i, [C.POINTER(DockauvParams), _i64, _i, C.POINTER(_vp)]),
    "dockauv_destroy": (_i, [_vp]),
    "dockauv_bind": (_i, [_vp, C.POINTER(DockauvBuffers)]),
    "dockauv_set_seed": (_i, [_vp, C.c_uint64]),
    "dockauv_reset": (_i, [_vp, _vp, _vp]),
    "dockauv_refresh_obstacles": (_i, [_vp, _vp]),
    "dockauv_step": (_i, [_vp, _vp, _i, _vp, C.POINTER(DockauvStepOut), C.POINTER(DockauvDebugOut), _i, _vp]),
    "dockauv_enable_step_graph": (_i, [_vp, _i]),
    "dockauv_step_graph_captures": (_i, [_vp, C.POINTER(_i64)]),
    "dockauv_step_host": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, C.POINTER(DockauvStepOut)]),
    "dockauv_rollout": (_i, [_vp, _vp, _i, _i, C.POINTER(DockauvRolloutOut), _i, _i, _vp]),
    "dockauv_rollout_policy": (_i, [_vp, C.POINTER(DockauvPolicy), _vp, _i, C.POINTER(DockauvRolloutOut),
                                    C.POINTER(DockauvPolicyOut), _i, _i, _vp]),
    "dockauv_set_taps": (_i, [_vp, C.POINTER(_i64), _i, _i, C.POINTER(DockauvTapBuffers)]),
    "dockauv_set_scenario_bank": (_i, [_vp, C.POINTER(DockauvScenarioBank), _vp]),
    "dockauv_gae": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i64, C.c_float, C.c_float, _vp, _vp, _vp]),
    "dockauv_replay_sample": (_i, [C.POINTER(DockauvReplayRing), _i, _i, _i64, _i, _i, _i64, _i64, _i64, C.c_uint64,
                                   C.c_uint64, C.POINTER(DockauvReplaySample), _vp]),
    "dockauv_replay_collect": (_i, [_vp, C.POINTER(DockauvSquashedActor), C.POINTER(DockauvReplayRing), _i, _i, _i, _i,
                                    _i, _vp]),
    "dockauv_stats_ptr": (_i, [_vp, C.POINTER(_vp)]),
    "dockauv_fold_stats": (_i, [_vp, _vp]),
    "dockauv_get_stats": (_i, [_vp, C.POINTER(C.c_double), _vp]),
    "dockauv_clear_stats": (_i, [_vp, _vp]),
    "dockauv_measure_peaks": (_i, [_i, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "dockauv_launch_count": (_i, [_vp, C.POINTER(_i64)]),
    "dockauv_last_list_counts": (_i, [_vp, C.POINTER(_i64), C.POINTER(_i64), _vp]),
    "dockauv_rollout_captures": (_i, [_vp, C.POINTER(_i64)]),
    "dockauv_rollout_policy_captures": (_i, [_vp, C.POINTER(_i64)]),
    "dockauv_replay_collect_captures": (_i, [_vp, C.POINTER(_i64)]),
    "dockauv_enable_timing": (_i, [_vp, _i]),
    "dockauv_last_step_ms": (_i, [_vp, C.POINTER(C.c_float)]),
    "dockauv_last_step_launch_ms": (_i, [_vp, C.POINTER(C.c_float), _i, C.POINTER(_i)]),
}


class DockauvError(RuntimeError):
    pass


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DockauvError(
            f"{LIB_PATH} is missing: build it with `python -m gym_dockauv_b200.build` (nvcc, sm_100a). "
            "gym_dockauv_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)       # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.dockauv_abi_version() != ABI_VERSION:
        raise DockauvError(f"ABI mismatch: library {lib.dockauv_abi_version()}, python {ABI_VERSION}")
    if lib.dockauv_sizeof_params() != C.sizeof(DockauvParams):
        raise DockauvError(f"DockauvParams size mismatch: library {lib.dockauv_sizeof_params()}, "
                           f"python {C.sizeof(DockauvParams)}")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise DockauvError(f"dockauv error {rc}: {load().dockauv_last_error().decode()}")
