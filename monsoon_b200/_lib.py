"""ctypes loader for libsb_b200.so (C ABI: include/sb_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``monsoon_b200.build.build_library()``
(nvcc, sm_100a).  There is no CPU fallback: if the library is missing, or no CUDA device is present,
the first call that needs the GPU raises.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("SB_LIB") or os.path.join(HERE, "libsb_b200.so")  # SB_LIB: development builds (tools/build_variant.sh)

_vp = ctypes.c_void_p
_int = ctypes.c_int

# name -> (restype, argtypes); mirrors include/sb_b200.h one to one (tests/test_abi.py checks it)
SIGNATURES = {
    "sb_abi_version": (_int, []),
    "sb_state_bytes": (_int, []),
    "sb_card_count": (_int, []),
    "sb_card_info": (_int, [_int, _vp]),
    "sb_create": (_int, [_int, ctypes.POINTER(_vp)]),
    "sb_destroy": (_int, [_vp]),
    "sb_last_error": (ctypes.c_char_p, [_vp]),
    "sb_device": (_int, [_vp]),
    "sb_sm_count": (_int, [_vp]),
    "sb_launch_count": (ctypes.c_uint64, [_vp]),
    "sb_set_option": (_int, [_vp, ctypes.c_char_p, _int]),
    "sb_reset": (_int, [_vp, _int, _vp, _vp, _int, _int, _vp, _vp, _vp]),
    "sb_legal_mask": (_int, [_vp, _int, _vp, _vp, _vp]),
    "sb_step": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_observe": (_int, [_vp, _int, _vp, _vp, _vp, _vp]),
    "sb_features": (_int, [_vp, _int, _vp, _vp, _vp, _vp]),
    "sb_select_action": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp]),
    "sb_generate_decks": (_int, [_vp, _int, _vp, ctypes.c_uint32, _int, _int, ctypes.c_double, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_es_offspring": (_int, [_vp, ctypes.c_uint64, ctypes.c_uint32, _int, _int, _int, ctypes.c_double, ctypes.c_double, ctypes.c_double, _vp, _vp, _vp, _vp]),
    "sb_es_select": (_int, [_vp, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_es_reset_sigmas": (_int, [_vp, ctypes.c_uint64, ctypes.c_uint32, _int, _int, ctypes.c_double, _vp, _vp]),
    "sb_es_inject_diversity": (_int, [_vp, ctypes.c_uint64, ctypes.c_uint32, _int, _int, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                      ctypes.c_double, _vp, _vp, _vp, _vp]),
    "sb_expert_action": (_int, [_vp, _int, _vp, _vp, _vp]),
    "sb_rollout_random": (_int, [_vp, _int, _vp, _int, _vp, _vp, _vp]),
    "sb_rollout_heuristic": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp]),
    "sb_env_reset": (_int, [_vp, _int, _vp, _vp, _int, _int, _vp, _int, _vp, _vp, _vp, _int, _vp, _vp, _vp, _vp, _vp]),
    "sb_env_step": (_int, [_vp, _int, _vp, _vp, _vp, _int, _int, _vp, _int, _vp, _vp, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_search_workspace_bytes": (ctypes.c_size_t, [_int, _int]),
    "sb_search_begin": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_search_simulate": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp, _vp, _vp, _vp,
                                  _vp, _vp, _vp]),
    "sb_search_end": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_determinize": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp]),
    "sb_ismcts_workspace_bytes": (ctypes.c_size_t, [_int, _int]),
    "sb_ismcts_begin": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_ismcts_simulate": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp]),
    "sb_ismcts_end": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_search_simulate_gumbel": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, _vp, _int, _int, _int, ctypes.c_double,
                                         ctypes.c_double, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_search_end_gumbel": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp, _vp,
                                    _vp, _vp, _vp, _vp]),
    "sb_ismcts_simulate_gumbel": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, _vp, _vp, _int, _int, _int, ctypes.c_double,
                                         ctypes.c_double, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_ismcts_end_gumbel": (_int, [_vp, _int, _int, _vp, ctypes.c_size_t, _vp, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp, _vp,
                                    _vp, _vp, _vp, _vp]),
    "sb_accumulate_fitness": (_int, [_vp, _int, _vp, _vp, _vp, _vp]),
    "sb_count_aborted": (_int, [_vp, _int, _vp, _vp, _vp, _vp]),
    "sb_eval_schedule": (_int, [_vp, _int, _int, _int, _int, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int64, _int, _vp, _vp, _vp, _vp]),
    "sb_eval_population": (_int, [_vp, _int, _int, _int, _int, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int64, ctypes.c_int64, _vp, _vp, _int, _vp,
                                  _int, _int, _vp, _vp, _vp]),
    "sb_step_host": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb_rollout_random_host": (_int, [_vp, _int, _vp, _vp, _int, _vp, _int, _vp, _vp, _vp]),
}

_lib = None


class SbError(RuntimeError):
    pass


def load():
    """Load the shared library (does not need a GPU) and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise SbError("libsb_b200.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no CPU fallback)")
    lib = ctypes.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = the .so does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
