"""ctypes binding of libtarok_b200.so (the C ABI declared in include/tarok_b200.h).

This is the stub a maintainer of the reference would add to call the CUDA path (INTEGRATION.md).
There is NO CPU fallback: if the shared library is missing or cannot run on this machine the
import / first call fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# TAROK_B200_LIB selects a variant build of the same library (occupancy A/B experiments, tarok_b200/build.py --variant)
LIB_PATH = os.environ.get("TAROK_B200_LIB") or os.path.join(_PKG, "libtarok_b200.so")

# name -> (restype, argtypes); must list every function declared in include/tarok_b200.h
_VP, _U64, _U32, _I = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
SIGNATURES = {
    "tarok_create": (_I, [_I, _U64, _U64, _U32, C.POINTER(_VP)]),
    "tarok_destroy": (_I, [_VP]),
    "tarok_last_error": (C.c_char_p, [_VP]),
    "tarok_set_option": (_I, [_VP, _I, C.c_int64]),
    "tarok_n_games": (_U64, [_VP]),
    "tarok_n_alloc": (_U64, [_VP]),
    "tarok_deal": (_I, [_VP, _U64, _VP]),
    "tarok_set_deals": (_I, [_VP, _VP, _U64, _VP]),
    "tarok_export_perm": (_I, [_VP, _VP, _VP]),
    "tarok_auction": (_I, [_VP, _VP, _VP]),
    "tarok_auction_synth": (_I, [_VP, _U32, _VP]),
    "tarok_force_contract": (_I, [_VP, _VP, _VP, _VP, _VP]),
    "tarok_force_contract_synth": (_I, [_VP, _U32, _VP]),
    "tarok_exchange": (_I, [_VP, _VP, _VP, _VP]),
    "tarok_exchange_synth": (_I, [_VP, _U32, _VP]),
    "tarok_auction_bots": (_I, [_VP, _VP, _VP, _VP]),
    "tarok_exchange_bots": (_I, [_VP, _VP, _VP, _VP, _VP]),
    "tarok_step_bots": (_I, [_VP, _VP, _VP, _VP]),
    "tarok_legal_mask": (_I, [_VP, _VP, _VP]),
    "tarok_hands_by_seat": (_I, [_VP, _VP, _VP]),
    "tarok_step": (_I, [_VP, _VP, _VP]),
    "tarok_step_random": (_I, [_VP, _VP]),
    "tarok_steps_random": (_I, [_VP, _U32, _VP]),
    "tarok_score": (_I, [_VP, _VP, _VP]),
    "tarok_reset_stats": (_I, [_VP, _VP]),
    "tarok_reseed": (_I, [_VP, _U64]),
    "tarok_read_stats": (_I, [_VP, _VP, _VP]),
    "tarok_allreduce_stats": (_I, [_VP, _VP, _VP, _VP]),
    "tarok_setup_synth": (_I, [_VP, _U32, _U64, _VP]),
    "tarok_rollout_stepwise": (_I, [_VP, _U32, _U64, _VP]),
    "tarok_rollout_fused": (_I, [_VP, _U32, _U64, _VP]),
    "tarok_rollout_host": (_I, [_VP, _VP, _VP, _VP, _VP, _U64, _I, _VP, _VP, _VP]),
    "tarok_pack_records": (C.c_int64, [_VP, _VP, _VP, _VP, _U64, _VP]),
    "tarok_rollout_records": (_I, [_VP, _VP, _U64, _VP, _VP, _VP]),
    "tarok_pack_records_mt": (C.c_int64, [_VP, _VP, _VP, _VP, _U64, _VP, _I]),
    "tarok_pack_uses_avx512": (_I, []),
    "tarok_pack_force_scalar": (_I, [_I]),
    "tarok_rollout_host_packed": (_I, [_VP, _VP, _VP, _VP, _VP, _U64, _I, _VP, _VP, _VP]),
    "tarok_obs_shape": (_I, [_VP, _VP, _VP, _VP]),
    "tarok_obs_buckets": (_I, [_VP, _I, _VP, _VP, _VP, _VP]),
    "tarok_obs_buckets_host": (_I, [_VP, _I, _VP, _VP, _VP, _VP, _VP]),
    "tarok_obs_expand_buckets": (_I, [_VP, _VP, _VP, _VP, _U64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "tarok_select_action_buckets": (_I, [_VP, _VP, _VP, _VP, _VP, _U64, _VP, _VP, _VP, _VP]),
    "tarok_select_action_buckets_tab": (_I, [_VP, _VP, _VP, _VP, _VP, _U64, _VP, _VP, _VP, _VP]),
    "tarok_obs_expand": (_I, [_VP, _I, _U32, _VP, _U64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "tarok_obs_expand_at": (_I, [_VP, _I, _I, _U32, _VP, _U64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "tarok_targets": (_I, [_VP, _VP, _U64, C.c_float, _VP, _VP, _VP, _VP]),
    "tarok_select_action": (_I, [_VP, _VP, _VP, _U64, C.c_float, _VP, _VP, _VP]),
    "tarok_obs_hands": (_I, [_VP, _VP, _VP]),
    "tarok_obs_exchange": (_I, [_VP, _VP, _U64, _VP, _VP, _VP, _VP, _VP]),
    "tarok_select_exchange": (_I, [_VP, _VP, _VP, _U64, C.c_float, _VP, _VP, _VP]),
    "tarok_obs_expand_at_ex": (_I, [_VP, _I, _I, _I, _U32, _VP, _U64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "tarok_obs_expand_buckets_ex": (_I, [_VP, _I, _VP, _VP, _VP, _U64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "tarok_obs_hands_ex": (_I, [_VP, _I, _VP, _VP]),
    "tarok_obs_exchange_ex": (_I, [_VP, _I, _VP, _U64, _VP, _VP, _VP, _VP, _VP]),
    "tarok_select_action_ex": (_I, [_VP, _I, _VP, _VP, _U64, C.c_float, _VP, _VP, _VP]),
    "tarok_select_action_buckets_tab_ex": (_I, [_VP, _I, _VP, _VP, _VP, _VP, _U64, _VP, _VP, _VP, _VP]),
    "tarok_select_exchange_ex": (_I, [_VP, _I, _VP, _VP, _U64, C.c_float, _VP, _VP, _VP]),
    "tarok_export": (_I, [_VP, _I, C.POINTER(_VP)]),
    "tarok_field_ptr": (_VP, [_VP, _I]),
    "tarok_launch_count": (_U64, [_VP]),
}

_lib = None


class TarokLibraryError(RuntimeError):
    pass


def load():
    """dlopen the CUDA library and type every entry point.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:                                   # build the product in-tree (nvcc, sm_100a); this is not a fallback
            from .build import build_library
            build_library()
        except Exception as ex:
            raise TarokLibraryError(
                "%s is missing and could not be built (%s): run `python -m tarok_b200.build` (nvcc, sm_100a). "
                "tarok_b200 has no CPU fallback." % (LIB_PATH, str(ex)[:200]))
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(handle, rc):
    if rc != 0:
        msg = load().tarok_last_error(handle)
        raise TarokLibraryError("tarok_b200 error %d: %s" % (rc, (msg or b"").decode()))
