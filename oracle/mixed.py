"""TEST INFRASTRUCTURE ONLY -- numpy/ctypes front-end of the mixed-table oracle (oracle/mixed.c): Bot_igralec seats beside
caller-driven (neural) seats, as tarok_auction_bots / tarok_exchange_bots / tarok_step_bots play them.  Same importers as
oracle.oracle; ``tarok_b200`` never imports it."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libtarok_oracle_mixed.so")
_SOURCES = [os.path.join(_HERE, f) for f in ("mixed.c", "tarok_oracle.c", "synth.c", "tarok_oracle.h")]
_lib = None


def build(force: bool = False) -> str:
    """Compile oracle/mixed.c (which includes the oracle sources) with the flags of oracle/Makefile."""
    stale = not os.path.exists(_LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in _SOURCES)
    if force or stale:
        cc = shutil.which("gcc") or "/usr/bin/gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-fopenmp", "-Wall", "-Wextra", "-std=c11", "-shared", "-o", _LIB_PATH,
                        os.path.join(_HERE, "mixed.c")], check=True)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def replay_bots(seed, first_gid, perm, intents, bots, group=None, discard=None, cards=None):
    """Mixed tables (``syn_replay_bots``): game i (global id first_gid + i) dealt ``perm[i]``, bit s of ``bots[i]`` = seat s is
    a Bot_igralec drawing its bids, king, exchange and cards from the Philox draws of mode 18; the other seats bid their
    index2igra ``intents`` (uint8 [n,4], 0..19), exchange ``group`` / ``discard`` and play ``cards`` (uint8 [n,48]).  Returns
    contract, declarer, king, group, discard, plays [n,48] (0xFF after the last), scores [n,4], err and mismatch (int8: the
    first play where a bot's card in ``cards`` differs from its draw, -1 none)."""
    n = len(perm)
    a = lambda x, t, shape: None if x is None else np.ascontiguousarray(x, t).reshape(shape)
    args = [a(perm, np.uint8, (n, 54)), a(intents, np.uint8, (n, 4)), a(bots, np.uint8, (n,)), a(group, np.uint8, (n,)),
            a(discard, np.uint64, (n,)), a(cards, np.uint8, (n, 48))]
    out = dict(contract=np.empty(n, np.uint8), declarer=np.empty(n, np.uint8), king=np.empty(n, np.uint8),
               group=np.empty(n, np.uint8), discard=np.empty(n, np.uint64), plays=np.empty((n, 48), np.uint8),
               scores=np.empty((n, 4), np.int16), err=np.empty(n, np.uint8), mismatch=np.empty(n, np.int8))
    lib().syn_replay_bots_batch(C.c_uint64(seed), C.c_uint64(first_gid), C.c_int64(n), *[_p(x) for x in args],
                                *[_p(out[k]) for k in ("contract", "declarer", "king", "group", "discard", "plays", "scores",
                                                       "err", "mismatch")])
    return out
