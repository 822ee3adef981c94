"""TEST INFRASTRUCTURE ONLY -- numpy/ctypes front-end of the C oracle (oracle/tarok_oracle.c).

The C library restates the reference rule engine (citations in the C source); this file only
marshals numpy arrays.  Allowed importers: ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs.  ``tarok_b200`` never imports it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libtarok_oracle.so")
_lib = None

NO_KING = 7
NO_GROUP = 0xFF
MODE_NAVADNA_MIX = 16
MODE_AUCTION_UNIFORM = 17
MODE_AUCTION_BOT = 18
CONTRACT_NAMES = ["Klop", "Tri", "Dve", "Ena", "Solo_tri", "Solo_dve", "Solo_ena", "Berac",
                  "Solo_brez", "Odprti_berac"]


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (gcc + OpenMP)."""
    srcs = [os.path.join(_HERE, f) for f in ("tarok_oracle.c", "synth.c", "tarok_oracle.h")]
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-B", "libtarok_oracle.so"], check=True,
                       stdout=subprocess.DEVNULL)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = C.CDLL(_LIB_PATH)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def replay(perm, contract, declarer, king, group, discard_mask, cards, want_state=True):
    """Teacher-forced replay of n deals.  Returns dict of numpy arrays."""
    n = len(perm)
    perm = np.ascontiguousarray(perm, np.uint8).reshape(n, 54)
    contract = np.ascontiguousarray(contract, np.uint8)
    declarer = np.ascontiguousarray(declarer, np.uint8)
    king = np.ascontiguousarray(king, np.uint8)
    group = np.ascontiguousarray(group, np.uint8)
    discard_mask = np.ascontiguousarray(discard_mask, np.uint64)
    cards = np.ascontiguousarray(cards, np.uint8).reshape(n, 48)
    out = dict(
        seat=np.empty((n, 48), np.uint8), mask=np.empty((n, 48), np.uint64),
        winner=np.empty((n, 12), np.uint8), scores=np.empty((n, 4), np.int16),
        plays=np.empty(n, np.uint8), err=np.empty(n, np.uint8),
    )
    if want_state:
        out.update(hands=np.empty((n, 4), np.uint64), piles=np.empty((n, 4), np.uint64),
                   talon=np.empty(n, np.uint64))
    lib().orc_replay_batch(
        C.c_int64(n), _p(perm), _p(contract), _p(declarer), _p(king), _p(group), _p(discard_mask),
        _p(cards), _p(out["seat"]), _p(out["mask"]), _p(out["winner"]), _p(out["scores"]),
        _p(out["plays"]), _p(out["err"]), _p(out.get("hands")), _p(out.get("piles")),
        _p(out.get("talon")))
    return out


def lists(perm, contract, declarer, king, group, discard_mask, cards):
    """Teacher-forced replay like ``replay``, returning the reference's ordered lists: mozne uint8 [n,48,16] (0xFF
    padded) + mozne_n [n,48], seat [n,48] (both also at the first 0xFF of a game still being played), trick_value int16 [n,12], zalozit uint8 [n,16] + zalozit_n [n] (the
    ``mozno_zalozit()`` list after the pick-up; empty without an exchange) and groups uint8 [n,6,3] (0xFF padded)."""
    n = len(perm)
    args = [np.ascontiguousarray(perm, np.uint8).reshape(n, 54), np.ascontiguousarray(contract, np.uint8),
            np.ascontiguousarray(declarer, np.uint8), np.ascontiguousarray(king, np.uint8),
            np.ascontiguousarray(group, np.uint8), np.ascontiguousarray(discard_mask, np.uint64),
            np.ascontiguousarray(cards, np.uint8).reshape(n, 48)]
    out = dict(mozne=np.empty((n, 48, 16), np.uint8), mozne_n=np.empty((n, 48), np.uint8),
               seat=np.empty((n, 48), np.uint8), trick_value=np.empty((n, 12), np.int16),
               zalozit=np.empty((n, 16), np.uint8), zalozit_n=np.empty(n, np.uint8), groups=np.empty((n, 6, 3), np.uint8))
    lib().orc_lists_batch(C.c_int64(n), *[_p(a) for a in args],
                          *[_p(out[k]) for k in ("mozne", "mozne_n", "seat", "trick_value", "zalozit", "zalozit_n",
                                                 "groups")])
    return out


def auction_fixed(intents):
    """intents: int8[n,4] Tip codes (-1 Naprej .. 9).  -> (declarer, contract, calls)"""
    intents = np.ascontiguousarray(intents, np.int8).reshape(-1, 4)
    n = len(intents)
    d, c, k = np.empty(n, np.uint8), np.empty(n, np.uint8), np.empty(n, np.uint8)
    lib().orc_auction_fixed_batch(C.c_int64(n), _p(intents), _p(d), _p(c), _p(k))
    return d, c, k


def auction_scripted(draws):
    """draws: int8[n,16] Tip codes consumed one per licitiram call (Bot model)."""
    draws = np.ascontiguousarray(draws, np.int8).reshape(-1, 16)
    n = len(draws)
    d, c, k = np.empty(n, np.uint8), np.empty(n, np.uint8), np.empty(n, np.uint8)
    lib().orc_auction_scripted_batch(C.c_int64(n), _p(draws), _p(d), _p(c), _p(k))
    return d, c, k


def prestej(ids_list):
    n = len(ids_list)
    stride = max([len(x) for x in ids_list] + [1])
    ids = np.zeros((n, stride), np.uint8)
    ln = np.zeros(n, np.uint8)
    for i, x in enumerate(ids_list):
        ids[i, :len(x)] = x
        ln[i] = len(x)
    out = np.empty(n, np.int32)
    lib().orc_prestej_batch(C.c_int64(n), _p(ids), _p(ln), C.c_int(stride), _p(out))
    return out


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    lib().syn_philox_kat(c, C.c_uint32(key[0]), C.c_uint32(key[1]))
    return [int(x) for x in c]


def draw(seed, gid, stream, idx, n):
    f = lib().syn_draw
    f.restype = C.c_uint32
    return int(f(C.c_uint64(seed), C.c_uint64(gid), C.c_uint32(stream), C.c_uint32(idx), C.c_uint32(n)))


def deal(seed, first_gid, n):
    out = np.empty((n, 54), np.uint8)
    lib().syn_deal_batch(C.c_uint64(seed), C.c_uint64(first_gid), C.c_int64(n), _p(out))
    return out


def rollout(seed, first_gid, n, mode, full=True):
    """Whole deals with uniform-random players on the CPU (OpenMP).  Returns dict."""
    out = dict(scores=np.empty((n, 4), np.int16), plays=np.empty(n, np.uint8),
               contract=np.empty(n, np.uint8), declarer=np.empty(n, np.uint8),
               king=np.empty(n, np.uint8), err=np.empty(n, np.uint8), stats=np.zeros(10, np.int64))
    if full:
        out.update(perm=np.empty((n, 54), np.uint8), cards=np.empty((n, 48), np.uint8),
                   group=np.empty(n, np.uint8), discard=np.empty(n, np.uint64))
    lib().syn_rollout_batch(
        C.c_uint64(seed), C.c_uint64(first_gid), C.c_int64(n), C.c_int(mode),
        _p(out["scores"]), _p(out["plays"]), _p(out["contract"]), _p(out["declarer"]), _p(out["king"]),
        _p(out["err"]), _p(out.get("perm")), _p(out.get("cards")), _p(out.get("group")),
        _p(out.get("discard")), _p(out["stats"]))
    return out


def rollout_injected(seed, first_gid, perm, contract, declarer, king=None):
    """The given deals (uint8 [n,54]) under forced contracts (uint8 [n] each; king None = no king), game i with global id
    first_gid + i, played like the host-buffer entries: talon group 0, Philox discards and cards.  Returns the dict of
    ``rollout`` plus ``hist`` (int64 [10]: finished games by contract)."""
    n = len(perm)
    perm = np.ascontiguousarray(perm, np.uint8).reshape(n, 54)
    contract = np.ascontiguousarray(contract, np.uint8)
    declarer = np.ascontiguousarray(declarer, np.uint8)
    king = None if king is None else np.ascontiguousarray(king, np.uint8)
    assert contract.shape == declarer.shape == (n,) and (king is None or king.shape == (n,))
    out = dict(scores=np.empty((n, 4), np.int16), plays=np.empty(n, np.uint8),
               contract=np.empty(n, np.uint8), declarer=np.empty(n, np.uint8),
               king=np.empty(n, np.uint8), err=np.empty(n, np.uint8), stats=np.zeros(10, np.int64),
               perm=np.empty((n, 54), np.uint8), cards=np.empty((n, 48), np.uint8),
               group=np.empty(n, np.uint8), discard=np.empty(n, np.uint64), hist=np.zeros(10, np.int64))
    lib().syn_rollout_injected_batch(
        C.c_uint64(seed), C.c_uint64(first_gid), C.c_int64(n), _p(perm), _p(contract), _p(declarer), _p(king),
        _p(out["scores"]), _p(out["plays"]), _p(out["contract"]), _p(out["declarer"]), _p(out["king"]),
        _p(out["err"]), _p(out["perm"]), _p(out["cards"]), _p(out["group"]), _p(out["discard"]), _p(out["stats"]),
        _p(out["hist"]))
    return out


def device_stats(ref):
    """What the device's statistics vector holds in entries 0..20 after the games of an oracle rollout (``rollout`` or
    ``rollout_injected``): seat sums, player sums, finished games by contract, finished games, env steps, error games."""
    fin = ref["err"] == 0
    hist = ref["hist"] if "hist" in ref else np.bincount(ref["contract"][fin], minlength=10)
    st = ref["stats"]
    return np.concatenate([st[0:8], hist, [hist.sum(), st[8], st[9]]]).astype(np.int64)


def rollout_stats_only(seed, first_gid, n, mode):
    """Timing leg for bench.py: no per-game outputs, only the 10-entry stats vector."""
    stats = np.zeros(10, np.int64)
    lib().syn_rollout_batch(
        C.c_uint64(seed), C.c_uint64(first_gid), C.c_int64(n), C.c_int(mode),
        None, None, None, None, None, None, None, None, None, None, _p(stats))
    return stats


def use_all_threads():
    """OpenMP over every core this process may run on (torchrun exports OMP_NUM_THREADS=1); returns the count."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    lib().syn_set_threads(C.c_int(n))
    return int(lib().syn_max_threads())


def set_threads(n: int) -> int:
    lib().syn_set_threads(C.c_int(int(n)))
    return int(lib().syn_max_threads())
