"""Batched Tarok environment: the host-side object over the C ABI (include/tarok_b200.h).

One ``TarokEnv`` owns ``n_games`` concurrent deals on one GPU.  The whole rule engine of the
reference -- ``Igra.razdeli`` (Igra.py:65-73), ``Igra.licitacija`` (Igra.py:75-114), the talon
exchange of ``Navadna_igra.start`` (Navadna_igra.py:36-68), ``mozne_karte`` / ``krog`` /
``pobere_stih`` (Navadna_igra.py:115-168, Klop.py:47-133, Berac.py:13-44) and the scoring
epilogues -- runs in hand-written sm_100a kernels; this class only passes pointers and streams.
PyTorch is used for device memory, streams and DLPack views, nothing else.

All state fields are zero-copy ``torch`` views of the library's HBM arrays (structure of arrays,
one int64 bitboard per game, bit i = card id i).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
from torch.utils import dlpack as _dlpack

from . import _lib

DEFAULT_SEED = 0x5EED7A20C0001
NO_KING = 7
MODE_NAVADNA_MIX = 16
MODE_AUCTION_UNIFORM = 17
MODE_AUCTION_BOT = 18
FLAG_HISTORY = 1

(F_HANDS, F_PILES, F_TALON, F_TALON_ORDER, F_META, F_MASK, F_SCORES, F_HIST, F_STATS, F_HANDS0,
 F_DISCARD, F_QMAX_HIST) = range(12)

# element types of the observation outputs and of the network outputs the selections read (TAROK_DTYPE_*)
DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


def dtype_code(dtype) -> int:
    """TAROK_DTYPE_* of a torch dtype; ValueError for anything but fp32 / bf16 / fp16."""
    if dtype not in DTYPES:
        raise ValueError("observations and network outputs must be float32, bfloat16 or float16, not %s" % (dtype,))
    return DTYPES[dtype]


def _net_out(q, dev):
    """Network outputs as the selections read them: fp32 / bf16 / fp16 pass through, any other dtype is cast to fp32."""
    return q.to(device=dev, dtype=q.dtype if q.dtype in DTYPES else torch.float32).contiguous()


# stats vector layout (include/tarok_b200.h)
S_SEAT, S_PLAYER, S_CONTRACT, S_FINISHED, S_STEPS, S_ERRORS, S_ERR_EVENTS = 0, 4, 8, 18, 19, 20, 21

# meta word layout (tarok_b200/csrc/tarok_rules.cuh)
M_CONTRACT, M_DECL, M_KING, M_TEAM, M_LEADER, M_POS, M_TRICKS, M_WINNER, M_TRICKDONE = 0, 4, 6, 9, 13, 15, 17, 21, 23
M_PHASE, M_ERR, M_GROUP, M_KLOPFAM, M_TRICK, M_PLAYS = 24, 26, 27, 30, 32, 56
PH_DEALT, PH_EXCHANGE, PH_PLAY, PH_DONE = 0, 1, 2, 3

_DLTENSOR = b"dltensor"
C.pythonapi.PyCapsule_New.restype = C.py_object
C.pythonapi.PyCapsule_New.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p]


def meta_field(meta, shift, bits):
    """Extract a bit field from the packed meta words (torch tensor or numpy array)."""
    return (meta >> shift) & ((1 << bits) - 1)


def _host_ptr(a):
    """Address of a contiguous HOST buffer (numpy array or CPU torch tensor), or None."""
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        assert a.device.type == "cpu" and a.is_contiguous()
        return C.c_void_p(a.data_ptr())
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


RECORD_BYTES = 20          # TAROK_RECORD_BYTES


def pack_records(perm, contract, declarer, king=None, out=None, threads: int = 1):
    """Serialises permutation rows (uint8 [n,54], ``Igra.razdeli`` order) + forced contracts (uint8 [n] each) into
    20-byte deal records (uint8 [n,20]; layout in include/tarok_b200.h) on the host, on ``threads`` host threads.
    Returns (records, number of invalid rows)."""
    n = int(perm.shape[0])
    if out is None:
        out = torch.empty((n, RECORD_BYTES), dtype=torch.uint8)
        if torch.cuda.is_available():
            out = out.pin_memory()
    bad = _lib.load().tarok_pack_records_mt(_host_ptr(perm), _host_ptr(contract), _host_ptr(declarer), _host_ptr(king), n,
                                            _host_ptr(out), int(threads))
    if bad < 0:
        raise ValueError("pack_records: perm, contract and declarer are required")
    return out, int(bad)


class TarokEnv:
    def __init__(self, n_games: int, seed: int = DEFAULT_SEED, device: int = 0, history: bool = False):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        self.device = int(device)
        self.n = int(n_games)
        self.seed = int(seed)
        rc = self._lib.tarok_create(self.device, self.n, self.seed & (2 ** 64 - 1),
                                    FLAG_HISTORY if history else 0, C.byref(self._h))
        if rc != 0:
            self._h = C.c_void_p()
            _lib.check(None, rc)
        self.n_alloc = int(self._lib.tarok_n_alloc(self._h))
        self.history = bool(history)
        self._views = {}
        self.torch_device = torch.device("cuda", self.device)

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._views.clear()
            self._bk = None
            rc = self._lib.tarok_destroy(self._h)
            if rc == 0:
                self._h = C.c_void_p()
            else:
                _lib.check(self._h, rc)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.torch_device).cuda_stream)

    def _check(self, rc):
        _lib.check(self._h, rc)

    def _dev_u8(self, x, shape):
        """Accept a CUDA uint8 tensor or anything numpy can read; returns a contiguous CUDA tensor."""
        if not isinstance(x, torch.Tensor):
            x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.uint8)).to(self.torch_device, non_blocking=True)
        if x.dtype != torch.uint8 or x.device != self.torch_device:
            x = x.to(device=self.torch_device, dtype=torch.uint8)
        x = x.contiguous()
        if tuple(x.shape) != tuple(shape):
            raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(x.shape)))
        return x

    def view(self, field: int) -> torch.Tensor:
        """Zero-copy torch view of a state field (DLPack, aliases the library's HBM array)."""
        t = self._views.get(field)
        if t is None:
            out = C.c_void_p()
            self._check(self._lib.tarok_export(self._h, field, C.byref(out)))
            cap = C.pythonapi.PyCapsule_New(out, _DLTENSOR, None)
            t = _dlpack.from_dlpack(cap)
            self._views[field] = t
        return t

    # zero-copy state
    hand_slots = property(lambda self: self.view(F_HANDS))       # int64 [4, n_alloc], row j = seat (leader + j) & 3 (zero-copy)

    @property
    def hands(self):
        """Hand bitboards by SEAT, int64 [4, n_alloc]: a fresh copy (the device keeps them in leader-relative slots)."""
        out = torch.empty((4, self.n_alloc), dtype=torch.int64, device=self.torch_device)
        self._check(self._lib.tarok_hands_by_seat(self._h, C.c_void_p(out.data_ptr()), self._stream()))
        return out
    piles = property(lambda self: self.view(F_PILES))            # int64 [4, n_alloc]
    talon = property(lambda self: self.view(F_TALON))            # int64 [n_alloc]
    talon_order = property(lambda self: self.view(F_TALON_ORDER))
    meta = property(lambda self: self.view(F_META))
    mask = property(lambda self: self.view(F_MASK))              # legal moves of the seat to move
    scores = property(lambda self: self.view(F_SCORES))          # int16 [n_alloc, 4]
    hist = property(lambda self: self.view(F_HIST))              # uint8 [48, n_alloc]
    stats_dev = property(lambda self: self.view(F_STATS))        # int64 [32]
    hands0 = property(lambda self: self.view(F_HANDS0))
    discard = property(lambda self: self.view(F_DISCARD))
    qmax_hist = property(lambda self: self.view(F_QMAX_HIST))    # float32 [48, n_alloc]

    def set_chunks(self, chunks: int):
        """Pipeline depth (1..32, default 8) of the host-buffer entries ``rollout_host(fused=True)`` / ``rollout_records``."""
        self._check(self._lib.tarok_set_option(self._h, 5, int(chunks)))

    def set_materialise(self, on: bool):
        """Whether ``score()`` writes the full piles / Klop talon back (default) or only produces scores + statistics."""
        self._check(self._lib.tarok_set_option(self._h, 4, 1 if on else 0))

    def set_lazy_mask(self, on: bool):
        """Chains of in-kernel random steps write the legal masks in their last launch only (default on)."""
        self._check(self._lib.tarok_set_option(self._h, 6, 1 if on else 0))

    def set_draw_cache(self, rows: int):
        """Trick positions (1..rows) whose in-kernel random draws are read from the cache the position-0 launch of a trick
        leaves behind instead of recomputed: 0 off, 2, 3; -1 = the default for this batch size.  Results are identical."""
        self._check(self._lib.tarok_set_option(self._h, 7, int(rows)))

    def set_graph(self, on: bool):
        """``rollout(fused=False)`` replays a CUDA graph of its 50 launches (default on; same results, ~4 us of host time)."""
        self._check(self._lib.tarok_set_option(self._h, 8, 1 if on else 0))

    def set_lockstep(self, on: bool):
        """Trick-position-specialised play_step for lock-step batches (default on; the kernel verifies the hint)."""
        self._check(self._lib.tarok_set_option(self._h, 3, 1 if on else 0))

    def set_pdl(self, on: bool):
        """Programmatic dependent launch between consecutive play_step kernels (default on)."""
        self._check(self._lib.tarok_set_option(self._h, 2, 1 if on else 0))

    @property
    def launches(self) -> int:
        return int(self._lib.tarok_launch_count(self._h))

    # ------------------------------------------------------------------ deal (Igra.razdeli)
    def deal(self, first_game_id: int = 0):
        self._check(self._lib.tarok_deal(self._h, int(first_game_id), self._stream()))

    def set_deals(self, perm, first_game_id: int = 0):
        """Inject deals: uint8 [n,54] permutations, as a patched ``Igra.shuffle`` would."""
        p = self._dev_u8(perm, (self.n, 54))
        self._check(self._lib.tarok_set_deals(self._h, C.c_void_p(p.data_ptr()), int(first_game_id), self._stream()))

    def export_perm(self) -> torch.Tensor:
        out = torch.empty((self.n, 54), dtype=torch.uint8, device=self.torch_device)
        self._check(self._lib.tarok_export_perm(self._h, C.c_void_p(out.data_ptr()), self._stream()))
        return out

    # ------------------------------------------------------------------ auction / dispatch
    def _bots(self, bots):
        """The per-game seat mask of a mixed table (uint8 [n], bit s = seat s is a Bot_igralec) as a device tensor."""
        return self._dev_u8(bots, (self.n,))

    def auction(self, intents, bots=None):
        """intents: uint8 [n,4] indices into ``Nevronski_igralec.index2igra`` (Igralec.py:717-745), 0..19 (18 Odprti_berac,
        19 Klop); a game with any intent in 20..255 becomes an error game.  ``bots`` (uint8 [n], bit s = seat s is a
        Bot_igralec): those seats bid as Bot_igralec and their intents are ignored (``tarok_auction_bots``)."""
        x = self._dev_u8(intents, (self.n, 4))
        if bots is None:
            self._check(self._lib.tarok_auction(self._h, C.c_void_p(x.data_ptr()), self._stream()))
        else:
            b = self._bots(bots)
            self._check(self._lib.tarok_auction_bots(self._h, C.c_void_p(x.data_ptr()), C.c_void_p(b.data_ptr()), self._stream()))

    def auction_synth(self, mode: int):
        self._check(self._lib.tarok_auction_synth(self._h, int(mode), self._stream()))

    def force_contract(self, contract, declarer, king=None):
        c = self._dev_u8(contract, (self.n,))
        d = self._dev_u8(declarer, (self.n,))
        k = None if king is None else self._dev_u8(king, (self.n,))
        self._check(self._lib.tarok_force_contract(
            self._h, C.c_void_p(c.data_ptr()), C.c_void_p(d.data_ptr()),
            C.c_void_p(k.data_ptr()) if k is not None else None, self._stream()))

    def force_contract_synth(self, mode: int):
        self._check(self._lib.tarok_force_contract_synth(self._h, int(mode), self._stream()))

    # ------------------------------------------------------------------ talon exchange
    def exchange(self, group, discard, bots=None):
        """group: uint8 [n], discard: [n] bitboards of the k cards laid down.  ``bots`` (uint8 [n] seat masks): games whose
        declarer is a bot seat take Bot_igralec's exchange and ignore their entries (``tarok_exchange_bots``)."""
        g = self._dev_u8(group, (self.n,))
        if not isinstance(discard, torch.Tensor):
            discard = torch.from_numpy(np.ascontiguousarray(discard).astype(np.uint64).view(np.int64))
        d = discard.to(device=self.torch_device, dtype=torch.int64).contiguous()
        if tuple(d.shape) != (self.n,):
            raise ValueError("discard must have shape (n,)")
        if bots is None:
            self._check(self._lib.tarok_exchange(self._h, C.c_void_p(g.data_ptr()), C.c_void_p(d.data_ptr()), self._stream()))
        else:
            b = self._bots(bots)
            self._check(self._lib.tarok_exchange_bots(self._h, C.c_void_p(g.data_ptr()), C.c_void_p(d.data_ptr()),
                                                      C.c_void_p(b.data_ptr()), self._stream()))

    def exchange_synth(self, random_group: bool = False):
        self._check(self._lib.tarok_exchange_synth(self._h, 1 if random_group else 0, self._stream()))

    # ------------------------------------------------------------------ play
    def legal_mask(self) -> torch.Tensor:
        """Recompute the legal-move masks from hands+meta (``mozne_karte``); int64 [n]."""
        out = torch.empty(self.n_alloc, dtype=torch.int64, device=self.torch_device)
        self._check(self._lib.tarok_legal_mask(self._h, C.c_void_p(out.data_ptr()), self._stream()))
        return out[: self.n]

    def step(self, cards, bots=None):
        """One card per live game (``igraj_karto``); cards: uint8 [n] card ids.  ``bots`` (uint8 [n] seat masks): a bot to
        move plays the uniform legal card ``step_random`` would and its card byte is ignored, except 0xFE (skip), which
        still holds the game (``tarok_step_bots``)."""
        if isinstance(cards, torch.Tensor) and cards.dtype == torch.uint8 and cards.device == self.torch_device \
                and cards.is_contiguous() and cards.numel() in (self.n, self.n_alloc):
            x = cards                    # used in place (the kernel reads the first n_games bytes only)
        else:
            x = self._dev_u8(cards, (self.n,))
        if bots is None:
            self._check(self._lib.tarok_step(self._h, C.c_void_p(x.data_ptr()), self._stream()))
        else:
            b = self._bots(bots)
            self._check(self._lib.tarok_step_bots(self._h, C.c_void_p(x.data_ptr()), C.c_void_p(b.data_ptr()), self._stream()))

    def step_random(self, count: int = 1):
        """``count`` back-to-back steps with in-kernel uniform-random legal cards (Bot_igralec, Igralec.py:158-159)."""
        if count == 1:
            self._check(self._lib.tarok_step_random(self._h, self._stream()))
        else:
            self._check(self._lib.tarok_steps_random(self._h, int(count), self._stream()))

    # ------------------------------------------------------------------ scoring / stats
    def score(self) -> torch.Tensor:
        """Scores by seat, int16 [n,4] (``pisejo``); also accumulates the statistics vector."""
        self._check(self._lib.tarok_score(self._h, None, self._stream()))
        return self.scores[: self.n]

    def reseed(self, seed: int):
        """A new run seed (the Philox key of every synthetic draw) for this environment, keeping its device buffers."""
        self._check(self._lib.tarok_reseed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF))
        self.seed = int(seed)

    def reset_stats(self):
        self._check(self._lib.tarok_reset_stats(self._h, self._stream()))

    def stats(self) -> np.ndarray:
        out = np.zeros(32, np.int64)
        self._check(self._lib.tarok_read_stats(self._h, out.ctypes.data_as(C.c_void_p), self._stream()))
        return out

    # ------------------------------------------------------------------ whole deals
    def setup_synth(self, mode: int, first_game_id: int = 0):
        """deal + contract(mode) + talon exchange with device-side decisions, one launch."""
        self._check(self._lib.tarok_setup_synth(self._h, int(mode), int(first_game_id), self._stream()))

    def rollout(self, mode: int, first_game_id: int = 0, fused: bool = False):
        """deal -> contract(mode) -> exchange -> random play -> score, all on the device."""
        fn = self._lib.tarok_rollout_fused if fused else self._lib.tarok_rollout_stepwise
        self._check(fn(self._h, int(mode), int(first_game_id), self._stream()))

    def rollout_host(self, perm, contract, declarer, king, scores_out, stats_out, first_game_id: int = 0,
                     fused: bool = False):
        """End-to-end entry with HOST buffers (numpy arrays or pinned CPU torch tensors).

        Uploads the injected deals + forced contracts, plays them with uniform-random players and
        downloads ``scores_out`` (int16 [n,4]) and ``stats_out`` (int64 [32]).  Asynchronous on the
        current stream when the buffers are pinned; the caller synchronises."""
        hp = _host_ptr
        self._check(self._lib.tarok_rollout_host(
            self._h, hp(perm), hp(contract), hp(declarer), hp(king), int(first_game_id), 1 if fused else 0,
            hp(scores_out), hp(stats_out), self._stream()))

    def rollout_host_packed(self, perm, contract, declarer, king, scores_out, stats_out, first_game_id: int = 0,
                            threads: int = 1):
        """``rollout_host(fused=True)`` with the rows serialised into 20-byte records by ``threads`` host threads inside the
        call, chunk by chunk ahead of each upload (PCIe carries 20 instead of 57 bytes per deal)."""
        hp = _host_ptr
        self._check(self._lib.tarok_rollout_host_packed(
            self._h, hp(perm), hp(contract), hp(declarer), hp(king), int(first_game_id), int(threads),
            hp(scores_out), hp(stats_out), self._stream()))

    def rollout_records(self, records, scores_out, stats_out, first_game_id: int = 0):
        """``rollout_host(fused=True)`` fed with 20-byte deal records (``pack_records``; layout in include/tarok_b200.h):
        the same deals, contracts and scores for 2.85x fewer bytes over PCIe."""
        hp = _host_ptr
        self._check(self._lib.tarok_rollout_records(self._h, hp(records), int(first_game_id), hp(scores_out),
                                                    hp(stats_out), self._stream()))

    # ------------------------------------------------------------------ observations (Igralec.py:453-533)
    def obs_shape(self):
        """Per game: (net type uint8 [n] -- 0 Klop 1 Navadna_igra 2 Solo 3 Berac, 255 = not to move; T uint8 [n])."""
        t = torch.empty(self.n, dtype=torch.uint8, device=self.torch_device)
        r = torch.empty(self.n, dtype=torch.uint8, device=self.torch_device)
        self._check(self._lib.tarok_obs_shape(self._h, C.c_void_p(t.data_ptr()), C.c_void_p(r.data_ptr()), self._stream()))
        return t, r

    def obs_buckets(self, players: int = 4):
        """Device-side bucketing of the games waiting for a card by (player, net type, T) -- ``predict_igraj_karto``'s
        queues of the ``players`` (1 or 4) players of ``Tarok.paralel_start``.  Returns (sel int32 [n] on the device: game
        indices grouped by key, counts: numpy uint32 [384] on the host = 128 bucket sizes, 128 offsets into ``sel`` (entry
        255 = games listed), 128 offsets in observation rows); key = player * 28 + net_type * 7 + (T / 8 - 1).
        One small device-to-host copy: the only synchronisation of a self-play step."""
        if getattr(self, "_bk", None) is None:
            self._bk = (torch.empty(self.n_alloc, dtype=torch.int32, device=self.torch_device),
                        torch.zeros(384, dtype=torch.int32, device=self.torch_device),
                        torch.zeros(384, dtype=torch.int32).pin_memory(),
                        torch.empty(self.n_alloc, dtype=torch.uint8, device=self.torch_device),
                        torch.zeros(128, dtype=torch.int64).pin_memory(),
                        torch.zeros(128, dtype=torch.int64, device=self.torch_device))
        sel, cnt, host, selkey = self._bk[:4]
        self._check(self._lib.tarok_obs_buckets_host(self._h, int(players), C.c_void_p(sel.data_ptr()), C.c_void_p(cnt.data_ptr()),
                                                     C.c_void_p(selkey.data_ptr()), C.c_void_p(host.data_ptr()), self._stream()))
        torch.cuda.current_stream(self.torch_device).synchronize()
        return sel, host.numpy().view(np.uint32)

    def obs_expand_buckets(self, n_total: int, opp, hand, talon, talon_klop, king, decl, discard):
        """ONE launch for every bucket of the last ``obs_buckets``: the arenas (flat CUDA tensors of one dtype -- fp32, bf16 or
        fp16 -- capacities n * 56 rows / n entries) receive each bucket's inputs as contiguous blocks (layout in
        include/tarok_b200.h)."""
        arenas = (opp, hand, talon, talon_klop, king, decl, discard)
        dtypes = {t.dtype for t in arenas}
        if len(dtypes) != 1:
            raise ValueError("the observation arenas mix dtypes: %s" % sorted(str(d) for d in dtypes))
        code = dtype_code(dtypes.pop())
        sel, cnt, _, selkey = self._bk[:4]
        p = lambda t: C.c_void_p(t.data_ptr())
        self._check(self._lib.tarok_obs_expand_buckets_ex(self._h, code, p(sel), p(selkey), p(cnt), int(n_total),
                                                          *[p(t) for t in arenas], self._stream()))

    def select_action_buckets(self, n_total: int, q_by_key: dict, random_card4, cards, qmax=None):
        """ONE launch of ``select_action`` for every bucket: ``q_by_key[key]`` = that bucket's [size, 54] network output
        (contiguous CUDA tensors, kept alive by the caller until the stream has run the launch).  fp32, bf16 and fp16 outputs
        are read as they are (one dtype for the whole table); other dtypes are cast to fp32."""
        dtypes = {q.dtype for q in q_by_key.values()}
        if len(dtypes) > 1:
            raise ValueError("the bucket outputs mix dtypes: %s" % sorted(str(d) for d in dtypes))
        q_by_key = {k: _net_out(q, self.torch_device) for k, q in q_by_key.items()}
        code = DTYPES[next(iter(q_by_key.values())).dtype] if q_by_key else 0
        sel, cnt, _, selkey = self._bk[:4]
        tab = (C.c_void_p * 128)()                                   # travels as kernel parameters
        for k, q in q_by_key.items():
            tab[k] = q.data_ptr()
        eps = (C.c_float * 4)(*[float(x) for x in random_card4])
        p = lambda t: C.c_void_p(t.data_ptr())
        self._check(self._lib.tarok_select_action_buckets_tab_ex(self._h, code, tab, p(sel), p(selkey), p(cnt), int(n_total), eps,
                                                                 p(cards), p(qmax) if qmax is not None else None, self._stream()))

    def obs_expand(self, net_type: int, rows: int, sel=None, play=None, dtype=torch.float32):
        """The network inputs of ``Nevronski_igralec.stanje_v_vektor_rek_navadna`` for the seat to move of the
        selected games (int32 indices; None = all), as ``dtype`` tensors (fp32, bf16 or fp16) in the reference's list order
        (A.4): Navadna [opp, king, hand, talon, decl, discard, mozne]; Solo [opp, hand, talon, decl, discard, mozne];
        Klop [opp, hand, talon, mozne]; Berac [opp, hand, decl, mozne].  Returns (list of tensors, ok uint8 [n_sel]).
        ``play=t`` gives the observation as it was at card play t, for the seat that made it (replay samples)."""
        if not self.history:
            raise ValueError("observations need TarokEnv(..., history=True)")
        if sel is None:
            n_sel, sel_ptr = self.n, None
        else:
            sel = torch.as_tensor(sel, dtype=torch.int32, device=self.torch_device).contiguous()
            n_sel, sel_ptr = int(sel.numel()), C.c_void_p(sel.data_ptr())
        code = dtype_code(dtype)
        dev, f = self.torch_device, dtype
        opp = torch.empty((n_sel, rows, 3, 54), dtype=f, device=dev)
        hand = torch.empty((n_sel, rows, 54), dtype=f, device=dev)
        talon = torch.empty((n_sel, 54) if net_type == 0 else (n_sel, 6, 55), dtype=f, device=dev) if net_type != 3 else None
        king = torch.empty((n_sel, 4), dtype=f, device=dev) if net_type == 1 else None
        decl = torch.empty((n_sel, 4), dtype=f, device=dev) if net_type != 0 else None
        disc = torch.empty((n_sel, 54), dtype=f, device=dev) if net_type in (1, 2) else None
        mozne = torch.empty((n_sel, 54), dtype=f, device=dev)
        ok = torch.empty(n_sel, dtype=torch.uint8, device=dev)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        self._check(self._lib.tarok_obs_expand_at_ex(self._h, code, -1 if play is None else int(play), int(net_type), int(rows),
                                                     sel_ptr, n_sel, p(opp), p(hand), p(talon), p(king), p(decl), p(disc), p(mozne),
                                                     p(ok), self._stream()))
        order = {1: [opp, king, hand, talon, decl, disc, mozne], 2: [opp, hand, talon, decl, disc, mozne],
                 0: [opp, hand, talon, mozne], 3: [opp, hand, decl, mozne]}[int(net_type)]
        return order, ok

    def select_action(self, q, sel=None, random_card: float = 0.0, cards=None, qmax=None):
        """``Nevronski_igralec.igraj_karto`` (Igralec.py:344-355) for the selected games: first argmax of ``q`` ([n_sel,54];
        fp32, bf16 and fp16 are read as they are, other dtypes cast to fp32) over the legal cards in the reference's ``mozne``
        order, epsilon-greedy with ``random_card``.  Writes into ``cards`` (uint8 [n], by game index; allocated if None) and
        returns (cards, qmax fp32)."""
        q = _net_out(q, self.torch_device)
        if sel is None:
            n_sel, sel_ptr = self.n, None
        else:
            sel = torch.as_tensor(sel, dtype=torch.int32, device=self.torch_device).contiguous()
            n_sel, sel_ptr = int(sel.numel()), C.c_void_p(sel.data_ptr())
        if tuple(q.shape) != (n_sel, 54):
            raise ValueError("q must have shape (n_sel, 54)")
        if cards is None:
            cards = torch.full((self.n_alloc,), 0xFF, dtype=torch.uint8, device=self.torch_device)
        if qmax is None:
            qmax = torch.zeros(self.n, dtype=torch.float32, device=self.torch_device)
        self._check(self._lib.tarok_select_action_ex(self._h, DTYPES[q.dtype], C.c_void_p(q.data_ptr()), sel_ptr, n_sel,
                                                     float(random_card), C.c_void_p(cards.data_ptr()), C.c_void_p(qmax.data_ptr()),
                                                     self._stream()))
        return cards, qmax

    def targets(self, sel=None, final_reword_factor: float = 0.1):
        """Replay targets of ``Nevronski_igralec.rezultat_stiha`` / ``rezultat_igre`` (Igralec.py:387-446) for finished games:
        (dy fp32 [n_sel,48,54], seat uint8 [n_sel,48] (0xFF = no play), T uint8 [n_sel,48])."""
        if not self.history:
            raise ValueError("replay targets need TarokEnv(..., history=True)")
        n_sel, sel_ptr, keep = self._sel(sel)
        dy = torch.empty((n_sel, 48, 54), dtype=torch.float32, device=self.torch_device)
        seat = torch.empty((n_sel, 48), dtype=torch.uint8, device=self.torch_device)
        rows = torch.empty((n_sel, 48), dtype=torch.uint8, device=self.torch_device)
        self._check(self._lib.tarok_targets(self._h, sel_ptr, n_sel, float(final_reword_factor), C.c_void_p(dy.data_ptr()),
                                            C.c_void_p(seat.data_ptr()), C.c_void_p(rows.data_ptr()), self._stream()))
        return dy, seat, rows

    def obs_hands(self, dtype=torch.float32) -> torch.Tensor:
        """``pripavi_licitiram`` (Igralec.py:278-281): [n,4,54] in ``dtype`` (fp32, bf16 or fp16), the hand of every seat."""
        code = dtype_code(dtype)
        out = torch.empty((self.n, 4, 54), dtype=dtype, device=self.torch_device)
        self._check(self._lib.tarok_obs_hands_ex(self._h, code, C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def _sel(self, sel):
        if sel is None:
            return self.n, None, None
        sel = torch.as_tensor(sel, dtype=torch.int32, device=self.torch_device).contiguous()
        return int(sel.numel()), C.c_void_p(sel.data_ptr()), sel

    def obs_exchange(self, sel=None, dtype=torch.float32):
        """``menjaj_talon_v_vektor`` (Igralec.py:535-543): ([hand (B,54), talon (B,54,6), game (B,15)] in ``dtype``, ok)."""
        code = dtype_code(dtype)
        n_sel, sel_ptr, keep = self._sel(sel)
        dev, f = self.torch_device, dtype
        hand = torch.empty((n_sel, 54), dtype=f, device=dev)
        talon = torch.empty((n_sel, 54, 6), dtype=f, device=dev)
        game = torch.empty((n_sel, 15), dtype=f, device=dev)
        ok = torch.empty(n_sel, dtype=torch.uint8, device=dev)
        self._check(self._lib.tarok_obs_exchange_ex(self._h, code, sel_ptr, n_sel, C.c_void_p(hand.data_ptr()),
                                                    C.c_void_p(talon.data_ptr()), C.c_void_p(game.data_ptr()), C.c_void_p(ok.data_ptr()),
                                                    self._stream()))
        return [hand, talon, game], ok

    def select_exchange(self, p, sel=None, random_card: float = 0.0, group_out=None, discard_out=None):
        """``menjaj_iz_talona`` (Igralec.py:365-385) from the exchange net's 60 outputs (fp32, bf16 and fp16 read as they are,
        other dtypes cast to fp32): (group uint8 [n], discard int64 [n]); ``group_out`` / ``discard_out`` let several calls
        (one per player) fill the same arrays."""
        n_sel, sel_ptr, keep = self._sel(sel)
        p = _net_out(p, self.torch_device)
        if tuple(p.shape) != (n_sel, 60):
            raise ValueError("p must have shape (n_sel, 60)")
        group = group_out if group_out is not None else torch.full((self.n,), 0xFF, dtype=torch.uint8, device=self.torch_device)
        discard = discard_out if discard_out is not None else torch.zeros(self.n, dtype=torch.int64, device=self.torch_device)
        self._check(self._lib.tarok_select_exchange_ex(self._h, DTYPES[p.dtype], C.c_void_p(p.data_ptr()), sel_ptr, n_sel,
                                                       float(random_card), C.c_void_p(group.data_ptr()), C.c_void_p(discard.data_ptr()),
                                                       self._stream()))
        return group, discard

    # ------------------------------------------------------------------ helpers
    def errors(self) -> int:
        """Number of games whose error bit is set (illegal action / invalid exchange / bad deal)."""
        return int(((self.meta[: self.n] >> M_ERR) & 1).sum().item())

    def live(self) -> torch.Tensor:
        """bool [n]: games still waiting for a card."""
        return meta_field(self.meta[: self.n], M_PHASE, 2) == PH_PLAY
