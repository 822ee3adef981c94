"""Batched neural self-play on the device (BASELINE config 4).

What ``Tarok.paralel_start`` does with four ``Nevronski_igralec`` (``Tarok.py:30-62``; ``main.py:48-66``;
``Igralec.py:278-385``) -- every player queues one observation per game it has to act in, runs one batched forward per
net type, then per game a ``.cpu()`` sync, an argmax over the legal cards and a Python state update -- becomes, per
phase, a handful of launches over the whole batch:

    deal -> obs_hands -> Vrednotenje_roke (per player) -> argmax/epsilon -> auction
         -> obs_exchange -> Zalaganje (per player) -> select_exchange -> exchange
         -> 48 x [ obs_buckets -> per (player, net, T) bucket: obs_expand -> net forward -> select_action ] -> step
         -> score

The reference seats FOUR players, each with its own six networks and its own epsilon (``main.py:48-66``,
``Igralec.py:190,235-248``); game i seats them rotated by i % 4 (``Tarok.py:34``), so the player of seat s in game i is
(s + i) % 4.  The buckets of ``predict_igraj_karto`` (one queue per net type per player, stacked per history length T,
``Igralec.py:316-342``) are formed on the DEVICE by a counting sort (``tarok_obs_buckets``): the host reads 128 counts
once per step -- the only synchronisation of a step -- and walks the non-empty ranges.

The environment, the bucketing, the observation expansion and the action selection are the CUDA kernels of this
repository; the forward passes stay in the reference's networks (here the PyTorch restatement in ``tarok_b200.mreze``,
because the upstream ``torch_models.py`` is missing).

Mixed tables: ``Samoigra(..., boti=(2, 3))`` seats ``Bot_igralec`` players beside the neural ones (the usual yardstick of a
self-play net is its score against uniform-random players).  A bot player needs no nets; its bids, king call, exchange and
cards are drawn in-kernel by the ``*_bots`` entries (``tarok_auction_bots`` / ``tarok_exchange_bots`` /
``tarok_step_bots``) from a per-game seat mask built once per rollout, its forwards are skipped (a bucket without a forward
is left alone by the action selection), it yields no replay samples, and ``stats[4 + p]`` is its score like anybody's.

Mixed precision: ``Samoigra(..., dtype=torch.bfloat16)`` (or ``torch.float16``) plays with observations written in that
dtype (every value is 0 or 1, so they are exact) and with inference copies of the nets cast to it; the selections read the
half outputs as they come.  The fp32 master nets, ``nauci`` and ``vzorci`` stay fp32.
"""
from __future__ import annotations

import copy
import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Union

import torch

from . import env as E
from .mreze import ustvari_mreze

_NET_OF_KIND = {0: "Klop", 1: "Navadna_igra", 2: "Solo", 3: "Berac"}          # Nevronski_igralec.Tipi_NN


class _Ura:
    """CUDA-event stopwatch per section (summed after one synchronise)."""

    def __init__(self, on):
        self.on, self.pairs = on, {}

    def __call__(self, name):
        return _Odsek(self, name)

    def ms(self) -> Dict[str, float]:
        torch.cuda.synchronize()
        return {k: sum(a.elapsed_time(b) for a, b in v) for k, v in self.pairs.items()}


class _Odsek:
    def __init__(self, ura, name):
        self.ura, self.name = ura, name

    def __enter__(self):
        if self.ura.on:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.ura.on:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            self.ura.pairs.setdefault(self.name, []).append((self.a, b))


class _Arena:
    """Output buffers of the observation kernels, allocated once for the largest bucket (n games, T = 56) and re-used by
    every bucket of every step (the launches of one stream are ordered, so a bucket's forward has consumed its inputs before
    the next expansion overwrites them)."""

    def __init__(self, n, dev, f=torch.float32):
        self.opp = torch.empty(n * 56 * 162, dtype=f, device=dev)
        self.hand = torch.empty(n * 56 * 54, dtype=f, device=dev)
        self.talon = torch.empty(n * 330, dtype=f, device=dev)
        self.talon_klop = torch.empty(n * 54, dtype=f, device=dev)
        self.king = torch.empty(n * 4, dtype=f, device=dev)
        self.decl = torch.empty(n * 4, dtype=f, device=dev)
        self.disc = torch.empty(n * 54, dtype=f, device=dev)


class Samoigra:
    """``igralci`` = 4 (default): four players with their own networks and epsilon, as in the reference; ``igralci`` = 1:
    one shared set plays every seat.  ``mreze``: None (fresh random nets), one dict (shared, implies one player) or a
    sequence of four dicts; ``random_card``: one epsilon or one per player (``Nevronski_igralec.random_card``);
    ``dtype``: element type of the observations and of the inference forwards (fp32, bf16 or fp16); ``boti``: the players
    (0..3, with ``igralci`` = 4) that are ``Bot_igralec`` -- their entry of ``mreze`` may be None and their ``random_card``
    is ignored."""

    def __init__(self, n_envs: int, mreze: Union[None, dict, Sequence[dict]] = None, device: int = 0,
                 seed: Optional[int] = None, random_card: Union[float, Sequence[float]] = 0.05, igralci: int = 4,
                 dtype: torch.dtype = torch.float32, boti: Sequence[int] = ()):
        E.dtype_code(dtype)                                            # ValueError for anything but fp32 / bf16 / fp16
        boti = frozenset(int(p) for p in boti)
        if boti and (igralci != 4 or isinstance(mreze, dict)):
            raise ValueError("Bot_igralec players need the four players of igralci=4")
        if any(p < 0 or p > 3 for p in boti):
            raise ValueError("boti holds player indices 0..3, got %s" % sorted(boti))
        if seed is None:
            seed = int.from_bytes(os.urandom(8), "little")
        self.env = E.TarokEnv(n_envs, seed=seed, device=device, history=True)
        self.n = n_envs
        self.dev = self.env.torch_device
        if isinstance(mreze, dict):
            mreze, igralci = [mreze], 1
        if igralci not in (1, 4):
            raise ValueError("igralci must be 1 (one shared set of nets) or 4 (the reference's four players)")
        self.igralci = igralci
        self.boti = boti
        self.mreze: List[Optional[dict]] = list(mreze) if mreze is not None else \
            [None if p in boti else ustvari_mreze(self.dev) for p in range(igralci)]
        if len(self.mreze) != igralci:
            raise ValueError("need %d sets of nets" % igralci)
        if any(d is None for p, d in enumerate(self.mreze) if p not in boti):
            raise ValueError("every player that is not a bot needs its nets")
        for d in self.mreze:
            for m in (d or {}).values():
                m.eval()                                               # Igralec.py:335
        eps = [float(random_card)] * igralci if isinstance(random_card, (int, float)) else [float(x) for x in random_card]
        if len(eps) != igralci:
            raise ValueError("need one random_card per player")
        self.random_card = eps
        self.gen = torch.Generator(device=self.dev)
        self.gen.manual_seed(seed & 0x7FFFFFFFFFFFFFFF)
        self.dtype = dtype
        self._kopije = {}                # (player, net name) -> (master net, its copy cast to dtype)
        self._arena = None
        self.zadnji_koraki = None        # per step: number of buckets walked (diagnostics)

    # ------------------------------------------------------------------ helpers
    def _igralec_sedeza(self, first_game_id: int) -> torch.Tensor:
        """int64 [n,4]: the player of every seat, (seat + global game id) % 4 (Tarok.py:34); zeros for one shared player."""
        if self.igralci == 1:
            return torch.zeros((self.n, 4), dtype=torch.int64, device=self.dev)
        gid = torch.arange(self.n, dtype=torch.int64, device=self.dev) + int(first_game_id)
        return (gid[:, None] + torch.arange(4, dtype=torch.int64, device=self.dev)[None, :]) & 3

    def _maska_botov(self, kdo: torch.Tensor) -> torch.Tensor:
        """uint8 [n]: bit s set = the player of seat s (``kdo``) is a bot -- the seat mask of the ``*_bots`` entries."""
        bot = torch.isin(kdo, torch.tensor(sorted(self.boti), dtype=kdo.dtype, device=self.dev))
        return (bot.to(torch.uint8) << torch.arange(4, dtype=torch.uint8, device=self.dev)).sum(dim=1, dtype=torch.uint8)

    def _vhod(self, vr: int, T: int, B: int, off: int, row: int):
        """The input list of one bucket (reference order, A.4) as views of the arenas ``obs_expand_buckets`` filled:
        ``off`` = the bucket's offset in games, ``row`` = its offset in observation rows."""
        a = self._arena
        opp = a.opp[row * 162: (row + B * T) * 162].view(B, T, 3, 54)
        hand = a.hand[row * 54: (row + B * T) * 54].view(B, T, 54)
        if vr == 0:
            return [opp, hand, a.talon_klop[off * 54: (off + B) * 54].view(B, 54)]
        decl = a.decl[off * 4: (off + B) * 4].view(B, 4)
        if vr == 3:
            return [opp, hand, decl]
        talon = a.talon[off * 330: (off + B) * 330].view(B, 6, 55)
        disc = a.disc[off * 54: (off + B) * 54].view(B, 54)
        if vr == 2:
            return [opp, hand, talon, decl, disc]
        return [opp, a.king[off * 4: (off + B) * 4].view(B, 4), hand, talon, decl, disc]

    def _mreze_igre(self) -> List[dict]:
        """The nets the forwards of ``odigraj`` run: the fp32 masters themselves, or for another dtype copies cast to it that
        take the masters' current weights and buffers at every rollout (a few hundred KB)."""
        if self.dtype == torch.float32:
            return self.mreze
        out = []
        for p, d in enumerate(self.mreze):
            if d is None:                                              # a bot player
                out.append(None)
                continue
            c = {}
            for k, m in d.items():
                izvor, kopija = self._kopije.get((p, k), (None, None))
                if izvor is not m:
                    kopija = copy.deepcopy(m).to(self.dtype)
                    self._kopije[(p, k)] = (m, kopija)
                else:
                    for a, b in zip(kopija.state_dict().values(), m.state_dict().values()):
                        a.copy_(b)
                c[k] = kopija.eval()
            out.append(c)
        return out

    # ------------------------------------------------------------------ one rollout
    @torch.no_grad()
    def odigraj(self, first_game_id: int = 0, meri: bool = False):
        """Plays the whole batch once.  Returns (stats int64[32], per-section milliseconds or None)."""
        env, n, ura, P, dt, mreze = self.env, self.n, _Ura(meri), self.igralci, self.dtype, self._mreze_igre()
        if self._arena is None:
            self._arena = _Arena(n, self.dev, dt)
        env.reset_stats()
        with ura("env"):
            env.deal(first_game_id)
        kdo = self._igralec_sedeza(first_game_id)                              # [n,4] player of each seat
        boti = self._maska_botov(kdo) if self.boti else None                  # seat masks of the *_bots entries
        # ---- bidding: Nevronski_igralec.pripavi_licitiram / predict_licitiram / licitiram (Igralec.py:278-306)
        with ura("obs"):
            x = env.obs_hands(dt)                                              # [n,4,54]
        namen = torch.zeros((n, 4), dtype=torch.int64, device=self.dev)
        vrsta_iger = torch.arange(n, device=self.dev)
        for p in range(P):
            if p in self.boti:                                                 # bids in-kernel: no forward
                continue
            if P == 4:                                                         # one seat per game belongs to player p
                with ura("bucket"):
                    sedez = (p - (vrsta_iger + int(first_game_id))) & 3
                    xp = x[vrsta_iger, sedez]
                with ura("forward"):
                    y = mreze[p]["Vrednotenje_roke"](xp)                       # [n,18]
                with ura("select"):
                    namen[vrsta_iger, sedez] = y.argmax(dim=-1)
            else:
                with ura("forward"):
                    y = mreze[0]["Vrednotenje_roke"](x.view(n * 4, 54)).view(n, 4, 18)
                with ura("select"):
                    namen = y.argmax(dim=-1)
        with ura("select"):                                                    # random.random() < random_card (Igralec.py:300-301)
            eps = torch.tensor(self.random_card, dtype=torch.float32, device=self.dev)[kdo]      # the seat's player's epsilon
            if max(self.random_card) > 0:
                razisci = torch.rand((n, 4), device=self.dev, generator=self.gen) < eps
                nakljucno = torch.randint(0, 18, (n, 4), device=self.dev, generator=self.gen)
                namen = torch.where(razisci, nakljucno, namen)
        with ura("env"):
            env.auction(namen.to(torch.uint8), bots=boti)
        # ---- talon exchange (Igralec.py:357-385): the declarer's player decides
        with ura("bucket"):
            meta = env.meta[:n]
            menja = E.meta_field(meta, E.M_PHASE, 2) == E.PH_EXCHANGE
            decl = E.meta_field(meta, E.M_DECL, 2)
            lastnik = torch.gather(kdo, 1, decl[:, None]).squeeze(1)
        kupcek = torch.full((n,), 0xFF, dtype=torch.uint8, device=self.dev)
        zalozi = torch.zeros(n, dtype=torch.int64, device=self.dev)
        for p in range(P):
            if p in self.boti:                                                 # exchanges in-kernel
                continue
            with ura("bucket"):
                sel = torch.nonzero(menja & (lastnik == p)).flatten().to(torch.int32)
            if sel.numel() == 0:
                continue
            with ura("obs"):
                vhod, _ = env.obs_exchange(sel, dt)
            with ura("forward"):
                q = mreze[p]["Zalaganje"](vhod)
            with ura("select"):
                env.select_exchange(q, sel, self.random_card[p], group_out=kupcek, discard_out=zalozi)
        with ura("env"):
            env.exchange(kupcek, zalozi, bots=boti)
        # ---- 48 card plays (Igralec.py:312-355)
        karte = torch.full((env.n_alloc,), 0xFF, dtype=torch.uint8, device=self.dev)
        qmax = torch.zeros(n, dtype=torch.float32, device=self.dev)
        eps4 = (self.random_card * 4)[:4]
        koraki, ar = [], self._arena
        for _ in range(48):
            with ura("bucket"):                                                # counting sort on the device + 1.5 KB to the host
                sel_all, stevci = env.obs_buckets(4 if P == 4 else 1)
            skupaj = int(stevci[255])
            if skupaj == 0:
                break
            with ura("obs"):                                                   # every bucket's inputs in one launch
                env.obs_expand_buckets(skupaj, ar.opp, ar.hand, ar.talon, ar.talon_klop, ar.king, ar.decl, ar.disc)
            polni = [k for k in range(127) if stevci[k] and k // 28 not in self.boti]   # a bot's bucket: no forward
            koraki.append(len(polni))
            q = {}
            with ura("forward"):
                for k in polni:
                    p, vr, T = k // 28, (k % 28) // 7, 8 * (k % 7 + 1)
                    vhod = self._vhod(vr, T, int(stevci[k]), int(stevci[128 + k]), int(stevci[256 + k]))
                    q[k] = mreze[p][_NET_OF_KIND[vr]](vhod).contiguous()           # the legal-mask vector is not a net input (Igralec.py:333)
            with ura("select"):                                                # every bucket's argmax / epsilon in one launch
                env.select_action_buckets(skupaj, q, eps4, karte, qmax)
            with ura("env"):
                env.step(karte, bots=boti)
        with ura("env"):
            env.score()
        self.zadnji_koraki = koraki
        st = env.stats()
        return st, (ura.ms() if meri else None)

    # ------------------------------------------------------------------ replay samples (Igralec.py:441-443)
    @torch.no_grad()
    def vzorci(self, final_reword_factor: float = 0.1, first_game_id: int = 0):
        """Replay samples of the batch just played, bucketed like ``Nevronski_igralec.zgodovina[(tip, T)]`` of each
        player (Igralec.py:441-443): yields (player, net name, T, stanje list without the legal-mask vector, dy [B,54])."""
        env, n = self.env, self.n
        dy, seat, rows = env.targets(final_reword_factor=final_reword_factor)
        vrsta = E.meta_field(env.meta[:n], E.M_CONTRACT, 4)
        kind = torch.full_like(vrsta, 2)                                   # Solo_* ...
        kind = torch.where(vrsta == 0, torch.zeros_like(kind), kind)       # Klop
        kind = torch.where((vrsta >= 1) & (vrsta <= 3), torch.ones_like(kind), kind)
        kind = torch.where((vrsta == 7) | (vrsta == 9), torch.full_like(kind, 3), kind)
        gid = torch.arange(n, dtype=torch.int64, device=self.dev) + int(first_game_id)
        boti = torch.tensor(sorted(self.boti), dtype=torch.int64, device=self.dev)
        for t in range(48):
            igrano = seat[:, t] != 0xFF
            if not bool(igrano.any()):
                break
            igralec = ((seat[:, t].to(torch.int64) + gid) & 3) if self.igralci == 4 else torch.zeros_like(gid)
            igrano &= ~torch.isin(igralec, boti)                          # a bot's plays are no samples
            kljuc = igralec * 256 + kind * 64 + rows[:, t].to(kind.dtype)
            for k in torch.unique(kljuc[igrano]).tolist():
                p, vr, T = k // 256, (k % 256) // 64, k % 64
                sel = torch.nonzero(igrano & (kljuc == k)).flatten().to(torch.int32)
                stanje, ok = env.obs_expand(vr, T, sel, play=t)
                yield p, _NET_OF_KIND[vr], T, stanje[:-1], dy[sel.long(), t]

    def nauci(self, final_reword_factor: float = 0.1, lr: float = 1e-3, first_game_id: int = 0):
        """One optimisation pass over the samples of the last batch: Huber(delta=25) + Adam per play net of each player, the
        loss and optimiser of the reference's models (train.py:23-25; Igralec.py:545-607 fits them with Lightning).
        Training is outside the accelerated path; this exists so the self-play loop closes.  Returns {(player, net): loss}."""
        opt = {(p, k): torch.optim.Adam(self.mreze[p][k].parameters(), lr=lr)
               for p in range(self.igralci) if p not in self.boti for k in _NET_OF_KIND.values()}
        izguba, stevec = {}, {}
        for p, ime, T, stanje, dy in self.vzorci(final_reword_factor, first_game_id):
            m = self.mreze[p][ime]
            m.train()
            with torch.enable_grad():
                for a in range(0, dy.shape[0], 4096):
                    x = [s[a:a + 4096] for s in stanje]
                    if x[0].shape[0] < 2:
                        continue                                           # BatchNorm needs more than one sample
                    l = torch.nn.functional.huber_loss(m(x), dy[a:a + 4096], delta=25.0)
                    opt[(p, ime)].zero_grad(set_to_none=True)
                    l.backward()
                    opt[(p, ime)].step()
                    izguba[(p, ime)] = izguba.get((p, ime), 0.0) + float(l.detach())
                    stevec[(p, ime)] = stevec.get((p, ime), 0) + 1
            m.eval()
        return {k: izguba[k] / stevec[k] for k in izguba}

    def zapri(self):
        self.env.close()
