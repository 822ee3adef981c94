"""TEST INFRASTRUCTURE ONLY -- parameter-free stand-ins for the six networks of a neural player, for judging whole
self-play rollouts decision by decision.

Every output is a small non-negative integer (below the player's modulus, at most 13) computed from the inputs with
integer weights, so it is exact in fp32, bf16 and fp16, and the same module run on CPU in float64 is the host reference.
Inputs are widened to fp32 (float64 stays float64) before any arithmetic, so no half-precision sum can round (the
contractions multiply 0/1 inputs by integer weights of at most 15, exact even where a GEMM rounds its inputs to TF32, and
every partial sum is an integer far below 2^24); the result is returned in the input dtype, which keeps the
half-precision selections of self-play on their own path.

What the modules are built to notice:
  * every tensor of the input list changes the output, each with its own card pattern (the king and decl one-hots, both
    [B,4], count differently);
  * history rows are weighted from the END of the sequence, w(r) = ((T - 1 - r) mod 5) + 1, so a game put in the wrong
    T bucket, or rows shifted by one, changes the values;
  * a per-player salt (and per net type, for the four play nets) and a per-player modulus m (7, 9, 11, 13): the same
    input gives different decisions for different players;
  * the final ``mod m`` makes ties at the top common but not universal, so the list-order tie rules are exercised.
"""
from __future__ import annotations

import numpy as np
import torch
from torch import nn

MODULI = (7, 9, 11, 13)


def _f(x):
    return torch.float64 if x.dtype == torch.float64 else torch.float32


def _pattern(a, salt, dev, f):
    """Card pattern [54] in 0..6: (a * card + salt + 1) mod 7."""
    return ((torch.arange(54, device=dev) * a + salt + 1) % 7).to(f)


def _rows_from_end(T, dev, f):
    return (((T - 1 - torch.arange(T, device=dev)) % 5) + 1).to(f)


class Igra(nn.Module):
    """Klop / Navadna_igra / Solo / Berac: the input list in the reference's order -> [B,54]."""

    def __init__(self, salt, m):
        super().__init__()
        self.salt, self.m = salt, m

    def forward(self, x):
        dt, dev, f = x[0].dtype, x[0].device, _f(x[0])
        y = _pattern(self.salt + 2, self.salt, dev, f) * self.salt
        for j, v in enumerate(x):
            v = v.to(f)
            if v.dim() == 4:                                            # opp [B,T,3,54]
                w = _rows_from_end(v.shape[1], dev, f)[:, None] * torch.arange(1, 4, device=dev).to(f)[None, :]
                u = torch.einsum("btoc,to->bc", v, w)
            elif v.dim() == 3 and v.shape[2] == 54:                     # hand [B,T,54]
                u = torch.einsum("btc,t->bc", v, _rows_from_end(v.shape[1], dev, f))
            elif v.dim() == 3:                                          # talon [B,6,55]: card rows, "in the chosen group"
                jw = torch.arange(1, 7, device=dev).to(f)
                chosen = (v[:, :, 54] * (jw + 1)).sum(1, keepdim=True)
                u = (v[:, :, :54] * jw[None, :, None]).sum(1) + chosen * _pattern(3 + 2 * j, self.salt, dev, f)
            elif v.shape[1] == 54:                                      # Klop talon, discards
                u = v
            else:                                                       # king / decl one-hot [B,4]
                idx = (v * torch.arange(1, 5, device=dev).to(f)).sum(1, keepdim=True)
                u = idx * _pattern(3 + 2 * j, self.salt, dev, f)
            y = y + (j + 1) * u
        return torch.remainder(y, self.m).to(dt)


class Roka(nn.Module):
    """Vrednotenje_roke: hand [B,54] -> [B,18] bid values."""

    def __init__(self, salt, m):
        super().__init__()
        self.salt, self.m = salt, m

    def forward(self, x):
        dt, dev, f = x.dtype, x.device, _f(x)
        c, b = torch.arange(54, device=dev)[:, None], torch.arange(18, device=dev)[None, :]
        a = ((c * (2 * b + 1 + self.salt) + self.salt) % 5).to(f)
        y = (x.to(f)[:, :, None] * a[None]).sum(1) + (self.salt * b.to(f)) % 3
        return torch.remainder(y, self.m).to(dt)


class Zalaganje(nn.Module):
    """Zalaganje: [hand (B,54), talon (B,54,6) card x group, game (B,15)] -> [B,60] (54 card values, 6 group values)."""

    def __init__(self, salt, m):
        super().__init__()
        self.salt, self.m = salt, m

    def forward(self, x):
        hand, talon, game = x
        dt, dev, f = hand.dtype, hand.device, _f(hand)
        hand, talon, game = hand.to(f), talon.to(f), game.to(f)
        gi = (game * torch.arange(1, 16, device=dev).to(f)).sum(1, keepdim=True)
        gw = torch.arange(6, device=dev)
        cards = hand * (self.salt + 2) + (talon * (3 * (gw + 1)).to(f)).sum(2) + gi * _pattern(5 + self.salt, self.salt, dev, f)
        cw = ((torch.arange(54, device=dev)[:, None] * (gw[None, :] + self.salt + 1)) % 5).to(f)
        groups = (talon * cw[None]).sum(1) + gi * ((gw * 3 + self.salt) % 4).to(f)
        return torch.remainder(torch.cat([cards, groups], dim=1), self.m).to(dt)


def nets(player):
    """The six stand-in networks of one player (salt and modulus from ``player``), keyed like ``ustvari_mreze``."""
    salt, m = 3 * player + 1, MODULI[player]
    play = {name: Igra(salt + kind, m) for kind, name in enumerate(("Klop", "Navadna_igra", "Solo", "Berac"))}
    return dict(play, Vrednotenje_roke=Roka(salt, m), Zalaganje=Zalaganje(salt, m))


def host(module, x):
    """Run ``module`` on CPU in float64 on 0/1 numpy arrays (one array, or a list); returns float64 numpy, checked to be
    integers in [-256, 256], which bf16 holds exactly."""
    with torch.no_grad():
        if isinstance(x, (list, tuple)):
            y = module([torch.from_numpy(np.ascontiguousarray(a)).to(torch.float64) for a in x])
        else:
            y = module(torch.from_numpy(np.ascontiguousarray(x)).to(torch.float64))
    y = y.numpy()
    assert (y == np.round(y)).all() and (np.abs(y) <= 256).all()
    return y
