"""The 32-bit talon-order decode of k_setup_synth against the 64-bit one it replaced, and (GPU) the setup state and the hand
slots of a random chain against the oracle / the eager-mask chain.

order_from_lehmer (tarok_kernels.cuh) maps the deal's Lehmer draw L < 720 and the talon bitboard to the ordered talon.  The
CPU test restates both the old decode (six ffs on the 64-bit talon, a Lehmer decode with 64-bit shifts on a 36-bit packed
list) and the new one (digits by constant multiplies, ranks as 4-bit fields of one 32-bit word, ids one per byte, a byte
permute with the rank nibbles as selectors) and checks them equal for every L over random talons."""
import numpy as np
import pytest

ALL54 = (1 << 54) - 1
M32 = 0xFFFFFFFF


def order_old(talon, L):
    rem = 0
    for i in range(6):
        c = (talon & -talon).bit_length() - 1
        talon &= talon - 1
        rem |= c << (6 * i)
    order = 0
    for i, f in enumerate((120, 24, 6, 2, 1, 1)):
        d = L // f
        L -= d * f
        sh = 6 * d
        order |= ((rem >> sh) & 63) << (6 * i)
        rem = (rem & ((1 << sh) - 1)) | ((rem >> (sh + 6)) << sh)
    return order


def byte_perm(a, b, s):
    """__byte_perm without the sign-replicate mode (selector nibbles < 8)."""
    src = (a | (b << 32)).to_bytes(8, "little")
    return sum(src[(s >> (4 * k)) & 7] << (8 * k) for k in range(4))


def order_new(talon, L):
    d0 = (L * 1093) >> 17; r1 = L - 120 * d0
    d1 = (r1 * 2731) >> 16; r2 = r1 - 24 * d1
    d2 = (r2 * 43) >> 8; r3 = r2 - 6 * d2
    d3, d4 = r3 >> 1, r3 & 1
    rank, perm = 0x543210, 0
    for i, d in enumerate((d0, d1, d2, d3, d4)):
        sh = 4 * d
        perm |= ((rank >> sh) & 15) << (4 * i)
        high = (M32 << sh) & M32
        rank = (rank & ~high & M32) | ((rank >> 4) & high)
    perm |= rank << 20
    lo, hi, a, b = talon & M32, talon >> 32, 0, 0
    for i in range(6):
        inlo = lo != 0
        w = lo if inlo else hi
        c = (w & -w).bit_length() - 1 + (0 if inlo else 32)
        if i < 4:
            a |= c << (8 * i)
        else:
            b |= c << (8 * (i - 4))
        if inlo:
            lo &= lo - 1
        else:
            hi &= hi - 1
    x, y = byte_perm(a, b, perm & 0xFFFF), byte_perm(a, b, perm >> 16)
    olo = (x & 0x3F) | ((x >> 2) & 0xFC0) | ((x >> 4) & 0x3F000) | ((x >> 6) & 0xFC0000)
    ohi = (y & 0x3F) | ((y >> 2) & 0xFC0)
    return olo | (ohi << 24)


def test_digit_multiplies_are_exact():
    assert all((L * 1093) >> 17 == L // 120 for L in range(720))
    assert all((r * 2731) >> 16 == r // 24 for r in range(120))
    assert all((r * 43) >> 8 == r // 6 for r in range(24))


def talons(rng, count):
    out = [0x3F, 0x3F << 48, (7 << 29) | (7 << 32), (1 << 31) | (31 << 49)]      # all low, all high, straddling the halves
    for _ in range(count - len(out)):
        out.append(sum(1 << int(c) for c in rng.choice(54, 6, replace=False)))
    return out


def test_talon_order_32bit_equals_64bit_for_every_lehmer_index():
    rng = np.random.default_rng(2026)
    for t in talons(rng, 40):
        assert bin(t).count("1") == 6 and t & ~ALL54 == 0
        ids = sorted(i for i in range(54) if t >> i & 1)
        seen = set()
        for L in range(720):
            o = order_old(t, L)
            assert order_new(t, L) == o, (hex(t), L)
            seen.add(o)
            assert sorted((o >> (6 * i)) & 63 for i in range(6)) == ids
        assert len(seen) == 720                                  # a bijection onto the talon's permutations


# ---- GPU ------------------------------------------------------------------------------------------------------------------
SETUP_MODES = list(range(10)) + [16, 17, 18]


def u64(t):
    return t.cpu().numpy().view(np.uint64)


def _bits(ids):
    """[n, k] card ids -> [n] uint64 bitboards."""
    return np.bitwise_or.reduce(np.left_shift(np.uint64(1), ids.astype(np.uint64)), axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1 << 20, 1000, 4097])
def test_setup_synth_state_equals_the_oracle(n):
    """k_setup_synth (deal with the 32-bit talon-order decode, contract, exchange with the table-finished discard picks)
    against the C oracle's deals, contracts, groups and discards, every synthetic mode, full and ragged batch sizes."""
    import tarok_b200.env as E
    from oracle import oracle as O

    seed, gid0 = 4242, 9
    env = E.TarokEnv(n, seed=seed, history=True)
    try:
        for mode in SETUP_MODES:
            env.setup_synth(mode, gid0)
            ref = O.rollout(seed, gid0, n, mode)
            perm = ref["perm"]
            h0 = u64(env.hands0)[:, :n]
            for s in range(4):
                np.testing.assert_array_equal(h0[s], _bits(perm[:, 12 * s:12 * s + 12]), err_msg="mode %d hand %d" % (mode, s))
            order = sum(perm[:, 48 + i].astype(np.uint64) << np.uint64(6 * i) for i in range(6))
            np.testing.assert_array_equal(u64(env.talon_order)[:n], order, err_msg="mode %d talon order" % mode)
            m = u64(env.meta)[:n]
            f = lambda sh, b: ((m >> np.uint64(sh)) & np.uint64((1 << b) - 1)).astype(np.int64)
            err = f(E.M_ERR, 1)
            np.testing.assert_array_equal(ref["err"], err, err_msg="mode %d error games" % mode)
            ok = err == 0
            for k, sh, b in (("contract", E.M_CONTRACT, 4), ("declarer", E.M_DECL, 2), ("king", E.M_KING, 3)):
                np.testing.assert_array_equal(ref[k][ok], f(sh, b)[ok], err_msg="mode %d %s" % (mode, k))
            exch = ok & (ref["group"] != 0xFF)
            np.testing.assert_array_equal(ref["group"][exch], f(E.M_GROUP, 3)[exch], err_msg="mode %d group" % mode)
            np.testing.assert_array_equal(ref["discard"][exch], u64(env.discard)[:n][exch], err_msg="mode %d discard" % mode)
    finally:
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [16, 17])
def test_hand_slots_after_every_launch_of_a_chain(mode):
    """The trick-closing launch re-seats the four hand slots to the trick's winner.  A chain of t random steps (interior
    launches without masks) leaves, for every t = 1..48, the same hand slots, meta and masks as t single launches with eager
    masks."""
    import tarok_b200.env as E

    n, seed = 40000, 31
    a, b = E.TarokEnv(n, seed=seed), E.TarokEnv(n, seed=seed)
    b.set_lazy_mask(False)
    try:
        b.setup_synth(mode, 0)
        for t in range(1, 49):
            b.step_random(1)
            a.setup_synth(mode, 0)
            a.step_random(t)
            for fld in ("hand_slots", "meta", "mask"):
                assert (u64(getattr(a, fld)) == u64(getattr(b, fld))).all(), (t, fld)
    finally:
        a.close(); b.close()
