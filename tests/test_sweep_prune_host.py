"""Host side of candidate pruning (BinSweep.candidates(prune=True)), no GPU needed: the widening / narrowing tables
the kernels use equal a hand-written list for all three lattices; oracle/sweep_prune.py equals a brute-force
per-entry loop on small random tables; the three pruning entry points refuse bad arguments before any CUDA call."""
import itertools

import numpy as np
import pytest

from nanomotif_b200 import _lib
from nanomotif_b200.sweep import prune_lattice
from oracle import sweep_prune as P

# one cover step up from each letter (the widenings); narrowings are the inverse
WIDEN_IUPAC = {"A": "RWM", "T": "YWK", "G": "RSK", "C": "YSM", "R": "DV", "Y": "BH", "S": "BV", "W": "DH", "K": "BD",
               "M": "HV", "B": "N", "D": "N", "H": "N", "V": "N", "N": ""}
WIDEN_BIP_ACGT = {"A": "*", "T": "*", "G": "*", "C": "*", "*": ""}
WIDEN_BIP_IUPAC = {**{x: y.replace("N", "*") for x, y in WIDEN_IUPAC.items() if x != "N"}, "*": ""}
STATES = "ATGC"  # state order; "other" is state 4
MEMBERS = {"A": "A", "T": "T", "G": "G", "C": "C", "R": "AG", "Y": "CT", "S": "GC", "W": "AT", "K": "GT", "M": "AC",
           "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGTo", "*": "ACGT"}
LATTICES = {  # name -> (letters in table order, hand-written widenings, oracle lattice)
    "contiguous": ("ATGCRYSWKMBDHVN", WIDEN_IUPAC, P.SWEEP_LATTICE),
    "bipartite_acgt": ("ATGC*", WIDEN_BIP_ACGT, P.BIP_ACGT_LATTICE),
    "bipartite_iupac": ("ATGCRYSWKMBDHV*", WIDEN_BIP_IUPAC, P.BIP_IUPAC_LATTICE),
}


def _narrow(widen):
    return {x: "".join(sorted(y for y, up in widen.items() if x in up)) for x in widen}


@pytest.mark.parametrize("name", list(LATTICES))
def test_kernel_lattices_equal_hand_written(name):
    letters, widen, oracle_lattice = LATTICES[name]
    states, up, down = prune_lattice(name)
    assert len(states) == len(letters) == len(oracle_lattice)
    narrow = _narrow(widen)
    for i, ch in enumerate(letters):
        want_states = sum(1 << (STATES + "o").index(s) for s in MEMBERS[ch])
        assert int(states[i]) == want_states, ch
        assert {letters[j] for j in range(len(letters)) if up[i] >> j & 1} == set(widen[ch]), ch
        assert {letters[j] for j in range(len(letters)) if down[i] >> j & 1} == set(narrow[ch]), ch
    # the oracle derives the same covers from its letter sets
    o_widen, o_narrow = P.lattice_covers(oracle_lattice)
    for i, ch in enumerate(letters):
        assert {letters[j] for j in o_widen[i]} == set(widen[ch]), ch
        assert {letters[j] for j in o_narrow[i]} == set(narrow[ch]), ch
        assert oracle_lattice[i] == {"other" if s == "o" else s for s in MEMBERS[ch]}, ch
    with pytest.raises(KeyError):
        prune_lattice("gapped")


def _random_tables(rng, letters, n_axes, n_states):
    """n_mod / n_nomod over n_axes letter axes: random concrete counts with a methylated context planted (state 2 on
    axis 0 and state 0 on axis 1, unless that is too few axes), summed over each letter's states."""
    shape = (n_states,) * n_axes
    mod = rng.poisson(1.0, shape)
    nomod = rng.poisson(12.0, shape)
    planted = (slice(2, 3), slice(0, 1)) if n_axes >= 2 else (slice(2, 3),)
    mod[planted] = rng.poisson(30.0, mod[planted].shape)
    nomod[planted] = rng.poisson(1.0, nomod[planted].shape)
    # a half-methylated context: state 1 on the last axis is methylated only under state 3 on axis 0
    sel = (slice(3, 4),) + (slice(None),) * (n_axes - 2) + (slice(1, 2),)
    mod[sel] = rng.poisson(25.0, mod[sel].shape)
    nomod[sel] = rng.poisson(2.0, nomod[sel].shape)
    expand = np.array([[int(s in MEMBERS[ch]) for s in (STATES + "o")[:n_states]] for ch in letters])
    out = []
    for t in (mod, nomod):
        for ax in range(n_axes):
            t = np.moveaxis(np.tensordot(expand, t, axes=([1], [ax])), 0, ax)
        out.append(t.reshape(-1))
    return out


def _brute_force(n_mod, n_nomod, letters, widen, n_axes, min_mean, min_mod):
    """Per-entry restatement of the rule, from the hand-written widenings; also counts the (a) and (b) prunes."""
    narrow = _narrow(widen)
    n_l = len(letters)
    mean = lambda a, b: (5.0 + a) / (10.0 + a + b)
    passes = lambda i: n_mod[i] >= min_mod and mean(n_mod[i], n_nomod[i]) >= min_mean
    keep = np.zeros(n_mod.size, dtype=bool)
    reasons = {"a": 0, "b": 0}
    for i in range(n_mod.size):
        if not passes(i):
            continue
        digits = [(i // n_l ** (n_axes - 1 - ax)) % n_l for ax in range(n_axes)]
        why = None
        for ax, d in enumerate(digits):
            at = n_l ** (n_axes - 1 - ax)
            for ch in widen[letters[d]]:
                j = i + (letters.index(ch) - d) * at
                if passes(j) and mean(n_mod[j] - n_mod[i], n_nomod[j] - n_nomod[i]) >= min_mean:
                    why = why or "a"
            for ch in narrow[letters[d]]:
                j = i + (letters.index(ch) - d) * at
                if passes(j) and mean(n_mod[i] - n_mod[j], n_nomod[i] - n_nomod[j]) < min_mean:
                    why = why or "b"
        if why:
            reasons[why] += 1
        else:
            keep[i] = True
    return keep, reasons


@pytest.mark.parametrize("name,n_axes,n_states", [("contiguous", 3, 5), ("bipartite_acgt", 5, 4),
                                                  ("bipartite_iupac", 5, 4)])
def test_oracle_equals_brute_force(name, n_axes, n_states):
    """k = 4 contiguous (3 table axes besides the modified letter) and (3, g, 3) bipartite (5 half letters)."""
    letters, widen, lattice = LATTICES[name]
    rng = np.random.default_rng({"contiguous": 41, "bipartite_acgt": 42, "bipartite_iupac": 43}[name])
    n_mod, n_nomod = _random_tables(rng, letters, n_axes, n_states)
    assert n_mod.size == len(letters) ** n_axes
    for min_mean, min_mod in ((0.7, 5), (0.6, 20)):
        got = P.sweep_prune(n_mod, n_nomod, lattice, min_mean, min_mod)
        want, reasons = _brute_force(n_mod, n_nomod, letters, widen, n_axes, min_mean, min_mod)
        np.testing.assert_array_equal(got, want)
        assert want.sum() > 0 and reasons["a"] > 0
        if name != "bipartite_acgt":  # ACGT halves have no narrowing
            assert reasons["b"] > 0
        # shaped tables give the same mask
        shaped = P.sweep_prune(n_mod.reshape((len(letters),) * n_axes), n_nomod.reshape((len(letters),) * n_axes),
                               lattice, min_mean, min_mod)
        np.testing.assert_array_equal(shaped.reshape(-1), got)
    with pytest.raises(ValueError):
        P.sweep_prune(n_mod[:-1], n_nomod[:-1], lattice, 0.7, 5)


def test_filters_refuse_bad_arguments_with_and_without_prune():
    lib = _lib.lib
    buf = np.zeros(16, dtype=np.uint32)
    p = buf.ctypes.data
    n_out = np.zeros(1, dtype=np.int64).ctypes.data

    f = lib.nmb_sweep_expand_filter
    g = lib.nmb_sweep_bipartite_filter
    h = lib.nmb_sweep_bip_iupac_expand_filter
    for prune in (0, 1):
        def contiguous(nm=p, nu=p, slots=1, inner=15 ** 3, k=5, mp=1, min_mod=5, prune=prune, out=p, cap=10, n=n_out):
            return f(nm, nu, slots, inner, k, mp, 0.7, min_mod, prune, out, cap, n, None)

        for kw in ({"out": None}, {"n": None}, {"nm": None}, {"nu": None}, {"slots": -1}, {"min_mod": -1}, {"cap": -1},
                   {"k": 3, "inner": 15 ** 1}, {"k": 9, "inner": 15 ** 7}, {"mp": 5}, {"mp": -1},
                   {"inner": 15 ** 2}, {"inner": 15 ** 4}, {"inner": 15 ** 9}, {"inner": 0}, {"prune": 2}):
            assert contiguous(**kw) == -1, (prune, kw)
            assert b"nmb_sweep_expand_filter" in lib.nmb_last_error(), (prune, kw)
        assert contiguous(out=None) == -1 and b"null output" in lib.nmb_last_error()
        assert contiguous(inner=15 ** 9) == -1 and b"15^(k-2)" in lib.nmb_last_error()  # table index past 32 bits

        def bipartite(hist=p, slots=1, canon=0, min_mod=5, prune=prune, out=p, cap=10, n=n_out):
            return g(hist, slots, canon, 0.7, min_mod, prune, out, cap, n, None)

        for kw in ({"out": None}, {"n": None}, {"hist": None}, {"slots": -1}, {"canon": 4}, {"canon": -1},
                   {"min_mod": -1}, {"cap": -1}, {"prune": 2}):
            assert bipartite(**kw) == -1, (prune, kw)
            assert b"nmb_sweep_bipartite_filter" in lib.nmb_last_error(), (prune, kw)
        assert bipartite(out=None) == -1 and b"null output" in lib.nmb_last_error()

        def iupac(nm=p, nu=p, slots=1, inner=14 ** 4, min_mod=5, prune=prune, out=p, cap=10, n=n_out):
            return h(nm, nu, slots, inner, 0.7, min_mod, prune, out, cap, n, None)

        for kw in ({"out": None}, {"n": None}, {"nm": None}, {"nu": None}, {"slots": -1}, {"min_mod": -1}, {"cap": -1},
                   {"inner": 0}, {"inner": 15}, {"inner": 14 ** 3 + 1}, {"inner": 14 ** 9}, {"prune": 2}):
            assert iupac(**kw) == -1, (prune, kw)
            assert b"nmb_sweep_bip_iupac_expand_filter" in lib.nmb_last_error(), (prune, kw)
        assert iupac(out=None) == -1 and b"null output" in lib.nmb_last_error()
        assert iupac(inner=14 ** 9) == -1 and b"bad argument" in lib.nmb_last_error()  # table index past 32 bits
        assert iupac(inner=15) == -1 and b"power of 14" in lib.nmb_last_error()
    arrays = [np.zeros(15, dtype=np.uint32) for _ in range(3)]
    assert lib.nmb_sweep_prune_lattice(3, *(a.ctypes.data for a in arrays)) == -1
    assert lib.nmb_sweep_prune_lattice(0, None, arrays[1].ctypes.data, arrays[2].ctypes.data) == -1
    assert lib.nmb_sweep_prune_lattice(0, *(a.ctypes.data for a in arrays)) == 15
