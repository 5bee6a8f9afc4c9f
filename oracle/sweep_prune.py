"""K8 candidate pruning restated in numpy (BinSweep.candidates(prune=True)): a candidate M is dropped when a one-letter
neighbour in the same table shows it is a redundant specialisation or a mixture.  Not a reference feature:
nanomotif's own answer is bin-motifs.tsv, the motifs themselves rather than every longer motif that contains one.
Checker only; nothing under nanomotif_b200/ imports it."""
from __future__ import annotations

import math

import numpy as np

from .restate import _IUPAC_MEMBERS, IUPAC_ORDER

# Letters as sets of letter states, in table order.  Contiguous k-mers: the 15 IUPAC letters over A T G C and
# "other" (the regex wildcard N also matches non-ACGT letters).  Bipartite halves: ACGT with the pseudo-letter
# * = {A, C, G, T} (never a row), or the 14 IUPAC letters other than N with *.
SWEEP_LATTICE = tuple(frozenset(_IUPAC_MEMBERS[ch]) | (frozenset({"other"}) if ch == "N" else frozenset())
                      for ch in IUPAC_ORDER)
BIP_ACGT_LATTICE = tuple(frozenset(s) for s in ("A", "T", "G", "C", "ACGT"))
BIP_IUPAC_LATTICE = tuple(frozenset(_IUPAC_MEMBERS[ch]) for ch in IUPAC_ORDER[:-1]) + (frozenset("ACGT"),)


def lattice_covers(lattice) -> tuple[list[list[int]], list[list[int]]]:
    """(widen, narrow): widen[i] = the letters j whose set is a smallest strict superset of letter i's in the
    lattice (one more base; N also takes "other"), narrow[j] the inverse."""
    sets = [frozenset(s) for s in lattice]
    n = len(sets)
    widen, narrow = [[] for _ in range(n)], [[] for _ in range(n)]
    for i in range(n):
        for j in range(n):
            if sets[i] < sets[j] and not any(sets[i] < sets[l] < sets[j] for l in range(n)):
                widen[i].append(j)
                narrow[j].append(i)
    return widen, narrow


def sweep_prune(n_mod, n_nomod, lattice, min_mean: float, min_mod: int) -> np.ndarray:
    """Boolean mask over full tables (every axis indexed by the letters of `lattice`; a flat table of len(lattice)^n
    entries is read as n axes, first most significant): True where the entry M passes the sweep filter (n_mod >=
    min_mod and (5 + n_mod) / (10 + n_mod + n_nomod) >= min_mean) and is not pruned.  The modified letter is not an
    axis of these tables, so it is never widened or narrowed.  On every axis, for each neighbour P that widens M's
    letter there by one cover step, Q = P - M; for each C that narrows it, Q = M - C (n_mod and n_nomod separately).
    M is pruned when (a) some widening P passes and mean(Q) >= min_mean, or (b) some narrowing C passes and
    mean(Q) < min_mean.  Neighbours need not be rows themselves (a flanking N, the pseudo-letter *)."""
    m = np.asarray(n_mod).astype(np.int64)
    u = np.asarray(n_nomod).astype(np.int64)
    n_letters = len(lattice)
    shape = m.shape
    n_axes = m.ndim
    if m.ndim == 1:
        n_axes = int(round(math.log(m.size) / math.log(n_letters))) if m.size > 1 else 0
        if n_letters ** n_axes != m.size:
            raise ValueError(f"{m.size} entries are not a power of {n_letters}")
        m, u = m.reshape((n_letters,) * n_axes), u.reshape((n_letters,) * n_axes)

    def mean(q_mod, q_nomod):
        return (5.0 + q_mod) / (10.0 + q_mod + q_nomod)

    passes = (m >= min_mod) & (mean(m, u) >= min_mean)
    pruned = np.zeros(m.shape, dtype=bool)
    widen, narrow = lattice_covers(lattice)
    for ax in range(n_axes):
        mv, uv, pv, out = (np.moveaxis(x, ax, 0) for x in (m, u, passes, pruned))
        for i in range(n_letters):
            hit = np.zeros(mv.shape[1:], dtype=bool)
            for j in widen[i]:
                hit |= pv[j] & (mean(mv[j] - mv[i], uv[j] - uv[i]) >= min_mean)
            for j in narrow[i]:
                hit |= pv[j] & (mean(mv[i] - mv[j], uv[i] - uv[j]) < min_mean)
            out[i] |= hit
    return (passes & ~pruned).reshape(shape)
