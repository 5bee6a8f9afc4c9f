"""Exhaustive candidate sweep (K8, BASELINE.json configs[4]): the (n_mod, n_nomod) counts that motif_model_bin
(nanomotif/find_motifs_bin.py:1265-1331) would return for EVERY IUPAC motif of length 4..8 and every modified
position, from one histogram pass over the assembly plus a subset-sum transform -- not one scan per motif.

    index = SweepIndex(assembly, pileup, modtype_index)            # one pass: window x offset x class histograms
    index.add(contig_begin, contig_end)                            # a bin, or everything
    n_mod, n_nomod = index.table(k, mod_pos, canonical="A")        # device uint32 [15^(k-1)]: all motifs of length k
    index.counts("GRNGAAGY", 5)                                    # one motif's counts (table lookup)
    index.candidates(k, mod_pos, "A", min_mean=0.7, min_mod=50)    # motifs above a posterior-mean / support bar

The same per bin, for all bins of a MultiBinScorer at once (one histogram launch for all of them):

    sw = BinSweep(scorer, "a")                                     # per-bin histograms, IUPAC + bipartite
    sw.counts("bin_3", "GRNGAAGY", 5)                              # == scorer.context("bin_3", "a").score(...)
    sw.index("bin_3")                                              # SweepIndex over that bin's histograms
    sw.candidates(min_mean=0.7, min_mod=50)                        # pandas frame: every bin's candidates
    sw.candidates(bipartite_letters="IUPAC")                       # bipartite halves over every IUPAC letter but N
    sw.candidates(prune=True)                                      # minus specialisations and mixtures (GATC, not GATCA)
    sw.bipartite_iupac_counts("bin_3", "GAA", 6, "RTCG", 2)        # GAANNNNNNRTCG, modified A at position 2
    sw.count_matrix(["GATC", "CCWGG", "GAANNNNNNRTCG"], [1, 1, 2])  # (n_mod, n_nomod) [bin][motif], one gather launch

Letters of a motif are indexed in the order of nanomotif/constants.py:2 (A T G C R Y S W K M B D H V N); the
modified position's own letter is fixed to the concrete canonical base and left out of the table index (a pileup
row of mod type 'a' only exists under an A, so every other letter there gives zero or a duplicate).
"""
from __future__ import annotations

import ctypes as C
import re

import numpy as np
import torch

from . import _lib
from ._lib import check, lib, ptr
from .device import DeviceAssembly, DevicePileup, _stream

IUPAC_ORDER = "ATGCRYSWKMBDHVN"
BIP_LETTERS = IUPAC_ORDER[:-1]  # letters of the halves of degenerate bipartite motifs: every IUPAC letter but N
_BASE_DIGIT = {"A": 0, "T": 1, "G": 2, "C": 3}
MIN_K, MAX_K = 4, 8


def hist_offset(k: int) -> int:
    return sum(j * 2 * 5 ** j for j in range(MIN_K, k))


def _class_records(pileup: DevicePileup, asm: DeviceAssembly, modtype: int) -> int:
    """Device address of the class records of one mod type (the pileup stacks them per mod type)."""
    return ptr(pileup.class_records) + modtype * asm.n_tiles * _lib.CLS_REC_WORDS * 4


def _slice(hist: torch.Tensor, n_slots: int, k: int, mod_pos: int, cls: int, canonical: str) -> torch.Tensor:
    """[n_slots][5^(k-1)]: the class-`cls` counters of the (k, mod_pos) block of the finished histograms stacked at
    HIST_SIZE from `hist` on, with the modified letter fixed to `canonical` (nmb_sweep_slice)."""
    n = 5 ** (k - 1)
    t = torch.empty(n_slots * n, dtype=torch.int32, device=hist.device)
    src = hist[hist_offset(k) + (mod_pos * 2 + cls) * 5 ** k:]
    check(lib.nmb_sweep_slice(ptr(src), HIST_SIZE, n_slots, ptr(t), n, 5 ** (k - 1 - mod_pos), _BASE_DIGIT[canonical],
                              _stream()), "nmb_sweep_slice")
    return t


def _bip_iupac_slice(bip: torch.Tensor, n_slots: int, a: int, g: int, b: int, mod_pos: int, cls: int,
                     canonical: str) -> torch.Tensor:
    """[n_slots][4^(a+b-1)]: the class-`cls` counters of shape (a, g, b) of the finished bipartite histograms stacked
    at BIP_SIZE from `bip` on, with the modified letter fixed to `canonical` (nmb_sweep_bip_iupac_slice)."""
    t = torch.empty(n_slots * 4 ** (a + b - 1), dtype=torch.int32, device=bip.device)
    check(lib.nmb_sweep_bip_iupac_slice(ptr(bip), n_slots, a, g, b, mod_pos, cls, _BASE_DIGIT[canonical], ptr(t),
                                        _stream()), "nmb_sweep_bip_iupac_slice")
    return t


def _expand(tables, states: int, steps: int) -> tuple:
    """Expands the last `steps` axes of each sliced class table, last axis first (the large final passes then run
    with a long contiguous inner): states = 5 gives the 15 IUPAC letters (nmb_sweep_expand), states = 4 the 14
    letters other than N (nmb_sweep_bip_iupac_expand)."""
    letters, fn = (15, lib.nmb_sweep_expand) if states == 5 else (14, lib.nmb_sweep_bip_iupac_expand)
    out = []
    for t in tables:
        for step in range(steps):
            inner = letters ** step
            outer = t.numel() // (states * inner)
            e = torch.empty(outer * letters * inner, dtype=torch.int32, device=t.device)
            check(fn(ptr(t), ptr(e), outer, inner, _stream()), fn.__name__)
            t = e
        out.append(t)
    return tuple(out)


class SweepIndex:
    """Window histograms of one mod type (nmb_sweep_hist), accumulated over the contig ranges added so far."""

    def __init__(self, assembly: DeviceAssembly, pileup: DevicePileup, modtype_index: int = 0):
        self.asm, self.pileup, self.modtype = assembly, pileup, int(modtype_index)
        if not 0 <= self.modtype < pileup.n_modtypes:
            raise ValueError("mod type index outside the pileup's class records")
        with torch.cuda.device(assembly.device):
            # RAW histogram (nmb_sweep_hist): k = 8 counted row by row, k < 8 only the contig-end windows; raw
            # histograms add (more contig ranges, other GPUs).  `hist` is the finalized copy, made on demand.
            self.raw = torch.zeros(int(lib.nmb_sweep_hist_size()), dtype=torch.int32, device=assembly.device)
        self._hist = None
        self.bip_raw = None
        self._bip = None
        self._tables: dict = {}

    @property
    def hist(self) -> torch.Tensor:
        """The finished histogram of every k = 4..8 (nmb_sweep_finalize applied to a copy of the raw one)."""
        if self._hist is None:
            with torch.cuda.device(self.asm.device):
                h = self.raw.clone()
                check(lib.nmb_sweep_finalize(ptr(h), 1, _stream()), "nmb_sweep_finalize")
            self._hist = h
        return self._hist

    def add(self, contig_begin: int = 0, contig_end: int | None = None) -> "SweepIndex":
        asm = self.asm
        contig_end = asm.n_contigs if contig_end is None else contig_end
        tile_begin, tile_count = asm.tile_span(contig_begin, contig_end)
        view = asm.view()
        with torch.cuda.device(asm.device):
            check(lib.nmb_sweep_hist(C.byref(view), _class_records(self.pileup, asm, self.modtype), tile_begin,
                                     tile_count, contig_begin, contig_end, None, 1, ptr(self.raw), _stream()),
                  "nmb_sweep_hist")
        self._tables.clear()
        self._hist = None
        return self

    # ---- bipartite shapes X{3,4} N{4..8} Y{3,4} over ACGT ----
    def add_bipartite(self, contig_begin: int = 0, contig_end: int | None = None) -> "SweepIndex":
        asm = self.asm
        contig_end = asm.n_contigs if contig_end is None else contig_end
        tile_begin, tile_count = asm.tile_span(contig_begin, contig_end)
        view = asm.view()
        with torch.cuda.device(asm.device):
            if self.bip_raw is None:
                self.bip_raw = torch.zeros(int(lib.nmb_sweep_bipartite_size()), dtype=torch.int32, device=asm.device)
            check(lib.nmb_sweep_bipartite(C.byref(view), _class_records(self.pileup, asm, self.modtype), tile_begin,
                                          tile_count, contig_begin, contig_end, None, 1, ptr(self.bip_raw), _stream()),
                  "nmb_sweep_bipartite")
        self._bip = None
        self._tables = {k: v for k, v in self._tables.items() if k[0] != "bip"}
        return self

    @classmethod
    def of_finished(cls, assembly: DeviceAssembly, pileup: DevicePileup, modtype_index: int, hist: torch.Tensor,
                    bip: torch.Tensor | None = None) -> "SweepIndex":
        """An index over histograms finished elsewhere (one bin's slice of a BinSweep): tables, counts and candidates
        read `hist` / `bip`; there is no raw histogram, so add() and all_reduce() do not apply."""
        self = cls.__new__(cls)
        self.asm, self.pileup, self.modtype = assembly, pileup, int(modtype_index)
        self.raw, self._hist, self.bip_raw, self._bip = None, hist, None, bip
        self._tables = {}
        return self

    @property
    def bip(self):
        """The finished bipartite histogram (nmb_sweep_bipartite_finalize applied to a copy of the raw one), or None."""
        if self._bip is None and self.bip_raw is not None:
            with torch.cuda.device(self.asm.device):
                h = self.bip_raw.clone()
                check(lib.nmb_sweep_bipartite_finalize(ptr(h), 1, _stream()), "nmb_sweep_bipartite_finalize")
            self._bip = h
        return self._bip

    @staticmethod
    def bipartite_block(a: int, g: int, b: int) -> tuple[int, int]:
        """(first counter, counters per (offset, class)) of shape X{a} N{g} Y{b} in the bipartite histogram."""
        if a not in (3, 4) or b not in (3, 4) or not 4 <= g <= 8:
            raise ValueError("bipartite shapes are X{3,4} N{4..8} Y{3,4}")
        block = lambda x, y: (x + y) * 2 * 4 ** (x + y)
        per_gap = block(3, 3) + block(3, 4) + block(4, 3) + block(4, 4)
        within = {(3, 3): 0, (3, 4): block(3, 3), (4, 3): block(3, 3) + block(3, 4),
                  (4, 4): block(3, 3) + block(3, 4) + block(4, 3)}[(a, b)]
        return (g - 4) * per_gap + within, 4 ** (a + b)

    def bipartite_table(self, a: int, g: int, b: int, mod_pos: int):
        """(n_mod, n_nomod) device views over all 4^(a+b) motifs of shape X{a} N{g} Y{b} with the modified base at
        motif position mod_pos (inside X or Y).  Entry index: bipartite_index(left, right)."""
        if a <= mod_pos < a + g or not 0 <= mod_pos < a + g + b:
            raise ValueError("the modified position must lie in one of the two concrete parts")
        o = mod_pos if mod_pos < a else mod_pos - g
        first, n = self.bipartite_block(a, g, b)
        base = first + o * 2 * n
        return self.bip[base:base + n], self.bip[base + n:base + 2 * n]

    @staticmethod
    def bipartite_index(left: str, right: str) -> int:
        a, b = len(left), len(right)
        x = lambda part: sum((_BASE_DIGIT[c] >> 1) << i for i, c in enumerate(part))
        y = lambda part: sum((_BASE_DIGIT[c] & 1) << i for i, c in enumerate(part))
        return x(left) | (y(left) << a) | (x(right) << (2 * a)) | (y(right) << (2 * a + b))

    def bipartite_counts(self, left: str, gap: int, right: str, mod_pos: int) -> tuple[int, int]:
        """(n_mod, n_nomod) of the motif left + N*gap + right with the modified base at mod_pos."""
        n_mod, n_nomod = self.bipartite_table(len(left), gap, len(right), mod_pos)
        i = self.bipartite_index(left, right)
        return int(n_mod[i].item()) & 0xFFFFFFFF, int(n_nomod[i].item()) & 0xFFFFFFFF

    # ---- degenerate bipartite motifs: the halves use the 14 IUPAC letters other than N (BIP_LETTERS) ----
    def bipartite_iupac_table(self, a: int, g: int, b: int, mod_pos: int, canonical: str = "A", keep: bool = False):
        """(n_mod, n_nomod) device views over all 14^(a+b-1) motifs of shape X{a} N{g} Y{b} whose halves use
        BIP_LETTERS, with `canonical` at motif position mod_pos (inside X or Y).  Entry index:
        bipartite_iupac_index(left, right, offset of mod_pos in left + right)."""
        self.bipartite_block(a, g, b)
        if a <= mod_pos < a + g or not 0 <= mod_pos < a + g + b:
            raise ValueError("the modified position must lie in one of the two concrete parts")
        if canonical not in _BASE_DIGIT:
            raise ValueError("the modified position must hold a concrete base")
        if self.bip is None:
            raise ValueError("no bipartite histogram: call add_bipartite() first")
        key = ("bip", a, g, b, mod_pos, canonical)
        if key in self._tables:
            return self._tables[key]
        with torch.cuda.device(self.asm.device):
            out = _expand([_bip_iupac_slice(self.bip, 1, a, g, b, mod_pos, cls, canonical) for cls in (0, 1)], 4,
                          a + b - 1)
        if keep:
            self._tables[key] = out
        return out

    @staticmethod
    def bipartite_iupac_index(left: str, right: str, offset: int) -> int:
        """Index in bipartite_iupac_table of the motif with halves left / right whose modified base is letter
        `offset` of left + right (the gap not counted): the other letters as base-14 digits (BIP_LETTERS), first
        letter most significant."""
        idx = 0
        for i, ch in enumerate(left + right):
            if i != offset:
                idx = idx * 14 + BIP_LETTERS.index(ch)
        return idx

    def bipartite_iupac_counts(self, left: str, gap: int, right: str, mod_pos: int, keep: bool = True) -> tuple[int, int]:
        """(n_mod, n_nomod) of the motif left + N*gap + right, halves over BIP_LETTERS, modified base at mod_pos."""
        if any(ch not in BIP_LETTERS for ch in left + right):
            raise ValueError(f"half letters must be among {BIP_LETTERS}")
        a = len(left)
        offset = mod_pos if mod_pos < a else mod_pos - gap
        if a <= mod_pos < a + gap or not 0 <= offset < a + len(right):
            raise ValueError("the modified position must lie in one of the two concrete parts")
        n_mod, n_nomod = self.bipartite_iupac_table(a, gap, len(right), mod_pos, (left + right)[offset], keep=keep)
        i = self.bipartite_iupac_index(left, right, offset)
        return int(n_mod[i].item()) & 0xFFFFFFFF, int(n_nomod[i].item()) & 0xFFFFFFFF

    def all_reduce(self) -> "SweepIndex":
        """Sum the histograms over the ranks of the default process group (contig-sharded assemblies)."""
        import torch.distributed as dist

        dist.all_reduce(self.raw)  # raw histograms add; the marginalisation runs once, on the sum
        if self.bip_raw is not None:
            dist.all_reduce(self.bip_raw)
        self._tables.clear()
        self._hist = self._bip = None
        return self

    def table(self, k: int, mod_pos: int, canonical: str = "A", keep: bool = False):
        """(n_mod, n_nomod): device uint32-as-int32 tensors of 15^(k-1) entries, index = the motif's letters except the
        modified position as base-15 digits (first letter most significant, IUPAC_ORDER)."""
        if not (MIN_K <= k <= MAX_K and 0 <= mod_pos < k):
            raise ValueError("k must be 4..8 and 0 <= mod_pos < k")
        key = (k, mod_pos, canonical)
        if key in self._tables:
            return self._tables[key]
        with torch.cuda.device(self.asm.device):
            out = _expand([_slice(self.hist, 1, k, mod_pos, cls, canonical) for cls in (0, 1)], 5, k - 1)
        if keep:
            self._tables[key] = out
        return out

    @staticmethod
    def motif_index(motif_iupac: str, mod_pos: int) -> int:
        idx = 0
        for i, ch in enumerate(motif_iupac):
            if i != mod_pos:
                idx = idx * 15 + IUPAC_ORDER.index(ch)
        return idx

    @staticmethod
    def index_motif(index: int, k: int, mod_pos: int, canonical: str = "A") -> str:
        letters = []
        for i in reversed(range(k)):
            if i == mod_pos:
                letters.append(canonical)
            else:
                letters.append(IUPAC_ORDER[index % 15])
                index //= 15
        return "".join(reversed(letters))

    def counts(self, motif_iupac: str, mod_pos: int, keep: bool = True) -> tuple[int, int]:
        """(n_mod, n_nomod) of one IUPAC motif of length 4..8 -- what motif_model_bin adds to the prior."""
        base = motif_iupac[mod_pos]
        if base not in _BASE_DIGIT:
            raise ValueError("the modified position must hold a concrete base")
        n_mod, n_nomod = self.table(len(motif_iupac), mod_pos, base, keep=keep)
        i = self.motif_index(motif_iupac, mod_pos)
        return int(n_mod[i].item()) & 0xFFFFFFFF, int(n_nomod[i].item()) & 0xFFFFFFFF

    def count_many(self, motifs, mod_positions) -> tuple[np.ndarray, np.ndarray]:
        """(n_mod, n_nomod): int64 arrays [len(motifs)], the exact counts of every listed motif (IUPAC 4..8-mers and
        X{3,4} N{4..8} Y{3,4} motifs with halves over BIP_LETTERS, see pack_queries) from one nmb_sweep_lookup launch;
        no table is expanded.  Every table entry equals its count mod 2^32."""
        records = _lookup_records(motifs, mod_positions, self.bip_raw is not None or self._bip is not None,
                                  "no bipartite histogram: call add_bipartite() first")
        with torch.cuda.device(self.asm.device):
            bip = self.bip if (records["kind"] == 1).any() else None
            out = _lookup(self.hist, bip, None, 1, records).cpu().numpy()
        return out[0, :, 0], out[0, :, 1]

    def candidates(self, k: int, mod_pos: int, canonical: str = "A", min_mean: float = 0.7, min_mod: int = 50,
                   canonical_form: bool = True) -> list[tuple[str, int, int]]:
        """[(motif, n_mod, n_nomod)] of length k with posterior mean >= min_mean and n_mod >= min_mod; with
        `canonical_form` motifs that start or end with N are left out (they are the shorter motif)."""
        n_mod, n_nomod = self.table(k, mod_pos, canonical)
        d = self.asm.device
        n = int(n_mod.numel())
        with torch.cuda.device(d):
            n_out = torch.zeros(1, dtype=torch.int64, device=d)
            check(lib.nmb_sweep_filter(ptr(n_mod), ptr(n_nomod), n, float(min_mean), int(min_mod), None, 0, ptr(n_out),
                                       _stream()), "nmb_sweep_filter")
            m = int(n_out.item())
            idx = torch.empty(max(m, 1), dtype=torch.int64, device=d)
            if m:
                check(lib.nmb_sweep_filter(ptr(n_mod), ptr(n_nomod), n, float(min_mean), int(min_mod), ptr(idx), m,
                                           ptr(n_out), _stream()), "nmb_sweep_filter")
            idx = idx[:m]
            a = n_mod[idx].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
            b = n_nomod[idx].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
            idx = idx.cpu().numpy()
        out = []
        for i, x, y in sorted(zip(idx.tolist(), a.tolist(), b.tolist())):
            s = self.index_motif(i, k, mod_pos, canonical)
            if canonical_form and (s[0] == "N" or s[-1] == "N"):
                continue
            out.append((s, x, y))
        return out


# ---- per-bin sweep ----
HIST_SIZE = int(lib.nmb_sweep_hist_size())  # counters of one IUPAC histogram (7 567 500)
BIP_SIZE = int(lib.nmb_sweep_bipartite_size())  # counters of one bipartite histogram (7 782 400)
_IUPAC_BYTES = np.frombuffer(IUPAC_ORDER.encode(), dtype=np.uint8)
_ACGT_BYTES = np.frombuffer(b"ATGC", dtype=np.uint8)  # letter code x << 1 | y, as in _BASE_DIGIT
_BIP_SHAPES = ((3, 3), (3, 4), (4, 3), (4, 4))  # storage order within one gap
_BIPARTITE = re.compile(r"([ACGT]{3,4})(N{4,8})([ACGT]{3,4})")


def decode_motifs(k: int, mod_pos: int, index, canonical: str = "A") -> np.ndarray:
    """Vectorised SweepIndex.index_motif: table indices of the (k, mod_pos) table -> numpy array of motif strings."""
    rest = np.asarray(index, dtype=np.int64).copy()
    letters = np.empty((rest.size, k), dtype=np.uint8)
    for i in reversed(range(k)):
        if i == mod_pos:
            letters[:, i] = ord(canonical)
        else:
            letters[:, i] = _IUPAC_BYTES[rest % 15]
            rest //= 15
    return letters.view(f"S{k}").ravel().astype(str)


def decode_bipartite(counter) -> tuple[np.ndarray, np.ndarray]:
    """Positions of n_mod counters in a bipartite histogram -> (motif strings left + "N" * gap + right, mod_position).
    Inverts SweepIndex.bipartite_block / bipartite_index."""
    counter = np.asarray(counter, dtype=np.int64)
    motifs = np.empty(counter.size, dtype=object)
    mod_pos = np.empty(counter.size, dtype=np.int64)
    per_gap = SweepIndex.bipartite_block(3, 5, 3)[0]
    gap, rem = counter // per_gap + 4, counter % per_gap
    for a, b in _BIP_SHAPES:
        first, n = SweepIndex.bipartite_block(a, 4, b)
        inside = (rem >= first) & (rem < first + (a + b) * 2 * n)
        for g in range(4, 9):
            sel = np.flatnonzero(inside & (gap == g))
            if not sel.size:
                continue
            r = rem[sel] - first
            o, code = r // (2 * n), r % n
            bits = lambda at: (code >> at) & 1
            letters = np.full((sel.size, a + g + b), ord("N"), dtype=np.uint8)
            for i in range(a):
                letters[:, i] = _ACGT_BYTES[bits(i) << 1 | bits(a + i)]
            for i in range(b):
                letters[:, a + g + i] = _ACGT_BYTES[bits(2 * a + i) << 1 | bits(2 * a + b + i)]
            motifs[sel] = letters.view(f"S{a + g + b}").ravel().astype(str)
            mod_pos[sel] = np.where(o < a, o, o + g)
    return motifs, mod_pos


def decode_bipartite_iupac(a: int, g: int, b: int, mod_pos: int, index, canonical: str = "A") -> np.ndarray:
    """Vectorised inverse of SweepIndex.bipartite_iupac_index: indices of the (a, g, b, mod_pos) table ->
    numpy array of motif strings left + "N" * g + right."""
    rest = np.asarray(index, dtype=np.int64).copy()
    offset = mod_pos if mod_pos < a else mod_pos - g
    halves = np.empty((rest.size, a + b), dtype=np.uint8)
    for i in reversed(range(a + b)):
        if i == offset:
            halves[:, i] = ord(canonical)
        else:
            halves[:, i] = _IUPAC_BYTES[rest % 14]
            rest //= 14
    letters = np.full((rest.size, a + g + b), ord("N"), dtype=np.uint8)
    letters[:, :a], letters[:, a + g:] = halves[:, :a], halves[:, a:]
    return letters.view(f"S{a + g + b}").ravel().astype(str)


PRUNE_LATTICES = {"contiguous": 0, "bipartite_acgt": 1, "bipartite_iupac": 2}


def prune_lattice(name: str) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(states, widen, narrow) of the letter lattice the pruning kernels use (nmb_sweep_prune_lattice), in table
    letter order with the widest letter (N or *) last: states[i] bit s = letter i stands for state s (A T G C other),
    widen[i] / narrow[i] bit j = letter j covers letter i / letter i covers letter j."""
    arrays = [np.zeros(15, dtype=np.uint32) for _ in range(3)]
    n = lib.nmb_sweep_prune_lattice(PRUNE_LATTICES[name], *(ptr(a) for a in arrays))
    check(n, "nmb_sweep_prune_lattice")
    return tuple(a[:n] for a in arrays)


# ---- lookup: the counts of any list of motifs, gathered from the finished histograms (nmb_sweep_lookup) ----
LOOKUP_REASONS = {
    1: "a letter outside the 15 IUPAC letters",
    2: "not a shape of the sweep tables (a 4..8-mer, or X{3,4} N{4..8} Y{3,4} without N in X and Y)",
    3: "the modified position lies outside the motif",
    4: "the modified position lies in the gap",
    5: "the modified position must hold A, C, G or T",
}
_LETTER_INDEX = np.full(256, -1, dtype=np.int64)  # byte -> IUPAC_ORDER index
_LETTER_INDEX[_IUPAC_BYTES] = np.arange(15)


def _letter_states(lattice: str, n: int) -> tuple[np.ndarray, np.ndarray]:
    """([n] number of states, [n][5] the state digits, padded with 0) of the first n letters of a prune lattice."""
    count = np.zeros(n, dtype=np.int64)
    digits = np.zeros((n, 5), dtype=np.int64)
    for i, m in enumerate(prune_lattice(lattice)[0][:n].tolist()):
        ds = [s for s in range(5) if m >> s & 1]
        count[i], digits[i, :len(ds)] = len(ds), ds
    return count, digits


_CONTIG_STATES = _letter_states("contiguous", 15)  # A T G C other; N also takes "other"
_BIP_STATES = _letter_states("bipartite_iupac", 14)  # the last letter of that lattice is the pseudo-letter *


def pack_queries(motifs, mod_positions) -> tuple[np.ndarray, np.ndarray]:
    """(records, status): one nmb_sweep_query per motif (_lib.SWEEP_QUERY_DTYPE) and int8 status, 0 when the tables
    hold the motif, else a key of LOOKUP_REASONS (its record then has kind -1, which nmb_sweep_lookup answers with -1).
    Covered: a contiguous motif of 4..8 of the 15 letters IUPAC_ORDER, or a motif of > 8 letters that fully matches
    [BIP_LETTERS]{3,4} N{4,8} [BIP_LETTERS]{3,4}; the modified position inside the motif (inside a half for bipartite
    motifs) and holding A, C, G or T -- what SweepIndex.counts and bipartite_iupac_counts accept."""
    text = np.asarray(list(motifs), dtype=str)
    mods = np.asarray(mod_positions, dtype=np.int64).reshape(-1)
    if mods.size != text.size:
        raise ValueError(f"{text.size} motifs but {mods.size} modified positions")
    n = text.size
    records = np.zeros(n, dtype=_lib.SWEEP_QUERY_DTYPE)
    records["kind"] = -1
    status = np.zeros(n, dtype=np.int8)
    lengths = np.char.str_len(text) if n else np.zeros(0, np.int64)
    for L in np.unique(lengths).tolist():
        sel = np.flatnonzero(lengths == L)
        if L < MIN_K or L == MAX_K + 1:
            status[sel] = 2
            continue
        code = text[sel].astype(f"U{L}").view(np.uint32).reshape(-1, L)
        letter = _LETTER_INDEX[np.minimum(code, 255)]
        mp = mods[sel]
        st = np.where((letter < 0).any(1), 1, 0)
        if L <= MAX_K:
            st, rec = _pack_contiguous(L, letter, mp, st)
        else:
            st, rec = _pack_bipartite(L, letter, mp, st)
        status[sel] = st
        records[sel[st == 0]] = rec
    return records, status


def _mod_status(st, letter, mp, L, in_gap):
    """Status of the modified positions of one length group whose letters and shape were checked (st)."""
    inside = (mp >= 0) & (mp < L)
    at = letter[np.arange(len(mp)), np.clip(mp, 0, L - 1)]
    st = np.where(st != 0, st, np.where(~inside, 3, np.where(in_gap, 4, np.where((at < 0) | (at > 3), 5, 0))))
    return st


def _place(records, deg, count, digits, strides, rank):
    """Fills n_states / offset of the degenerate positions (deg[:, i]) at their rank in the record."""
    for i in range(deg.shape[1]):
        rows = np.flatnonzero(deg[:, i])
        r = rank[rows, i]
        records["n_states"][rows, r] = count[rows, i]
        records["offset"][rows, r, :] = strides(i, digits[rows, i, :])
    records["n_pos"] = deg.sum(1)


def _pack_contiguous(L, letter, mp, st):
    st = _mod_status(st, letter, mp, L, np.zeros(len(mp), bool))
    ok = st == 0
    lid, mpo = letter[ok], mp[ok]
    count, digits = _CONTIG_STATES[0][lid], _CONTIG_STATES[1][lid]  # [m][L], [m][L][5]
    stride = 5 ** (L - 1 - np.arange(L))
    deg = count > 1  # the modified letter is concrete, so it goes into base
    rec = np.zeros(len(lid), dtype=_lib.SWEEP_QUERY_DTYPE)
    rec["base"] = hist_offset(L) + mpo * 2 * 5 ** L + (np.where(deg, 0, digits[..., 0]) * stride).sum(1)
    rec["class_step"] = 5 ** L
    # motif order: the last degenerate letter, the one with the smallest stride, is the least significant digit
    _place(rec, deg, count, digits, lambda i, d: d * stride[i], np.cumsum(deg, 1) - 1)
    return st, rec


def _pack_bipartite(L, letter, mp, st):
    half = (letter >= 0) & (letter < 14)  # BIP_LETTERS: IUPAC_ORDER without N (index 14)
    shape = np.full(len(mp), -1, dtype=np.int64)  # index in _BIP_SHAPES; the run of N fixes a, g and b
    for j, (a, b) in enumerate(_BIP_SHAPES):
        g = L - a - b
        if 4 <= g <= 8:
            shape[half[:, :a].all(1) & (letter[:, a:a + g] == 14).all(1) & half[:, a + g:].all(1)] = j
    st = np.where((st == 0) & (shape < 0), 2, st)
    a_of, b_of = (np.array(x)[shape] for x in zip(*_BIP_SHAPES))
    st = _mod_status(st, letter, mp, L, (mp >= a_of) & (mp < L - b_of))
    ok = np.flatnonzero(st == 0)
    rec = np.zeros(len(ok), dtype=_lib.SWEEP_QUERY_DTYPE)
    for j, (a, b) in enumerate(_BIP_SHAPES):
        at = np.flatnonzero(shape[ok] == j)
        if not at.size:
            continue
        g, rows = L - a - b, ok[at]
        halves = np.concatenate([letter[rows, :a], letter[rows, a + g:]], axis=1)  # [m][a + b]
        o = np.where(mp[rows] < a, mp[rows], mp[rows] - g)
        count, digits = _BIP_STATES[0][halves], _BIP_STATES[1][halves]
        p = np.arange(a + b)
        xbit, ybit = np.where(p < a, p, a + p), np.where(p < a, a + p, a + b + p)  # the header's window index
        bits = lambda i, d: (d >> 1) << xbit[i] | (d & 1) << ybit[i]
        deg = count > 1
        first, n = SweepIndex.bipartite_block(a, g, b)
        r = np.zeros(len(rows), dtype=_lib.SWEEP_QUERY_DTYPE)
        r["kind"] = 1
        r["base"] = first + o * 2 * n + np.where(deg, 0, bits(p, digits[..., 0])).sum(1)
        r["class_step"] = n
        # reversed motif order: the first letter of the left half, at the lowest window bits, is the least significant
        _place(r, deg, count, digits, bits, np.cumsum(deg[:, ::-1], 1)[:, ::-1] - 1)
        rec[at] = r
    return st, rec


def covers(motifs, mod_positions) -> np.ndarray:
    """bool per motif: whether the sweep tables hold it (pack_queries' status 0).  Motifs with N inside a bipartite
    half or gaps of more than 8 do not occur in the tables; filter a motif list with this before counting it."""
    return pack_queries(motifs, mod_positions)[1] == 0


def _lookup_records(motifs, mod_positions, has_bipartite: bool, missing: str) -> np.ndarray:
    """pack_queries, raising ValueError for the first uncovered motif, and `missing` when a bipartite motif is asked
    of histograms without the bipartite kind."""
    motifs, mod_positions = list(motifs), np.asarray(mod_positions).reshape(-1)
    records, status = pack_queries(motifs, mod_positions)
    bad = np.flatnonzero(status)
    if bad.size:
        i = int(bad[0])
        raise ValueError(f"motif {i} ({motifs[i]!r}, mod_position {mod_positions[i]}): {LOOKUP_REASONS[int(status[i])]}")
    if not has_bipartite and (records["kind"] == 1).any():
        raise ValueError(missing)
    return records


def _bin_rows(known, bins) -> list:
    """The rows of a count matrix: `bins`, or every bin of `known` for None; KeyError for an unknown bin."""
    rows = list(known) if bins is None else list(bins)
    for b in rows:
        if b not in known:
            raise KeyError(b)
    if len(set(rows)) != len(rows):
        raise ValueError("a bin is listed twice")
    return rows


def _lookup(hist: torch.Tensor, bip, slots, n_rows: int, records: np.ndarray) -> torch.Tensor:
    """[n_rows][len(records)][2] int64 device tensor: nmb_sweep_lookup over the stacked finished histograms."""
    d = hist.device
    out = torch.empty((n_rows, len(records), 2), dtype=torch.int64, device=d)
    if n_rows and len(records):
        q = torch.from_numpy(records.view(np.uint8)).to(d)
        check(lib.nmb_sweep_lookup(ptr(hist), ptr(bip), ptr(slots), n_rows, ptr(q), len(records), ptr(out),
                                   _stream()), "nmb_sweep_lookup")
    return out


def bip_iupac_scratch_bytes() -> int:
    """Device bytes per bin of one degenerate bipartite candidate pass (shape (4, g, 4), the largest): the largest
    expansion step's input + output, both classes (the fused last step writes no table).  16 x 14^5 + 4 x 14^6
    entries: 310 MB."""
    n = 7
    sizes = [4 ** n] + [4 ** (n - 1 - s) * 14 ** (s + 1) for s in range(n - 1)]
    return 2 * 4 * max(x + y for x, y in zip(sizes, sizes[1:]))


def table_scratch_bytes(k: int) -> int:
    """Device bytes per bin of one (k, mod_pos) candidate pass: the largest expansion step's input + output, both
    classes (the fused last step writes no table).  k = 8: 607.5 MB."""
    sizes = [5 ** (k - 1)] + [5 ** (k - 2 - s) * 15 ** (s + 1) for s in range(k - 2)]
    return 2 * 4 * max(x + y for x, y in zip(sizes, sizes[1:]))


class BinSweep:
    """The sweep of every listed bin of a MultiBinScorer for one mod type: one histogram per bin ("slot"), all of
    them filled by ONE launch over the bins' tiles (+ one for the bipartite shapes).  Answers "which motifs are
    methylated in which bin" for every IUPAC motif of length 4..8 and every bipartite X{3,4} N{4..8} Y{3,4} motif.

    Device memory per bin: 30.3 MB of raw IUPAC counters and 31.1 MB of raw bipartite ones (400 bins: 12.1 + 12.5
    GB), and the same again for the finished copies once tables or candidates are read; `bins=` sweeps a subset.
    candidates() needs `scratch_bytes` more (at least table_scratch_bytes(max k) per bin of a chunk)."""

    def __init__(self, scorer, mod_type, bins=None, bipartite: bool = True):
        from .search import CANONICAL

        self.asm, self.pileup, self.mod_type = scorer.assembly, scorer.pileup, mod_type
        self.modtype = list(scorer.mod_types).index(mod_type)
        self.canonical = CANONICAL[str(mod_type)]
        self.bins = list(scorer._ranges) if bins is None else list(bins)
        self.slot = {}
        for b in self.bins:
            if b not in scorer._ranges:
                raise KeyError(b)
            if b in self.slot:
                raise ValueError(f"bin {b!r} listed twice")
            self.slot[b] = len(self.slot)
        asm = self.asm
        contig_slot = np.full(asm.n_contigs, -1, dtype=np.int32)
        first, last = asm.n_tiles, 0
        for b, s in self.slot.items():
            lo, hi = scorer._ranges[b]
            contig_slot[lo:hi] = s
            t0, n = asm.tile_span(lo, hi)
            if n:
                first, last = min(first, t0), max(last, t0 + n)
        self.tile_begin, self.tile_count = (first, last - first) if last > first else (0, 0)
        n = len(self.bins)
        with torch.cuda.device(asm.device):
            self.contig_slot = torch.from_numpy(np.append(contig_slot, np.int32(-1))).to(asm.device)
            self.raw = torch.zeros(n * HIST_SIZE, dtype=torch.int32, device=asm.device)
            self.bip_raw = torch.zeros(n * BIP_SIZE, dtype=torch.int32, device=asm.device) if bipartite else None
        self._hist = self._bip = None
        self.add()
        if bipartite:
            self.add_bipartite()

    def _launch(self, fn, hist):
        if not self.bins:
            return
        with torch.cuda.device(self.asm.device):
            check(fn(C.byref(self.asm.view()), _class_records(self.pileup, self.asm, self.modtype), self.tile_begin,
                     self.tile_count, 0, 0, ptr(self.contig_slot), len(self.bins), ptr(hist), _stream()), fn.__name__)

    def add(self) -> "BinSweep":
        """One more pass over the listed bins into the raw IUPAC histograms (counters add)."""
        self._launch(lib.nmb_sweep_hist, self.raw)
        self._hist = None
        return self

    def add_bipartite(self) -> "BinSweep":
        """One more pass into the raw bipartite histograms (counters add)."""
        if self.bip_raw is None:
            raise ValueError("this BinSweep was made with bipartite=False")
        self._launch(lib.nmb_sweep_bipartite, self.bip_raw)
        self._bip = None
        return self

    @property
    def hist(self) -> torch.Tensor:
        """Finished IUPAC histograms [bin][HIST_SIZE] (nmb_sweep_finalize on a copy of the raw ones)."""
        if self._hist is None:
            with torch.cuda.device(self.asm.device):
                h = self.raw.clone()
                if self.bins:
                    check(lib.nmb_sweep_finalize(ptr(h), len(self.bins), _stream()), "nmb_sweep_finalize")
            self._hist = h
        return self._hist.view(-1, HIST_SIZE)

    @property
    def bip(self):
        """Finished bipartite histograms [bin][BIP_SIZE], or None without bipartite."""
        if self.bip_raw is None:
            return None
        if self._bip is None:
            with torch.cuda.device(self.asm.device):
                h = self.bip_raw.clone()
                if self.bins:
                    check(lib.nmb_sweep_bipartite_finalize(ptr(h), len(self.bins), _stream()),
                          "nmb_sweep_bipartite_finalize")
            self._bip = h
        return self._bip.view(-1, BIP_SIZE)

    def index(self, bin_name) -> SweepIndex:
        """SweepIndex over one bin's finished histograms: table / counts / candidates / bipartite_* as for a
        SweepIndex of that bin's contig range."""
        s = self.slot[bin_name]
        return SweepIndex.of_finished(self.asm, self.pileup, self.modtype, self.hist[s],
                                      None if self.bip_raw is None else self.bip[s])

    def counts(self, bin_name, motif_iupac: str, mod_pos: int) -> tuple[int, int]:
        """(n_mod, n_nomod) of one motif in one bin: an IUPAC motif of length 4..8, or left + "N" * gap + right of a
        bipartite shape."""
        index = self.index(bin_name)
        m = _BIPARTITE.fullmatch(motif_iupac)
        if m and len(motif_iupac) > MAX_K:
            return index.bipartite_counts(m.group(1), len(m.group(2)), m.group(3), mod_pos)
        return index.counts(motif_iupac, mod_pos, keep=False)

    def bipartite_iupac_counts(self, bin_name, left: str, gap: int, right: str, mod_pos: int) -> tuple[int, int]:
        """(n_mod, n_nomod) of the motif left + "N" * gap + right in one bin, halves over BIP_LETTERS."""
        return self.index(bin_name).bipartite_iupac_counts(left, gap, right, mod_pos, keep=False)

    def count_matrix(self, motifs, mod_positions, bins=None) -> tuple[np.ndarray, np.ndarray]:
        """(n_mod, n_nomod): int64 arrays [len(bins)][len(motifs)], the exact counts of every listed motif in every
        listed bin (rows follow `bins`, default the sweep's bins), from ONE nmb_sweep_lookup launch over the finished
        histograms: a motif costs the cells it stands for, not a table expansion.  Motifs as SweepIndex.count_many
        takes them (covers() tells which a list holds); BinSweep.counts(b, m, p) is the entry mod 2^32."""
        records = _lookup_records(motifs, mod_positions, self.bip_raw is not None,
                                  "this BinSweep was made with bipartite=False")
        rows = _bin_rows(self.slot, bins)
        out = self._count_device(records, [self.slot[b] for b in rows]).cpu().numpy()
        return out[..., 0], out[..., 1]

    def _count_device(self, records: np.ndarray, slots) -> torch.Tensor:
        """[len(slots)][len(records)][2] int64 device tensor of checked records in the given slots of this sweep."""
        d = self.asm.device
        with torch.cuda.device(d):
            if not len(slots) or not len(records):
                return torch.zeros((len(slots), len(records), 2), dtype=torch.int64, device=d)
            slot = torch.tensor(slots, dtype=torch.int32, device=d)
            bip = self.bip if (records["kind"] == 1).any() else None
            return _lookup(self.hist, bip, slot, len(slots), records)

    def candidates(self, min_mean: float = 0.7, min_mod: int = 50, ks=range(MIN_K, MAX_K + 1), bipartite: bool = True,
                   scratch_bytes: int = 8 << 30, capacity: int = 1 << 20, bipartite_letters: str = "ACGT",
                   prune: bool = False):
        """Every bin's motifs with posterior mean (5 + n_mod) / (10 + n_mod + n_nomod) >= min_mean and n_mod >=
        min_mod, as SweepIndex.candidates finds them per (k, mod_pos), plus the bipartite ones whose modified position
        holds the canonical base.  pandas frame with columns bin, mod_type, motif (IUPAC; bipartite as left + "N" *
        gap + right), mod_position, n_mod, n_nomod, mean; rows in bin order, then k, then mod_position, then table
        index, the bipartite shapes after k = 8 (by gap, then (3,3) (3,4) (4,3) (4,4), then mod_position, then
        index).  Bins are processed in chunks of max(1, scratch_bytes // table_scratch_bytes(max k)); `capacity` is
        the initial number of hit records per pass (a pass with more hits runs again with the exact count).
        bipartite_letters="IUPAC" enumerates bipartite halves over the 14 letters BIP_LETTERS instead of ACGT (index
        = SweepIndex.bipartite_iupac_index, bins in chunks of scratch_bytes // bip_iupac_scratch_bytes()).

        prune=True drops every candidate that a one-letter neighbour in its own table shows to be a redundant
        specialisation (a widening P of a letter other than the modified one passes and Q = P - M has posterior mean
        >= min_mean: GATCA next to GATCM) or a mixture (a narrowing C passes and Q = M - C has mean < min_mean: CCHGG
        next to CCWGG), in the same passes on the device (the filters' prune flag); the frame is the matching
        subsequence of the prune=False one.  Lattices: the 15 IUPAC letters for k-mers, ACGT + * or the 14 letters + *
        for the bipartite halves (* = any of ACGT, never a row)."""
        groups, bip_groups, parts = self._hits(min_mean, min_mod, ks, bipartite, scratch_bytes, capacity,
                                               bipartite_letters, prune)
        return _frame(parts, groups, bip_groups, self.bins, self.mod_type, self.canonical)

    def _hits(self, min_mean, min_mod, ks, bipartite, scratch_bytes, capacity, bipartite_letters, prune):
        """(groups, bip_groups, [(group number, hit records)]) of candidates(): every pass's records, with the slots of
        this sweep."""
        ks, groups, bip_groups = _candidate_groups(min_mod, ks, bipartite, bipartite_letters, self.bip_raw is not None)
        d, n_bins = self.asm.device, len(self.bins)
        state = {"cap": max(int(capacity), 1)}
        parts = []  # (group, hit records)

        def collect(group, launch, slot0=0):
            with torch.cuda.device(d):
                n_out = torch.zeros(1, dtype=torch.int64, device=d)
                if "buf" not in state or state["buf"].numel() < state["cap"] * 16:
                    state["buf"] = torch.empty(state["cap"] * 16, dtype=torch.uint8, device=d)
                launch(ptr(state["buf"]), state["cap"], ptr(n_out))
                m = int(n_out.item())
                if m > state["cap"]:  # count-then-fill: run again with room for every hit
                    state["cap"] = m
                    state["buf"] = torch.empty(m * 16, dtype=torch.uint8, device=d)
                    launch(ptr(state["buf"]), m, ptr(n_out))
                hits = state["buf"][:m * 16].cpu().numpy().view(_lib.SWEEP_HIT_DTYPE)
                hits["slot"] += slot0
                parts.append((group, hits))

        # groups read from expanded tables, bins in chunks: (scratch bytes per bin, number of the first group, groups)
        passes = []
        if groups and n_bins:
            passes.append((table_scratch_bytes(ks[-1]), 0, groups))
        if bip_groups and n_bins:
            passes.append((bip_iupac_scratch_bytes(), len(groups), bip_groups))
        for per_bin, first, todo in passes:
            chunk = max(1, int(scratch_bytes) // per_bin)
            for s0 in range(0, n_bins, chunk):
                ns = min(chunk, n_bins - s0)
                for j, group in enumerate(todo):
                    with torch.cuda.device(d):
                        if len(group) == 2:  # (k, mod_pos): 5 states -> 15 IUPAC letters, every axis but the first
                            k, mp = group
                            tab = _expand([_slice(self.hist.view(-1)[s0 * HIST_SIZE:], ns, k, mp, cls, self.canonical)
                                           for cls in (0, 1)], 5, k - 2)
                            fn, args = lib.nmb_sweep_expand_filter, (15 ** (k - 2), k, mp)
                        else:  # (a, g, b, mod_pos): halves from 4 states -> the 14 letters other than N
                            a, g, b, mp = group
                            tab = _expand([_bip_iupac_slice(self.bip.view(-1)[s0 * BIP_SIZE:], ns, a, g, b, mp, cls,
                                                            self.canonical) for cls in (0, 1)], 4, a + b - 2)
                            fn, args = lib.nmb_sweep_bip_iupac_expand_filter, (14 ** (a + b - 2),)

                    def launch(out, cap, n_out, tab=tab, ns=ns, fn=fn, args=args):
                        check(fn(ptr(tab[0]), ptr(tab[1]), ns, *args, float(min_mean), int(min_mod), int(prune), out,
                                 cap, n_out, _stream()), fn.__name__)

                    collect(first + j, launch, s0)
                    del tab
        if bipartite and n_bins and bip_groups is None:
            def launch_bip(out, cap, n_out):
                check(lib.nmb_sweep_bipartite_filter(ptr(self.bip), n_bins, _BASE_DIGIT[self.canonical],
                                                     float(min_mean), int(min_mod), int(prune), out, cap, n_out,
                                                     _stream()),
                      "nmb_sweep_bipartite_filter")

            collect(len(groups), launch_bip)
        return groups, bip_groups, parts


def _candidate_groups(min_mod, ks, bipartite: bool, bipartite_letters: str, has_bipartite: bool) -> tuple:
    """The argument checks of BinSweep.candidates and its record groups: (sorted ks, [(k, mod_pos)], bip_groups),
    bip_groups None for ACGT halves (one pass over the finished histograms after the (k, mod_pos) groups), else the
    (a, g, b, mod_pos) of every degenerate bipartite group."""
    if min_mod < 1:
        raise ValueError("min_mod must be >= 1: every motif without rows has the prior mean 0.5")
    ks = sorted(set(int(k) for k in ks))
    if any(not MIN_K <= k <= MAX_K for k in ks):
        raise ValueError("ks must lie in 4..8")
    if bipartite_letters not in ("ACGT", "IUPAC"):
        raise ValueError('bipartite_letters must be "ACGT" or "IUPAC"')
    if bipartite and not has_bipartite:
        raise ValueError("this BinSweep was made with bipartite=False")
    groups = [(k, mp) for k in ks for mp in range(k)]
    bip_groups = None
    if bipartite and bipartite_letters == "IUPAC":
        bip_groups = [(a, g, b, o if o < a else o + g) for g in range(4, 9) for a, b in _BIP_SHAPES
                      for o in range(a + b)]
    return ks, groups, bip_groups


def _frame(parts, groups, bip_groups, bins, mod_type, canonical: str):
    """The candidate frame of hit records [(group number, records)] whose slots index `bins`: rows in slot order, then
    group, then table index.  bip_groups: None for the ACGT bipartite records (one group after `groups`), else the
    (a, g, b, mod_pos) of each degenerate bipartite group, numbered from len(groups) on."""
    import pandas as pd

    group = np.concatenate([np.full(len(h), g, dtype=np.int64) for g, h in parts]) if parts else np.zeros(0, np.int64)
    hits = np.concatenate([h for _, h in parts]) if parts else np.zeros(0, _lib.SWEEP_HIT_DTYPE)
    n_groups = len(groups) + (1 if bip_groups is None else len(bip_groups))
    key = (hits["slot"].astype(np.int64) * n_groups + group) << 32 | hits["index"].astype(np.int64)
    order = np.argsort(key, kind="stable")
    hits, group = hits[order], group[order]
    motif = np.empty(len(hits), dtype=object)
    mod_position = np.empty(len(hits), dtype=np.int64)
    for g in np.unique(group):
        sel = np.flatnonzero(group == g)
        if g < len(groups):
            k, mp = groups[g]
            motif[sel] = decode_motifs(k, mp, hits["index"][sel], canonical)
            mod_position[sel] = mp
        elif bip_groups is None:
            motif[sel], mod_position[sel] = decode_bipartite(hits["index"][sel])
        else:
            a, gap, b, mp = bip_groups[g - len(groups)]
            motif[sel] = decode_bipartite_iupac(a, gap, b, mp, hits["index"][sel], canonical)
            mod_position[sel] = mp
    n_mod, n_nomod = hits["n_mod"].astype(np.int64), hits["n_nomod"].astype(np.int64)
    names = np.empty(len(bins), dtype=object)
    names[:] = bins
    return pd.DataFrame({"bin": names[hits["slot"]], "mod_type": np.full(len(hits), mod_type, dtype=object),
                         "motif": motif, "mod_position": mod_position, "n_mod": n_mod, "n_nomod": n_nomod,
                         "mean": (5.0 + n_mod) / (10.0 + n_mod + n_nomod)})
