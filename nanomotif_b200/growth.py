"""Motif-growth step on the device: methylation windows, active-set filter, PSSM and KL children.

Mirrors, for the part of ``find_best_candidates`` / ``MotifSearcher`` that touches sequence data:

    DNAsequence.sample_at_indices              nanomotif/seq.py:170-189   (strict bounds)
    EqualLengthDNASet.reverse_compliment       nanomotif/seq.py:387-389
    EqualLengthDNASet.convert_to_DNAarray      nanomotif/seq.py:474-478
    DNAarray.filter_sequence_matches / pssm    nanomotif/seq.py:499-537
    EqualLengthDNASet.pssm (background)        nanomotif/seq.py:391-422
    _motif_child_nodes_kl_dist_max             nanomotif/find_motifs_bin.py:957-1023

A window is 3 x uint64 on the device instead of a (W, 4) int64 one-hot row; the search's control flow
(heap, graph, thresholds) stays on the host.
"""
from __future__ import annotations

import ctypes as C
import math
import random
import warnings

import numpy as np
import torch

from . import _lib
from ._lib import check, lib, ptr
from .device import DeviceAssembly, _stream, _to_device, sequence_of
from .motif import BASES, Motif, as_motif, window_masks

_WILD_ROW = np.ones(4, dtype=int)


def _one_hot_to_masks(one_hot: np.ndarray) -> np.ndarray:
    """(W, 4) 0/1 matrix in A,T,G,C order -> nmb_motif record (allowed-set per column)."""
    oh = np.asarray(one_hot)
    rec = np.zeros(1, dtype=_lib.MOTIF_DTYPE)
    width = oh.shape[0]
    if width > _lib.MAX_WINDOW:
        raise ValueError(f"window width {width} exceeds {_lib.MAX_WINDOW}")
    bits = ((oh[:, 0] >= 1) * 1 + (oh[:, 1] >= 1) * 2 + (oh[:, 2] >= 1) * 4 + (oh[:, 3] >= 1) * 8).astype(np.uint8)
    rec["allowed"][0, :width] = bits
    rec["len"][0] = width
    return rec


def _window_width(padding: int) -> int:
    """2 * padding + 1, refused with ValueError when it is not a window the device can hold (1..MAX_WINDOW)."""
    width = 2 * int(padding) + 1
    if padding < 0 or width > _lib.MAX_WINDOW:
        raise ValueError(f"window width {width} (padding {padding}) is outside 1..{_lib.MAX_WINDOW}")
    return width


class DeviceDNAarray:
    """Drop-in for the reference's ``DNAarray`` as the motif search uses it: ``shape``, ``copy()``,
    ``filter_sequence_matches(one_hot, keep_matches)`` and ``pssm()``.  Rows live on the GPU as
    bit-packed windows plus an `alive` mask; filtering never moves the windows."""

    def __init__(self, windows: torch.Tensor, width: int, alive: torch.Tensor | None = None, n_alive: int | None = None,
                 hist: np.ndarray | None = None):
        self.windows = windows  # int64 tensor [N, 3] holding x / y / n bit words
        self.width = int(width)
        self.n_total = int(windows.shape[0])
        self.alive = alive
        self.n_alive = self.n_total if n_alive is None else int(n_alive)
        self._hist = hist  # (W, 4) column sums of the alive rows when already known

    # -- construction ---------------------------------------------------------------------------
    @classmethod
    def from_positions(cls, assembly: DeviceAssembly, contig_index, position, strand, padding: int):
        """Windows of +-padding around forward-strand positions (strand 1 = reverse-complemented).
        Positions violating the reference's strict bound padding < i < len - padding must already have
        been dropped (see `methylation_windows`)."""
        width = _window_width(padding)
        d = assembly.device
        ci = np.asarray(contig_index, dtype=np.int64)
        gpos = assembly.starts[ci] + np.asarray(position, dtype=np.int64)
        n = len(gpos)
        win = torch.empty((n, 3), dtype=torch.int64, device=d)
        if n:
            with torch.cuda.device(d):
                g = _to_device(gpos, d)
                st = _to_device(np.asarray(strand, dtype=np.uint8), d)
                view = assembly.view()
                check(lib.nmb_extract_windows(C.byref(view), ptr(g), ptr(st), n, int(padding), ptr(win), _stream()),
                      "nmb_extract_windows")
                torch.cuda.current_stream().synchronize()
        return cls(win, width)

    # -- DNAarray surface -----------------------------------------------------------------------
    @property
    def shape(self):
        return (self.n_alive, self.width, 4)

    def __len__(self):
        return self.n_alive

    def copy(self) -> "DeviceDNAarray":
        return DeviceDNAarray(self.windows, self.width, self.alive, self.n_alive, self._hist)

    def _hist_call(self, masks: np.ndarray, n_counts_all: int, want_keep: bool):
        d = self.windows.device
        m = len(masks)
        with torch.cuda.device(d):
            masks_d = _to_device(masks.view(np.uint8).reshape(-1), d)
            hist = torch.empty((m, self.width, 4), dtype=torch.int32, device=d)
            n_active = torch.empty(m, dtype=torch.int64, device=d)
            keep = torch.empty((m, self.n_total), dtype=torch.uint8, device=d) if want_keep else None
            check(lib.nmb_window_hist(ptr(self.windows), ptr(self.alive), self.n_total, self.width, ptr(masks_d), m,
                                      n_counts_all, ptr(hist), ptr(n_active), ptr(keep), _stream()), "nmb_window_hist")
        return hist, n_active, keep

    def filter_sequence_matches(self, sequence: np.ndarray, keep_matches: bool = True):
        """Rows whose one-hot encoding is <= `sequence` everywhere (keep_matches) or the others
        (seq.py:499-524).  Returns a new array, or None with a warning when nothing is left."""
        assert isinstance(sequence, np.ndarray), "Sequence must be a numpy array"
        assert sequence.shape == (self.width, 4), "Sequence must have the same length as sequences in the array"
        hist, n_active, keep = self._hist_call(_one_hot_to_masks(sequence), 1, True)
        keep = keep[0]
        if keep_matches:
            n = int(n_active[0].item())
            new_alive, new_hist = keep, hist[0].cpu().numpy().astype(np.int64)
        else:
            new_alive = (1 - keep) if self.alive is None else (self.alive & (1 - keep))
            n = self.n_alive - int(n_active[0].item())
            new_hist = None
        if n == 0:
            warnings.warn("No sequences left after filtering")
            return None
        return DeviceDNAarray(self.windows, self.width, new_alive, n, new_hist)

    def column_counts(self, n_counts_all: int = 1) -> np.ndarray:
        """(W, 4) integer column sums of the alive rows (A,T,G,C)."""
        if self._hist is not None and n_counts_all == 1:
            return self._hist
        wild = np.zeros(1, dtype=_lib.MOTIF_DTYPE)
        wild["allowed"][0, : self.width] = 0xF
        wild["len"][0] = self.width
        hist, _, _ = self._hist_call(wild, n_counts_all, False)
        out = hist[0].cpu().numpy().astype(np.int64)
        if n_counts_all == 1:
            self._hist = out
        return out

    def pssm(self) -> np.ndarray:
        """(4, W) float64 column frequencies, N counted for all four bases (seq.py:526-537)."""
        return self.column_counts(1).transpose() / self.n_alive

    def exact_pssm(self) -> np.ndarray:
        """(4, W) exact-letter frequencies, N counted for none (EqualLengthDNASet.pssm, seq.py:391-422)."""
        return self.column_counts(0).transpose() / self.n_alive

    # -- batched expansion ----------------------------------------------------------------------
    def expand(self, motifs, bin_pssm: np.ndarray):
        """For every motif (full-width strings): active-set size, PSSM (4, W) and per-column
        KL(meth || background) -- one hist launch + one PSSM/KL launch for the whole batch."""
        motifs = list(motifs)
        masks = window_masks(motifs, self.width)
        d = self.windows.device
        hist, n_active, _ = self._hist_call(masks, 1, False)
        m = len(motifs)
        with torch.cuda.device(d):
            bg = _to_device(np.ascontiguousarray(bin_pssm, dtype=np.float64), d)
            pssm = torch.empty((m, 4, self.width), dtype=torch.float64, device=d)
            kl = torch.empty((m, self.width), dtype=torch.float64, device=d)
            check(lib.nmb_pssm_kl(ptr(hist), ptr(n_active), m, self.width, ptr(bg), ptr(pssm), ptr(kl), _stream()),
                  "nmb_pssm_kl")
        return n_active.cpu().numpy(), pssm.cpu().numpy(), kl.cpu().numpy()


class WindowPool:
    """The methylation windows of MANY (bin, mod_type) searches in one device array, so that a lock-step
    round of searches is served by ONE histogram launch (nmb_window_hist_ranges) instead of one per search.
    Search `slot` owns rows [begin, end) and the matching slice of the shared `alive` mask."""

    def __init__(self, arrays: list):
        if not arrays:
            raise ValueError("WindowPool needs at least one window array")
        self.width = arrays[0].width
        if any(a.width != self.width for a in arrays):
            raise ValueError("all searches of a pool must use the same window width")
        self.windows = torch.cat([a.windows for a in arrays], dim=0).contiguous()
        d = self.windows.device
        self.n_total = int(self.windows.shape[0])
        self.alive = torch.ones(self.n_total, dtype=torch.uint8, device=d)
        sizes = np.array([a.n_total for a in arrays], dtype=np.int64)
        self.begin = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
        self.end = (self.begin + sizes).astype(np.int64)
        self.n_alive = sizes.copy()
        for a, b, e in zip(arrays, self.begin, self.end):
            if a.alive is not None:
                self.alive[b:e] = a.alive

    @classmethod
    def from_ranges(cls, windows: torch.Tensor, width: int, begin, end) -> "WindowPool":
        """Pool over windows that are already one device array: search `slot` owns rows [begin[slot], end[slot])."""
        self = cls.__new__(cls)
        self.width = int(width)
        self.windows = windows.contiguous()
        self.n_total = int(windows.shape[0])
        self.alive = torch.ones(self.n_total, dtype=torch.uint8, device=windows.device)
        self.begin = np.asarray(begin, dtype=np.int64).copy()
        self.end = np.asarray(end, dtype=np.int64).copy()
        self.n_alive = (self.end - self.begin).astype(np.int64)
        return self

    def _launch(self, slots, motifs, keep_rows):
        d = self.windows.device
        masks = window_masks(motifs, self.width)
        m = len(motifs)
        rb, re = self.begin[slots], self.end[slots]
        with torch.cuda.device(d):
            masks_d = _to_device(masks.view(np.uint8).reshape(-1), d)
            rb_d, re_d = _to_device(rb, d), _to_device(re, d)
            hist = torch.empty((m, self.width, 4), dtype=torch.int32, device=d)
            n_active = torch.empty(m, dtype=torch.int64, device=d)
            check(lib.nmb_window_hist_ranges(ptr(self.windows), ptr(self.alive), self.n_total, self.width, ptr(masks_d),
                                             m, ptr(rb_d), ptr(re_d), int((re - rb).max()) if m else 0, 1, ptr(hist),
                                             ptr(n_active), ptr(keep_rows), _stream()), "nmb_window_hist_ranges")
        return hist, n_active

    def expand_batch(self, requests: list) -> list:
        """requests: [(slot, motif)] -> per request None | (n_active, pssm (4, W)); any number per slot."""
        if not requests:
            return []
        slots = np.array([s for s, _ in requests], dtype=np.int64)
        hist, n_active = self._launch(slots, [m for _, m in requests], None)
        hist, n_active = hist.cpu().numpy().astype(np.int64), n_active.cpu().numpy()
        return [None if n == 0 else (int(n), h.transpose() / n) for h, n in zip(hist, n_active)]

    def remove_batch(self, requests: list) -> list:
        """requests: [(slot, motif)], at most one per slot: drop the matching windows of each slot from its
        alive set; returns the remaining count per request (None when nothing is left)."""
        if not requests:
            return []
        slots = np.array([s for s, _ in requests], dtype=np.int64)
        if len(set(slots.tolist())) != len(slots):
            raise ValueError("remove_batch takes at most one request per search")
        keep_rows = torch.zeros(self.n_total, dtype=torch.uint8, device=self.windows.device)
        _, n_active = self._launch(slots, [m for _, m in requests], keep_rows)
        self.alive &= 1 - keep_rows
        self.n_alive[slots] -= n_active.cpu().numpy()
        return [None if self.n_alive[s] == 0 else int(self.n_alive[s]) for s in slots]


def window_rows(lengths, contig_id, position, strand, fraction_mod, high: float, padding: int):
    """(contig index, position, strand) of the confidently methylated rows that get a window, in the reference's
    order: per contig, '+' sites then '-' sites, each in row order (find_motifs_bin.py:625-672); a site needs
    padding < position < len - padding (seq.py:186, strict on both sides).  One stable sort, no per-contig pass."""
    contig_id = np.asarray(contig_id, dtype=np.int64)
    position = np.asarray(position, dtype=np.int64)
    strand = np.asarray(strand).astype(np.uint8)
    lens = np.asarray(lengths, dtype=np.int64)
    keep = (np.asarray(fraction_mod, dtype=np.float64) >= high) & (contig_id >= 0) & (contig_id < len(lens)) & (strand <= 1)
    keep &= (position > padding) & (position < lens[np.clip(contig_id, 0, max(len(lens) - 1, 0))] - padding)
    rows = np.flatnonzero(keep)
    rows = rows[np.lexsort((strand[rows], contig_id[rows]))]  # stable: row order survives inside (contig, strand)
    return contig_id[rows], position[rows], strand[rows]


def methylation_windows(assembly: DeviceAssembly, contig_id, position, strand, fraction_mod, high: float,
                        padding: int) -> DeviceDNAarray | None:
    """Windows around confidently methylated sites in the reference's row order: per contig, '+' sites
    then reverse-complemented '-' sites (find_motifs_bin.py:625-672).  Columns as numpy arrays;
    contig_id indexes the assembly, strand is 0/1."""
    _window_width(padding)
    ci, pos, st = window_rows(assembly.lengths, contig_id, position, strand, fraction_mod, high, padding)
    if len(pos) == 0:
        return None
    return DeviceDNAarray.from_positions(assembly, ci, pos, st, padding)


def sample_background_starts(sequence: str, length: int, n: int, base: str) -> list[int]:
    """Start positions chosen exactly like DNAsequence.sample_n_subsequences_unique (seq.py:202-225):
    the same ``random.sample`` call on the same list, so a seeded run reproduces the reference's picks."""
    sequence = sequence_of(sequence)
    max_start = len(sequence) - length + 1
    if n > max_start:
        raise ValueError("Too many samples requested for unique subsequences")
    mid = length // 2
    arr = np.frombuffer(sequence.encode("ascii"), dtype=np.uint8)
    valid = np.flatnonzero(arr[mid : mid + max_start] == ord(base)).tolist()
    if len(valid) < n:
        raise ValueError(f"Not enough subsequences with 'C' in the middle (found {len(valid)}, need {n})")
    return random.sample(valid, n)


def background_pssm(assembly: DeviceAssembly, contigs, mod_base: str, padding: int,
                    sampling_frequency: float = 0.01) -> np.ndarray:
    """bin_pssm of find_best_candidates (find_motifs_bin.py:629-650,685): per contig
    max(ceil(0.01 L), 50) random windows centred on the canonical base, exact-letter frequencies."""
    ci, pos = [], []
    for name, seq in contigs.items():
        s = sequence_of(seq)
        n = int(max(math.ceil(len(s) * sampling_frequency), 50))  # :633
        starts = sample_background_starts(s, 2 * padding + 1, n, mod_base)
        ci.append(np.full(n, assembly.index[name], dtype=np.int64))
        pos.append(np.asarray(starts, dtype=np.int64) + padding)
    arr = DeviceDNAarray.from_positions(assembly, np.concatenate(ci), np.concatenate(pos),
                                        np.zeros(sum(len(p) for p in pos), dtype=np.uint8), padding)
    return arr.exact_pssm()


class MTStream:
    """`random.sample(range(n), k)` on the module-level `random` generator, drawn natively.

    The reference samples its background windows with `random.sample(valid_starts, n)` (seq.py:202-225).  CPython's
    `sample` draws `randbelow(n)` until k distinct values have come up (or shuffles a small pool), and `randbelow(n)`
    is `getrandbits(n.bit_length())` = one MT19937 output word shifted right, redrawn while >= n.  The picks are
    therefore a pure function of the generator's 32-bit word stream: `nmb_mt_sample` (host code in libnmb200, the
    standard MT19937 recurrence + the two branches of Lib/random.py) runs on a copy of the Python generator's state
    at ~10 ns per pick instead of ~500, and `sync()` leaves the Python generator exactly where the loop of
    `random.sample` calls would have left it (cfg 3 draws 45 M picks)."""

    def __init__(self):
        from ._lib import NmbMT19937

        self._ver, internal, self._gauss = random.getstate()
        self._state = NmbMT19937()
        self._state.key[:] = internal[:-1]
        self._state.pos = int(internal[-1])

    def sync(self) -> None:
        """Put the module-level `random` generator where the equivalent random.sample calls would have left it."""
        random.setstate((self._ver, tuple(self._state.key) + (int(self._state.pos),), self._gauss))

    def sample(self, n: int, k: int) -> np.ndarray:
        if not 0 <= k <= n:
            raise ValueError("Sample larger than population or is negative")
        out = np.empty(k, dtype=np.int64)
        check(lib.nmb_mt_sample(C.byref(self._state), int(n), int(k), out.ctypes.data), "nmb_mt_sample")
        return out

    def sample_many(self, n, k) -> np.ndarray:
        """The concatenation of random.sample(range(n[i]), k[i]) for consecutive i (one native call)."""
        n = np.ascontiguousarray(n, dtype=np.int64)
        k = np.ascontiguousarray(k, dtype=np.int64)
        if np.any((k < 0) | (k > n)):
            raise ValueError("Sample larger than population or is negative")
        out = np.empty(int(k.sum()), dtype=np.int64)
        check(lib.nmb_mt_sample_many(C.byref(self._state), n.ctypes.data, k.ctypes.data, len(n), out.ctypes.data),
              "nmb_mt_sample_many")
        return out


def prepare_searches(scorer, mod_type, padding: int, high: float, bin_names=None, sampling_frequency: float = 0.01,
                     seeds=None):
    """Everything find_best_candidates builds before its search loop (find_motifs_bin.py:625-686), for EVERY bin of a
    MultiBinScorer at once and on the device: the methylation windows of all bins as one WindowPool and each bin's
    background PSSM.  Returns (pool, bin_pssms, totals): search slot i belongs to bin_names[i].

    Windows: the confidently methylated rows (fraction_mod >= high) of `mod_type` that satisfy the strict bound
    padding < position < len - padding (seq.py:186), in the reference's order -- per contig '+' sites then '-' sites,
    each in row order -- selected and ordered by ONE stable device sort over the rows the scorer already holds, then
    ONE nmb_extract_windows launch.
    Background (seq.py:202-225 + 391-422): per contig max(ceil(0.01 L), 50) windows centred on the canonical base.  The
    reference draws them with random.sample(valid_starts, n); its picks depend only on len(valid_starts) and n, so the
    host draws random.sample(range(N), n) from the SAME global `random` stream (bins and contigs in order; `seeds[i]`
    re-seeds before bin i) while the valid starts themselves are enumerated on the device: the canonical base's match
    plane (K3) compacted once for the whole assembly, per-contig ranges by binary search."""
    from .api import _match_plane, _compact
    from .motif import Motif as _Motif

    asm = scorer.assembly
    d = asm.device
    names = list(scorer._ranges) if bin_names is None else list(bin_names)
    mti = scorer.mod_types.index(mod_type)
    width = _window_width(padding)
    if not scorer.rows:
        raise ValueError("the scorer keeps no pileup rows (built with keep_rows=False or from_device)")
    from .search import CANONICAL

    base = CANONICAL[str(mod_type)]
    with torch.cuda.device(d):
        cat = lambda k: torch.cat([getattr(r, k) for r in scorer.rows]) if len(scorer.rows) > 1 else getattr(scorer.rows[0], k)
        cid, pos, strand, frac, mt = cat("contig_id"), cat("position"), cat("strand"), cat("fraction_mod"), cat("mod_type")
        safe = cid.clamp(min=0).long()
        keep = (mt == mti) & (frac >= high) & (strand <= 1) & (cid >= 0)
        keep &= (pos > padding) & (pos < asm.contig_len[safe] - padding)
        idx = torch.nonzero(keep).view(-1)
        key = cid[idx].long() * 2 + strand[idx].long()
        key, perm = torch.sort(key, stable=True)  # row order survives inside (contig, strand)
        idx = idx[perm]
        gpos = (asm.contig_start[cid[idx].long()] + pos[idx]).contiguous()
        st = strand[idx].contiguous()
        n = int(idx.numel())
        win = torch.empty((n, 3), dtype=torch.int64, device=d)
        view = asm.view()
        if n:
            check(lib.nmb_extract_windows(C.byref(view), ptr(gpos), ptr(st), n, int(padding), ptr(win), _stream()),
                  "nmb_extract_windows")
        bounds = np.array([[2 * scorer._ranges[b][0], 2 * scorer._ranges[b][1]] for b in names], dtype=np.int64)
        edges = torch.searchsorted(key, torch.from_numpy(bounds.reshape(-1)).to(d)).cpu().numpy().reshape(-1, 2)
        pool = WindowPool.from_ranges(win, width, edges[:, 0], edges[:, 1])

        # ---- background: valid window centres = positions of the canonical base, enumerated on the device ----
        plane, _, _ = _match_plane(asm, _Motif(base, 0), align=0)
        P = _compact(plane, 0, asm.n_tiles * _lib.TILE_BP)  # every position holding `base`, ascending (global)
        contigs = [c for b in names for c in range(*scorer._ranges[b])]
        L = asm.lengths[contigs]
        max_start = L - width + 1
        lo_pos = asm.starts[contigs] + padding
        q = torch.from_numpy(np.stack([lo_pos, lo_pos + np.maximum(max_start, 0)], axis=1).reshape(-1)).to(d)
        lohi = torch.searchsorted(P, q).cpu().numpy().reshape(-1, 2)
        n_valid = lohi[:, 1] - lohi[:, 0]
        # samples per contig (find_motifs_bin.py:633) and the reference's two refusals (seq.py:210, :219)
        k_all = np.maximum(np.ceil(L * sampling_frequency), 50).astype(np.int64)
        if np.any(k_all > max_start):
            raise ValueError("Too many samples requested for unique subsequences")
        short = np.flatnonzero(n_valid < k_all)
        if len(short):
            ci = int(short[0])
            raise ValueError(f"Not enough subsequences with 'C' in the middle (found {int(n_valid[ci])}, need {int(k_all[ci])})")
        picks, at, bg_begin, bg_end = [], 0, [], []
        ci = 0
        stream = MTStream()
        for i, b in enumerate(names):
            if seeds is not None:
                random.seed(seeds[i])
                stream = MTStream()
            nc = scorer._ranges[b][1] - scorer._ranges[b][0]
            k_bin = k_all[ci:ci + nc]
            got = stream.sample_many(n_valid[ci:ci + nc], k_bin)  # one call per bin, contigs in order
            picks.append(got + np.repeat(lohi[ci:ci + nc, 0], k_bin))
            bg_begin.append(at)
            at += int(k_bin.sum())
            bg_end.append(at)
            ci += nc
        stream.sync()  # the module-level generator continues where the reference's calls would have left it
        centre = P[_to_device(np.concatenate(picks), d)].contiguous()  # start + padding = the base's own position
        nb = int(centre.numel())
        bgw = torch.empty((nb, 3), dtype=torch.int64, device=d)
        zeros = torch.zeros(nb, dtype=torch.uint8, device=d)
        check(lib.nmb_extract_windows(C.byref(view), ptr(centre), ptr(zeros), nb, int(padding), ptr(bgw), _stream()),
              "nmb_extract_windows")
        wild = np.zeros(len(names), dtype=_lib.MOTIF_DTYPE)
        wild["allowed"][:, :width] = 0xF
        wild["len"][:] = width
        masks_d = _to_device(wild.view(np.uint8).reshape(-1), d)
        rb, re = np.asarray(bg_begin, dtype=np.int64), np.asarray(bg_end, dtype=np.int64)
        rb_d, re_d = _to_device(rb, d), _to_device(re, d)
        hist = torch.empty((len(names), width, 4), dtype=torch.int32, device=d)
        n_active = torch.empty(len(names), dtype=torch.int64, device=d)
        check(lib.nmb_window_hist_ranges(ptr(bgw), None, nb, width, ptr(masks_d), len(names), ptr(rb_d), ptr(re_d),
                                         int((re - rb).max()), 0, ptr(hist), ptr(n_active), None, _stream()),
              "nmb_window_hist_ranges")
        hist = hist.cpu().numpy().astype(np.int64)
    pssms = [h.transpose() / float(e - b) for h, b, e in zip(hist, bg_begin, bg_end)]  # exact-letter frequencies
    return pool, pssms, [int(x) for x in (edges[:, 1] - edges[:, 0])]


def column_kl(pk: np.ndarray, qk: np.ndarray) -> np.ndarray:
    """scipy.stats.entropy(pk, qk) (axis 0, natural log; find_motifs_bin.py:974) as the same numpy / scipy.special
    operations in the same order, without the array-API and nan-policy wrappers around it: those cost ~0.4 ms per call,
    which is 90 % of the host time of a lock-step search round (one call per search and expansion)."""
    from scipy.special import rel_entr

    pk = np.asarray(pk, dtype=np.float64)
    qk = np.broadcast_to(np.asarray(qk, dtype=np.float64), pk.shape)
    with np.errstate(invalid="ignore", divide="ignore"):
        qk = qk / np.sum(qk, axis=0, keepdims=True)
        pk = pk / np.sum(pk, axis=0, keepdims=True)
    return np.sum(rel_entr(pk, qk), axis=0)


def kl_children(motif, meth_pssm: np.ndarray, bin_pssm: np.ndarray, kl: np.ndarray | None = None, min_kl: float = 0.05,
                freq_threshold: float = 0.15) -> list[Motif]:
    """Children of `motif` at the wildcard position of maximum KL divergence
    (_motif_child_nodes_kl_dist_max, find_motifs_bin.py:957-1023).  `kl` may come from
    DeviceDNAarray.expand; otherwise it is computed here exactly like scipy.stats.entropy."""
    m = as_motif(motif)
    split = m.split()
    if kl is None:
        kl = column_kl(meth_pssm, bin_pssm)
    wild = np.fromiter((b == "." for b in split), dtype=bool, count=len(split))
    if not wild.any():
        return []
    masked = np.where(wild, np.asarray(kl, dtype=np.float64), 0.0)  # KL of the fixed positions forced to 0 (:983-985)
    if np.max(masked) < min_kl:
        return []
    pos = int(np.argmax(masked))
    ok = np.logical_and(meth_pssm[:, pos] > bin_pssm[:, pos] * 0.5, meth_pssm[:, pos] > freq_threshold)
    out = []
    for i in np.argwhere(ok).reshape(-1):
        toks = list(split)
        toks[pos] = BASES[int(i)]
        out.append(Motif("".join(toks), m.mod_position))
    return out
