"""Contig x motif methylation-pattern table (K5) -- the operator `nanomotif detect_contamination` /
`include_contigs` obtain from the external Rust package ``epymetheus`` (call site
nanomotif/main.py:167-178; output schema nanomotif/main.py:157-161).

The Rust source is not part of the reference tree, so the semantics are fixed by the written spec in
DESIGN.md (section 4, K5) and SURVEY.md 8c; parity is "exact against oracle/restate.py::
methylation_pattern, unpinned against epimetheus-py 0.7.5".

For every motif string ``<IUPAC>_<mod_type>_<mod_position>`` and contig: occurrences of the motif on
'+' and of its reverse complement on '-' (IUPAC letters with SET semantics) are joined to the pileup
rows of that mod type at the modified base; rows need n_valid_cov >= min_valid_read_coverage and
n_valid_cov / (n_valid_cov + n_diff) >= min_valid_cov_to_diff_fraction.  Per (contig, motif):
n_motif_obs = kept occurrences, mean_read_cov = mean n_valid_cov, methylation_value = median of
n_mod / n_valid_cov (Median) or sum n_mod / sum n_valid_cov (WeightedMean).  Pairs without
observations are omitted.
"""
from __future__ import annotations

import ctypes as C
import enum

import numpy as np
import torch

from . import _lib
from ._lib import check, lib, ptr
from .device import DeviceAssembly, MotifPrograms, _stream, _to_device, _work_counter, sm_count
from .motif import Motif
from .pileup import PileupTable, strand_codes

COLUMNS = ["contig", "motif", "mod_type", "mod_position", "methylation_value", "mean_read_cov", "n_motif_obs"]


class MethylationOutput(enum.Enum):
    Median = "median"
    WeightedMean = "weighted_mean"


def parse_motif_spec(spec: str) -> tuple[str, str, int]:
    """'GATC_a_1' -> ('GATC', 'a', 1)  (nanomotif/main.py:136-140 builds these strings)."""
    iupac, mod_type, pos = spec.rsplit("_", 2)
    return iupac, mod_type, int(pos)


def _planes(asm: DeviceAssembly, regex_motif: Motif):
    progs = MotifPrograms([regex_motif], asm.device, strip=False)
    view = asm.view()
    out = []
    for strand in (0, 1):
        plane = torch.empty(asm.n_words, dtype=torch.int32, device=asm.device)
        check(lib.nmb_match_plane(C.byref(view), ptr(progs.programs), 0, strand, progs.max_len, 0, asm.n_tiles,
                                  ptr(plane), _stream()), "nmb_match_plane")
        out.append(plane)
    return out


class PatternIndex:
    """Join index of ONE mod type on the device (nmb_pattern_index_build): valid-row bit-planes per tile, rank
    directory and (n_mod, n_valid_cov) payload.  `rows`: device tensors contig_id int32 (index into the
    assembly), position int64, strand uint8, n_mod / Nvalid_cov / n_diff int64 and optionally mod_type uint8
    (then only rows with mod_type == want_modtype take part)."""

    def __init__(self, asm: DeviceAssembly, rows: dict, want_modtype: int = 0, min_valid_read_coverage: int = 3,
                 min_valid_cov_to_diff_fraction: float = 0.8):
        self.asm = asm
        d = asm.device
        n = int(rows["position"].numel())
        with torch.cuda.device(d):
            self.valid = torch.empty(asm.n_tiles * 2 * _lib.TILE_WORDS, dtype=torch.int32, device=d)
            self.rank_dir = torch.empty(2 * asm.n_words, dtype=torch.int32, device=d)
            self.payload = torch.empty((max(n, 1), 2), dtype=torch.int32, device=d)
            scratch = torch.empty(2 * asm.n_words // 2048 + 3, dtype=torch.int64, device=d)
            n_valid = torch.zeros(1, dtype=torch.int64, device=d)
            view = asm.view()
            check(lib.nmb_pattern_index_build(C.byref(view), ptr(rows["contig_id"]), ptr(rows["position"]), ptr(rows["strand"]),
                                              ptr(rows.get("mod_type")), int(want_modtype), ptr(rows["n_mod"]),
                                              ptr(rows["Nvalid_cov"]), ptr(rows["n_diff"]), n, int(min_valid_read_coverage),
                                              float(min_valid_cov_to_diff_fraction), ptr(self.valid), ptr(self.rank_dir),
                                              ptr(scratch), ptr(self.payload), ptr(n_valid), _stream()),
                  "nmb_pattern_index_build")
            self.n_valid_rows = int(n_valid.item())


def pattern_table(index: PatternIndex, motifs, median: bool = True, batch: int = 64, motifs_per_item: int | None = None,
                  on_device: bool = False):
    """(stats int64 [n_motifs, n_contigs, 3] = n_motif_obs / sum n_mod / sum n_valid_cov, value float64
    [n_motifs, n_contigs] = median of the per-occurrence fractions, or None) on the host, for regex `Motif`s
    scored against one mod type's index.  Two tile-driven passes per batch of motifs (count, then write +
    exact medians); a batch's results travel to pinned host memory while the next batch is scanned.
    on_device=True keeps both arrays on the GPU (device tensors) for consumers that stay there
    (tables.bin_feature_matrix_device)."""
    asm = index.asm
    d, nc = asm.device, asm.n_contigs
    motifs = list(motifs)
    view = asm.view()
    batch = max(1, min(batch, len(motifs)))
    if on_device:
        with torch.cuda.device(d):
            stats_all = torch.zeros((len(motifs), nc, 3), dtype=torch.int64, device=d)
            value_all = torch.full((len(motifs), nc), float("nan"), dtype=torch.float64, device=d) if median else None
            for b0 in range(0, len(motifs), batch):
                chunk = motifs[b0:b0 + batch]
                progs = MotifPrograms(chunk, d, strip=False)
                nb = len(chunk)
                mpi = motifs_per_item or int(min(_lib.MAX_MOTIFS_PER_ITEM, max(1, nb * asm.n_tiles // (16 * sm_count(d)))))
                stats = stats_all[b0:b0 + nb].view(nb * nc, 3)  # contiguous slice: the scan adds into it in place

                def scan_d(phase, offsets=None, cursor=None, fractions=None):
                    check(lib.nmb_pattern_scan_balanced(C.byref(view), ptr(index.valid), ptr(index.rank_dir), ptr(index.payload),
                                                        ptr(progs.programs), nb, mpi, progs.max_len, phase, ptr(stats),
                                                        ptr(offsets), ptr(cursor), ptr(fractions), 0, ptr(_work_counter(d)),
                                                        _stream()), "nmb_pattern_scan_balanced")

                scan_d(0)
                if median:
                    offsets = torch.empty(nb * nc + 1, dtype=torch.int64, device=d)
                    cursor = torch.empty(nb * nc, dtype=torch.int32, device=d)
                    check(lib.nmb_segment_offsets(ptr(stats), nb * nc, ptr(offsets), ptr(cursor), _stream()), "nmb_segment_offsets")
                    total = int(offsets[-1].item())
                    fractions = torch.empty(max(1, total), dtype=torch.float64, device=d)
                    scan_d(1, offsets, cursor, fractions)
                    med = value_all[b0:b0 + nb].view(nb * nc)
                    check(lib.nmb_segment_median(ptr(fractions), ptr(offsets), nb * nc, ptr(med), _stream()), "nmb_segment_median")
        return stats_all, value_all
    stats_out = np.zeros((len(motifs), nc, 3), dtype=np.int64)
    value_out = np.full((len(motifs), nc), np.nan) if median else None
    with torch.cuda.device(d):
        host = [(torch.empty((batch * nc, 3), dtype=torch.int64, pin_memory=True),
                 torch.empty(batch * nc, dtype=torch.float64, pin_memory=True) if median else None) for _ in range(2)]
        pending = None  # (b0, nb, slot, event, device tensors kept alive until the copy has finished)

        def collect(job):
            b0, nb, slot, ev, _keep = job
            ev.synchronize()
            stats_out[b0:b0 + nb] = host[slot][0][:nb * nc].numpy().reshape(nb, nc, 3)
            if median:
                value_out[b0:b0 + nb] = host[slot][1][:nb * nc].numpy().reshape(nb, nc)

        for bi, b0 in enumerate(range(0, len(motifs), batch)):
            chunk = motifs[b0:b0 + batch]
            progs = MotifPrograms(chunk, d, strip=False)
            nb = len(chunk)
            mpi = motifs_per_item or int(min(_lib.MAX_MOTIFS_PER_ITEM, max(1, nb * asm.n_tiles // (16 * sm_count(d)))))
            stats = torch.zeros((nb * nc, 3), dtype=torch.int64, device=d)

            def scan(phase, offsets=None, cursor=None, fractions=None):
                check(lib.nmb_pattern_scan_balanced(C.byref(view), ptr(index.valid), ptr(index.rank_dir), ptr(index.payload),
                                                    ptr(progs.programs), nb, mpi, progs.max_len, phase, ptr(stats),
                                                    ptr(offsets), ptr(cursor), ptr(fractions), 0, ptr(_work_counter(d)),
                                                    _stream()), "nmb_pattern_scan_balanced")

            scan(0)
            med = None
            if median:
                offsets = torch.empty(nb * nc + 1, dtype=torch.int64, device=d)
                cursor = torch.empty(nb * nc, dtype=torch.int32, device=d)
                check(lib.nmb_segment_offsets(ptr(stats), nb * nc, ptr(offsets), ptr(cursor), _stream()), "nmb_segment_offsets")
                total = int(offsets[-1].item())
                fractions = torch.empty(max(1, total), dtype=torch.float64, device=d)
                med = torch.empty(nb * nc, dtype=torch.float64, device=d)
                scan(1, offsets, cursor, fractions)
                check(lib.nmb_segment_median(ptr(fractions), ptr(offsets), nb * nc, ptr(med), _stream()), "nmb_segment_median")
            slot = bi & 1
            host[slot][0][:nb * nc].copy_(stats, non_blocking=True)
            if median:
                host[slot][1][:nb * nc].copy_(med, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            if pending is not None:
                collect(pending)  # the previous batch, while this one runs
            pending = (b0, nb, slot, ev, (stats, med, progs))
        if pending is not None:
            collect(pending)
    return stats_out, value_out


def load_contigs(assembly) -> dict:
    """{name: sequence str} of a FASTA path or of a {name: str or DNAsequence-like} mapping."""
    from . import dataload

    if isinstance(assembly, str):
        return dataload.load_fasta(assembly)
    return {k: (v if isinstance(v, str) else v.sequence) for k, v in assembly.items()}


def pileup_rows(pileup, names, mod_types, allow_assembly_pileup_mismatch: bool, device, renumber=None):
    """(rows, mismatch) of methylation_pattern: `rows` = the device columns PatternIndex takes, contig ids indexing
    `names`, mod_type indexing `mod_types`; `mismatch` = with allow_assembly_pileup_mismatch=False, whether a row names a
    contig absent from `names` (always False otherwise).  `pileup`: a bedMethyl path (parsed on the device, K6) or a table
    with n_mod and n_diff.  `renumber` (int32 [len(names)], optional): the new id of every contig, -1 to drop its rows --
    a table is cut on the host before the copy, parsed rows are renumbered and compacted on the device."""
    from . import dataload

    d = device
    if isinstance(pileup, str):
        dr = dataload.load_pileup_device(pileup, names, mod_types, with_counts=True, device=d,
                                         keep_unknown_contigs=not allow_assembly_pileup_mismatch)
        mismatch = not allow_assembly_pileup_mismatch and bool((dr.contig_id < 0).any())
        if renumber is not None:
            with torch.cuda.device(d):
                lut = _to_device(np.append(np.asarray(renumber, dtype=np.int32), np.int32(-1)), d)
                dr.contig_id = lut[torch.where(dr.contig_id < 0, len(names), dr.contig_id).long()]
                dr = dr.take_mask((dr.contig_id >= 0).to(torch.uint8))
        return dict(contig_id=dr.contig_id, position=dr.position, strand=dr.strand, mod_type=dr.mod_type, n_mod=dr.n_mod,
                    Nvalid_cov=dr.Nvalid_cov, n_diff=dr.n_diff), mismatch
    table = PileupTable.from_frame(pileup)
    counts = {}
    for k in ("n_mod", "n_diff"):  # in `extra` of a PileupTable, plain columns of a pandas / pyarrow / polars frame
        col = table.extra.get(k)
        if col is None:
            col = dataload._frame_column(pileup, k)
        if col is None:
            raise KeyError("methylation_pattern needs the n_mod and n_diff pileup columns")
        counts[k] = dataload._numeric_column(col, np.int64)
    index = {n: i for i, n in enumerate(names)}
    contig = np.asarray(table.contig).astype(str)
    uniq, inv = np.unique(contig, return_inverse=True)
    lut = np.fromiter((index.get(u, -1) for u in uniq), dtype=np.int32, count=len(uniq))
    cid = lut[inv] if len(uniq) else np.zeros(0, dtype=np.int32)
    mismatch = not allow_assembly_pileup_mismatch and bool((cid < 0).any())
    take = slice(None)
    if renumber is not None:
        cid = np.append(np.asarray(renumber, dtype=np.int32), np.int32(-1))[cid]
        take = np.flatnonzero(cid >= 0)
        cid = cid[take]
    mt_names = np.asarray(table.mod_type).astype(str)[take]
    mt_code = np.full(len(mt_names), 255, dtype=np.uint8)
    for i, m in enumerate(mod_types):
        mt_code[mt_names == m] = i
    with torch.cuda.device(d):
        rows = dict(contig_id=_to_device(cid.astype(np.int32), d),
                    position=_to_device(np.asarray(table.position, dtype=np.int64)[take], d),
                    strand=_to_device(strand_codes(table.strand)[take], d), mod_type=_to_device(mt_code, d),
                    n_mod=_to_device(counts["n_mod"][take], d),
                    Nvalid_cov=_to_device(np.asarray(table.Nvalid_cov, dtype=np.int64)[take], d),
                    n_diff=_to_device(counts["n_diff"][take], d))
    return rows, mismatch


MISMATCH_ERROR = "pileup contains contigs that are absent from the assembly"


def pattern_frame(stats: np.ndarray, value, specs, names, median: bool):
    """The methylation_pattern DataFrame of the [n_motifs, n_contigs] arrays of pattern_table over ALL contigs (`names`
    order): rows motif-major, contigs ascending, pairs without observations omitted.  `specs` = parse_motif_spec of each
    motif; `value` is ignored unless `median` (the weighted mean is sum n_mod / sum n_valid_cov)."""
    import pandas as pd

    if not median:
        with np.errstate(divide="ignore", invalid="ignore"):
            value = stats[:, :, 1] / stats[:, :, 2]
    mi, ci = np.nonzero(stats[:, :, 0] > 0)  # motif-major, contigs ascending; pairs without observations are omitted
    obs = stats[mi, ci, 0]
    return pd.DataFrame({
        "contig": np.array(names, dtype=object)[ci],
        "motif": np.array([s[0] for s in specs], dtype=object)[mi],
        "mod_type": np.array([s[1] for s in specs], dtype=object)[mi],
        "mod_position": np.array([s[2] for s in specs], dtype=np.int8)[mi],
        "methylation_value": value[mi, ci].astype(np.float64),
        "mean_read_cov": stats[mi, ci, 2] / obs,
        "n_motif_obs": obs.astype(np.int32),
    }, columns=COLUMNS)


def methylation_pattern(pileup, assembly, motifs, threads: int = 1, min_valid_read_coverage: int = 3,
                        batch_size: int = 1000, min_valid_cov_to_diff_fraction: float = 0.8, output: str | None = None,
                        allow_assembly_pileup_mismatch: bool = True,
                        output_type: MethylationOutput = MethylationOutput.Median, device=None):
    """Same keyword arguments as ``epymetheus.methylation_pattern``.  `pileup`: path to a bedMethyl file, a
    pandas / pyarrow / polars frame with n_mod and n_diff columns, or a PileupTable with them in ``extra``;
    `assembly`: FASTA path or {name: sequence}.  Returns a pandas DataFrame with the columns of
    nanomotif/main.py:157-161 (and writes it as TSV to `output`).
    `threads` and `batch_size` are accepted for signature compatibility (the GPU needs neither)."""
    contigs = load_contigs(assembly)
    asm = DeviceAssembly.from_sequences(contigs, device)
    d = asm.device
    motifs = [str(m) for m in motifs]
    specs = [parse_motif_spec(m) for m in motifs]
    mod_types = sorted({mt for _, mt, _ in specs})
    rows, mismatch = pileup_rows(pileup, asm.names, mod_types, allow_assembly_pileup_mismatch, d)
    if mismatch:
        raise ValueError(MISMATCH_ERROR)

    median = output_type == MethylationOutput.Median
    nc = asm.n_contigs
    stats = np.zeros((len(specs), nc, 3), dtype=np.int64)
    value = np.full((len(specs), nc), np.nan)
    for ti, mt in enumerate(mod_types):
        sel = [i for i, s in enumerate(specs) if s[1] == mt]
        index = PatternIndex(asm, rows, ti, min_valid_read_coverage, min_valid_cov_to_diff_fraction)
        st, val = pattern_table(index, [Motif(specs[i][0], specs[i][2]).from_iupac() for i in sel], median)
        stats[sel] = st
        if median:
            value[sel] = val
        del index
    df = pattern_frame(stats, value, specs, asm.names, median)
    if output is not None:
        df.to_csv(output, sep="\t", index=False)
    return df


def methylation_pattern_rows(table, contigs, spec: str, min_valid_read_coverage: int = 3,
                             min_valid_cov_to_diff_fraction: float = 0.8, device=None):
    """One motif through the ROW-driven kernels (nmb_pattern_stats / nmb_pattern_median: every filtered pileup row
    tests its bit of the motif's match plane).  Kept as an independent implementation for cross-checks of the
    tile-driven path; returns (stats [n_contigs, 3], median [n_contigs])."""
    asm = DeviceAssembly.from_sequences(contigs, device)
    d = asm.device
    iupac, mod_type, mod_pos = parse_motif_spec(spec)
    names = np.asarray(table.contig).astype(str)
    cid = np.fromiter((asm.index.get(u, -1) for u in names), dtype=np.int64, count=len(names))
    pos = np.asarray(table.position, dtype=np.int64)
    cov = np.asarray(table.Nvalid_cov, dtype=np.int64)
    diff = np.asarray(table.extra["n_diff"], dtype=np.int64)
    ok = (cid >= 0) & (pos >= 0) & (pos < asm.lengths[np.maximum(cid, 0)]) & (cov >= min_valid_read_coverage)
    ok &= np.asarray(table.mod_type).astype(str) == mod_type
    with np.errstate(divide="ignore", invalid="ignore"):
        ok &= (cov / (cov + diff)) >= min_valid_cov_to_diff_fraction
    sel = np.flatnonzero(ok)
    sel = sel[np.lexsort((pos[sel], cid[sel]))]  # the row-driven kernels want contig-sorted rows
    nc = asm.n_contigs
    with torch.cuda.device(d):
        gpos = _to_device(asm.starts[cid[sel]] + pos[sel], d)
        st = _to_device(strand_codes(table.strand)[sel], d)
        c32 = _to_device(cid[sel].astype(np.int32), d)
        nmod = _to_device(np.asarray(table.extra["n_mod"], dtype=np.int64)[sel].astype(np.int32), d)
        cv = _to_device(cov[sel].astype(np.int32), d)
        fwd, rev = _planes(asm, Motif(iupac, mod_pos).from_iupac())
        stats = torch.empty((nc, 3), dtype=torch.int64, device=d)
        offsets = torch.empty(nc + 1, dtype=torch.int64, device=d)
        cursor = torch.empty(nc, dtype=torch.int32, device=d)
        check(lib.nmb_pattern_stats(ptr(gpos), ptr(st), ptr(c32), ptr(nmod), ptr(cv), len(sel), ptr(fwd), ptr(rev), nc,
                                    ptr(stats), ptr(offsets), ptr(cursor), _stream()), "nmb_pattern_stats")
        total = int(offsets[-1].item())
        fractions = torch.empty(max(1, total), dtype=torch.float64, device=d)
        median = torch.empty(nc, dtype=torch.float64, device=d)
        check(lib.nmb_pattern_median(ptr(gpos), ptr(st), ptr(c32), ptr(nmod), ptr(cv), len(sel), ptr(fwd), ptr(rev), nc,
                                     ptr(offsets), ptr(cursor), ptr(fractions), ptr(median), _stream()), "nmb_pattern_median")
        return stats.cpu().numpy(), median.cpu().numpy()
