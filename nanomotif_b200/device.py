"""Device-resident data model of the scoring path: packed assembly, pileup class planes, scan launches.

torch is used for device memory, streams and H2D/D2H copies only; every byte of arithmetic on the
path happens in libnmb200's CUDA kernels (nanomotif_b200/csrc).  Layout: DESIGN.md section 3.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Mapping, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import NmbAssembly, check, lib, ptr
from .motif import pack_motifs


def _require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("nanomotif_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"nanomotif_b200 runs on CUDA devices only, got {dev}")
    return dev


_NP_OF = {torch.int32: np.int32, torch.int64: np.int64, torch.uint8: np.uint8, torch.float64: np.float64,
          torch.uint16: np.uint16}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


_TORCH_OF = {np.dtype(k): v for k, v in ((np.int32, torch.int32), (np.int64, torch.int64), (np.uint8, torch.uint8),
                                         (np.int8, torch.int8), (np.float64, torch.float64), (np.uint16, torch.uint16),
                                         (np.int16, torch.int16), (np.float32, torch.float32), (np.bool_, torch.bool))}
_STAGERS: dict[int, int] = {}
STAGE_MIN_BYTES = 4 << 20   # smaller copies go through cudaMemcpy directly
STAGE_SLOT_BYTES = 4 << 20


def stager_threads() -> int:
    """Host threads of the staging copies: NMB_STAGE_THREADS, else the cores this process may run on (at most 16)."""
    import os

    env = os.environ.get("NMB_STAGE_THREADS")
    if env:
        return max(0, int(env))
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        n = os.cpu_count() or 1
    return max(1, min(16, n))


def _stager(device: torch.device):
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _STAGERS:
        n = stager_threads()
        handle = C.c_void_p()
        if n > 0:
            with torch.cuda.device(idx):
                check(lib.nmb_stager_create(STAGE_SLOT_BYTES, n, C.byref(handle)), "nmb_stager_create")
        _STAGERS[idx] = handle.value or 0
    return _STAGERS[idx]


_AsUTF8AndSize = C.pythonapi.PyUnicode_AsUTF8AndSize
_AsUTF8AndSize.restype = C.c_void_p
_AsUTF8AndSize.argtypes = [C.py_object, C.POINTER(C.c_ssize_t)]


def _ascii_pointers(strings) -> np.ndarray | None:
    """Addresses of the character data of ASCII str objects (valid while the strings live), or None when one of
    them is not pure ASCII."""
    out = np.empty(len(strings), dtype=np.uint64)
    size = C.c_ssize_t()
    for i, s in enumerate(strings):
        p = _AsUTF8AndSize(s, C.byref(size))
        if not p or size.value != len(s):
            return None
        out[i] = p
    return out


def _to_device_narrow(arr: np.ndarray, device: torch.device) -> torch.Tensor | None:
    """int64 host array -> int32 device tensor through the stager's narrowing copy (half the PCIe bytes), or None
    when the array is small, no stager is configured or a value does not fit."""
    arr = np.ascontiguousarray(arr)
    if arr.dtype != np.int64 or arr.nbytes < STAGE_MIN_BYTES:
        return None
    st = _stager(device)
    if not st:
        return None
    flag = C.c_int32(0)
    with torch.cuda.device(device):
        out = torch.empty(arr.shape, dtype=torch.int32, device=device)
        check(lib.nmb_stager_copy_narrow(st, ptr(out), arr.ctypes.data, arr.size, C.byref(flag), _stream()),
              "nmb_stager_copy_narrow")
    return None if flag.value else out


def _to_device(arr: np.ndarray, device: torch.device) -> torch.Tensor:
    """Host array -> device tensor on the current stream.  Large pageable arrays (the Arrow buffers of a pileup table)
    go through the multi-threaded pinned stager (csrc/stage.cu); the source is never modified."""
    arr = np.ascontiguousarray(arr)
    tdt = _TORCH_OF.get(arr.dtype)
    if arr.nbytes >= STAGE_MIN_BYTES and tdt is not None:
        st = _stager(device)
        if st:
            with torch.cuda.device(device):
                out = torch.empty(arr.shape, dtype=tdt, device=device)
                check(lib.nmb_stager_copy(st, ptr(out), arr.ctypes.data, arr.nbytes, _stream()), "nmb_stager_copy")
            return out
    if not arr.flags.writeable:  # e.g. np.frombuffer over a bytes object; torch wants writable memory
        arr = arr.copy()
    return torch.from_numpy(arr).to(device, non_blocking=True)


def sequence_of(obj) -> str:
    """Contig text of a str or of a reference ``DNAsequence`` (nanomotif/seq.py:21-60)."""
    return obj if isinstance(obj, str) else obj.sequence


def plan_layout(lengths: Sequence[int]) -> tuple[np.ndarray, int]:
    """Global start position of every contig (aligned to CHUNK_BP = 512 bp, >= 64 flagged positions apart) and
    the number of 65536-bp tiles."""
    # every start is a multiple of CHUNK_BP, so a contig advances the cursor by its length + gap rounded up to chunks
    lengths = np.asarray(lengths, dtype=np.int64)
    step = -(-(lengths + _lib.MIN_GAP_BP) // _lib.CHUNK_BP) * _lib.CHUNK_BP
    ends = np.cumsum(step)
    starts = ends - step
    cur = int(ends[-1]) if len(lengths) else 0
    n_tiles = max(1, -(-cur // _lib.TILE_BP))
    return starts, n_tiles


class DeviceAssembly:
    """Contigs packed as 2-bit planes in tile records on one GPU (replaces the ``dict[str, DNAsequence]``
    of Python strings the reference scans, nanomotif/seq.py:11-19)."""

    def __init__(self, names, lengths, ascii_u8, ascii_off, device=None, sync: bool = True):
        self.device = _require_cuda(device)
        self.names = list(names)
        self.index = {n: i for i, n in enumerate(self.names)}
        self.lengths = np.asarray(lengths, dtype=np.int64)
        self.starts, self.n_tiles = plan_layout(self.lengths)
        self.n_contigs = len(self.names)
        self.n_words = self.n_tiles * _lib.TILE_WORDS
        with torch.cuda.device(self.device):
            d = self.device
            self.seq_records = torch.empty(self.n_tiles * _lib.SEQ_REC_WORDS, dtype=torch.int32, device=d)
            self.nonacgt = torch.empty(self.n_words + 2 * _lib.HALO_WORDS, dtype=torch.int32, device=d)
            self.contig_start = _to_device(self.starts, d)
            self.contig_len = _to_device(self.lengths, d)
            if isinstance(ascii_u8, torch.Tensor):  # device tensor, or (pinned) host tensor
                ascii_d = ascii_u8.to(d, non_blocking=True)
            else:
                ascii_d = _to_device(ascii_u8, d)
            off_d = _to_device(np.asarray(ascii_off, dtype=np.int64), d)
            check(
                lib.nmb_pack_sequence(ptr(ascii_d), ptr(off_d), ptr(self.contig_start), ptr(self.contig_len),
                                      self.n_contigs, self.n_tiles, ptr(self.seq_records), ptr(self.nonacgt),
                                      _stream()),
                "nmb_pack_sequence",
            )
            # ascii_d / off_d go back to torch's caching allocator, whose reuse is ordered on this stream; the
            # synchronisation only matters to callers that touch the records from ANOTHER stream right away
            if sync:
                torch.cuda.current_stream().synchronize()
        self._view = NmbAssembly(ptr(self.seq_records), ptr(self.nonacgt), ptr(self.contig_start),
                                 ptr(self.contig_len), self.n_contigs, self.n_tiles)

    @classmethod
    def from_sequences(cls, contigs: Mapping[str, object], device=None) -> "DeviceAssembly":
        names = list(contigs.keys())
        seqs = [sequence_of(contigs[n]) for n in names]
        lengths = np.fromiter((len(s) for s in seqs), dtype=np.int64, count=len(seqs))
        off = np.zeros(len(seqs), dtype=np.int64)
        if len(seqs):
            off[1:] = np.cumsum(lengths)[:-1]
        total = int(lengths.sum())
        if total >= STAGE_MIN_BYTES:
            # large assemblies: the contig strings' own buffers are gathered straight into the pinned staging slots
            # (no "".join, no .encode copy): CPython keeps ASCII text as one byte per character
            dev = _require_cuda(device)
            st = _stager(dev)
            ptrs = _ascii_pointers(seqs) if st else None
            if ptrs is not None:
                piece_off = np.zeros(len(seqs) + 1, dtype=np.int64)
                np.cumsum(lengths, out=piece_off[1:])
                with torch.cuda.device(dev):
                    ascii_d = torch.empty(total, dtype=torch.uint8, device=dev)
                    check(lib.nmb_stager_gather(st, ptr(ascii_d), ptrs.ctypes.data, piece_off.ctypes.data, len(seqs),
                                                _stream()), "nmb_stager_gather")
                return cls(names, lengths, ascii_d, off, dev)
        buf = np.frombuffer("".join(seqs).encode("ascii"), dtype=np.uint8) if len(seqs) else np.zeros(0, np.uint8)
        if buf.size == 0:
            buf = np.zeros(1, dtype=np.uint8)
        return cls(names, lengths, buf, off, device)

    def view(self) -> NmbAssembly:
        return self._view

    def tile_span(self, contig_begin: int, contig_end: int) -> tuple[int, int]:
        """Tiles [begin, begin+count) that cover contigs [contig_begin, contig_end)."""
        if contig_end <= contig_begin:
            return 0, 0
        first = int(self.starts[contig_begin]) // _lib.TILE_BP
        last_pos = int(self.starts[contig_end - 1] + self.lengths[contig_end - 1]) - 1
        last = max(first, last_pos // _lib.TILE_BP)
        return first, last - first + 1

    @property
    def total_bp(self) -> int:
        return int(self.lengths.sum())


class DevicePileup:
    """Methylated / unmethylated x strand bit-planes per mod type (class records)."""

    def __init__(self, assembly: DeviceAssembly, n_modtypes: int, low: float, high: float):
        self.assembly = assembly
        self.n_modtypes = int(n_modtypes)
        self.low, self.high = float(low), float(high)
        self.class_records = torch.empty(self.n_modtypes * assembly.n_tiles * _lib.CLS_REC_WORDS,
                                         dtype=torch.int32, device=assembly.device)

    def clear(self) -> "DevicePileup":
        view = self.assembly.view()
        with torch.cuda.device(self.assembly.device):
            check(lib.nmb_clear_class_planes(C.byref(view), self.n_modtypes, ptr(self.class_records), _stream()),
                  "nmb_clear_class_planes")
        self._dups = None
        return self

    def add_columns(self, contig_id, position, strand, fraction_mod, mod_type=None, sync: bool = True) -> "DevicePileup":
        """OR rows into the class records (several tables, e.g. one per (bin, mod_type) as the reference partitions
        its pileup, find_motifs_bin.py:416).  Same columns as from_columns.  Rows that repeat a (contig, position,
        strand, mod type) are counted in `duplicate_rows` -- bit-planes collapse them, the reference counts them twice."""
        assembly, d = self.assembly, self.assembly.device

        def dev(a, dt):
            if a is None:
                return None
            if isinstance(a, torch.Tensor):
                return a.to(device=d, dtype=dt, non_blocking=True).contiguous()
            return _to_device(np.asarray(a).astype(_NP_OF[dt], copy=False), d)

        with torch.cuda.device(d):
            cid, pos = dev(contig_id, torch.int32), dev(position, torch.int64)
            st, fr, mt = dev(strand, torch.uint8), dev(fraction_mod, torch.float64), dev(mod_type, torch.uint8)
            n = int(cid.numel())
            for t in (pos, st, fr) + ((mt,) if mt is not None else ()):
                if int(t.numel()) != n:
                    raise ValueError("pileup columns differ in length")
            if getattr(self, "_dups", None) is None:
                self._dups = torch.zeros(1, dtype=torch.int64, device=d)
            view = assembly.view()
            check(
                lib.nmb_add_class_planes(ptr(cid), ptr(pos), ptr(st), ptr(mt), ptr(fr), n, self.low, self.high,
                                         C.byref(view), self.n_modtypes, ptr(self.class_records), ptr(self._dups),
                                         _stream()),
                "nmb_add_class_planes",
            )
            if sync:
                torch.cuda.current_stream().synchronize()
        return self

    @property
    def duplicate_rows(self) -> int:
        """Rows seen so far whose class bit was already set (synchronises)."""
        dups = getattr(self, "_dups", None)
        return 0 if dups is None else int(dups.item())

    def check_unique(self) -> "DevicePileup":
        n = self.duplicate_rows
        if n:
            import warnings

            warnings.warn(f"pileup holds {n} row(s) that repeat a (contig, position, strand, mod_type): they are counted "
                          "once here but once per row by the reference (np.isin keeps duplicates)", RuntimeWarning,
                          stacklevel=3)
        return self

    @classmethod
    def from_columns(cls, assembly: DeviceAssembly, contig_id, position, strand, fraction_mod, low, high,
                     mod_type=None, n_modtypes: int = 1) -> "DevicePileup":
        """contig_id int32 (index into the assembly, negative = ignore), position int64, strand uint8
        (0 '+', 1 '-'), fraction_mod float64, mod_type uint8 or None.  numpy arrays or device tensors."""
        self = cls(assembly, n_modtypes, low, high)
        self.clear().add_columns(contig_id, position, strand, fraction_mod, mod_type)
        return self.check_unique()

    @classmethod
    def from_compact(cls, assembly: DeviceAssembly, position, flags, percent_x100, contig_row_off, low, high,
                     n_modtypes: int = 1) -> "DevicePileup":
        """Rows grouped by contig in 7 bytes each: position int32, flags uint8 (strand | mod type << 1),
        percent_x100 uint16 (see threshold_keys); contig_row_off int64 [n_contigs + 1]."""
        self = cls(assembly, n_modtypes, low, high)
        d = assembly.device
        key_low, key_high = threshold_keys(low, high)

        def dev(a, dt):
            if isinstance(a, torch.Tensor):
                return a.to(device=d, dtype=dt, non_blocking=True).contiguous()
            return _to_device(np.asarray(a).astype(_NP_OF[dt], copy=False), d)

        with torch.cuda.device(d):
            pos, fl = dev(position, torch.int32), dev(flags, torch.uint8)
            key = dev(percent_x100, torch.uint16)
            off = dev(contig_row_off, torch.int64)
            n = int(pos.numel())
            if int(fl.numel()) != n or int(key.numel()) != n or int(off.numel()) != assembly.n_contigs + 1:
                raise ValueError("compact pileup columns differ in length")
            view = assembly.view()
            check(
                lib.nmb_build_class_planes_compact(ptr(pos), ptr(fl), ptr(key), ptr(off), n, key_low, key_high,
                                                   C.byref(view), self.n_modtypes, ptr(self.class_records), _stream()),
                "nmb_build_class_planes_compact",
            )
            torch.cuda.current_stream().synchronize()
        return self


def threshold_keys(low: float, high: float) -> tuple[int, int]:
    """Integer images of the reference's float64 classification on modkit's two-decimal grid.

    A pileup percentage printed with two decimals is k/100 for an integer key k in 0..10000; the reference
    turns it into fraction_mod = fl(fl(k/100)/100) (dataload.py:85) and tests >= high / <= low
    (find_motifs_bin.py:1308-1309).  Both tests are monotone in k, so they equal k >= key_high / k <= key_low
    with the keys found by evaluating the SAME float expression on all 10001 grid values."""
    k = np.arange(10001, dtype=np.float64)
    frac = (k / 100.0) / 100.0
    is_high, is_low = frac >= high, frac <= low
    key_high = int(np.argmax(is_high)) if is_high.any() else 10001
    key_low = int(len(k) - 1 - np.argmax(is_low[::-1])) if is_low.any() else -1
    if not (np.array_equal(is_high, np.arange(10001) >= key_high) and np.array_equal(is_low, np.arange(10001) <= key_low)):
        raise AssertionError("threshold tests are not monotone on the percent grid")  # cannot happen
    return key_low, key_high


def percent_keys(fraction_mod: np.ndarray) -> np.ndarray | None:
    """uint16 keys of fractions that sit exactly on modkit's two-decimal grid, else None."""
    f = np.asarray(fraction_mod, dtype=np.float64)
    k = np.rint(f * 10000.0)
    if not np.all((k >= 0) & (k <= 10000)):
        return None
    if not np.array_equal((k / 100.0) / 100.0, f):  # the exact float the reference's loader produces
        return None
    return k.astype(np.uint16)


def compact_rows(contig_id, position, strand, fraction_mod, mod_type=None, n_contigs: int = 1) -> dict | None:
    """Columns of DevicePileup.from_compact for a pileup whose percentages sit on modkit's two-decimal grid,
    or None when the pileup cannot be represented (off-grid fractions, positions >= 2^31, > 127 mod types).
    Rows of unknown contigs (negative id) are dropped; rows are grouped by contig (stable)."""
    key = percent_keys(fraction_mod)
    position = np.asarray(position, dtype=np.int64)
    if key is None or (len(position) and (position.max() >= 2**31 or position.min() < 0)):
        return None
    cid = np.asarray(contig_id, dtype=np.int64)
    mt = np.zeros(len(position), dtype=np.uint8) if mod_type is None else np.asarray(mod_type, dtype=np.uint8)
    if len(mt) and mt.max() > 127:
        mt = np.where(mt > 127, 127, mt)  # out-of-range types are ignored by the kernel (>= n_modtypes)
    strand = np.asarray(strand, dtype=np.uint8)
    flags = (strand & 1) | (mt << 1)
    # strand code 2 = neither '+' nor '-': dropped like the reference does.  Ids past the contig list are dropped too
    # (from_columns ignores them): grouped after the last contig, the kernel would take them for rows of that contig
    keep = (cid >= 0) & (cid < n_contigs) & (strand <= 1)
    if not keep.all():
        cid, position, flags, key = cid[keep], position[keep], flags[keep], key[keep]
    if len(cid) > 1 and np.any(cid[1:] < cid[:-1]):
        order = np.argsort(cid, kind="stable")
        cid, position, flags, key = cid[order], position[order], flags[order], key[order]
    off = np.zeros(n_contigs + 1, dtype=np.int64)
    np.cumsum(np.bincount(cid, minlength=n_contigs)[:n_contigs], out=off[1:])
    return dict(position=position.astype(np.int32), flags=flags, percent_x100=key, contig_row_off=off)


import os as _os

# Sibling runs in K2 (nmb_scan_count_siblings): the children of one search expansion -- consecutive motifs of a work
# item that differ at one common position -- are scored as one parent chain pair plus a four-base split of the parent's
# occurrences at that position, instead of one chain pair each.  Same counts (tests/test_gpu_siblings.py); motifs
# without siblings take the general path inside the same kernel.  NMB_FAMILIES=0 selects the general path everywhere.
FAMILIES = _os.environ.get("NMB_FAMILIES", "1") != "0"


BALANCED = _os.environ.get("NMB_BALANCED", "1") != "0"  # dynamic item scheduling in K2 (nmb_scan_count_balanced)
_COUNTERS: dict = {}


def _work_counter(device: torch.device) -> torch.Tensor:
    """The {next item, finished CTAs} pair of nmb_scan_count_balanced for the current stream of `device`: zeroed once,
    left at zero by every launch, so launches that are ordered on one stream share it."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    t = _COUNTERS.get(key)
    if t is None:
        t = _COUNTERS[key] = torch.zeros(2, dtype=torch.int32, device=device)
    return t


def make_jobs(n: int) -> np.ndarray:
    return np.zeros(n, dtype=_lib.JOB_DTYPE)


def choose_motifs_per_item(jobs: np.ndarray, sm_count: int) -> int:
    """Motifs per work item (tile x motif block): as many as the kernel takes (the tile copy, the barrier and the
    flush are paid per item), unless that leaves fewer than ~16 items per SM.  Measured on one B200 (3000 motifs x
    71 tiles, tools/kbench.py --mpi 32 28 30 24 16): 1.354 / 1.380 / 1.357 / 1.356 / 1.358 ms -- flat: the four
    resident CTAs of an SM share its ALUs, so neither the fill of the last round of the persistent grid nor the
    per-item overhead matters at this size."""
    motif_tiles = int((jobs["motif_count"].astype(np.int64) * jobs["tile_count"]).sum())
    target_items = 16 * sm_count  # ~4 items per resident CTA keeps the tail short
    mpi = motif_tiles // max(1, target_items)
    return int(min(_lib.MAX_MOTIFS_PER_ITEM, max(1, mpi)))


_SM_COUNT: dict[int, int] = {}


def sm_count(device: torch.device) -> int:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _SM_COUNT:
        _SM_COUNT[idx] = torch.cuda.get_device_properties(idx).multi_processor_count
    return _SM_COUNT[idx]


class MotifPrograms:
    """Motifs compiled on the device into forward / reverse-complement scan programs."""

    def __init__(self, motifs: Iterable, device: torch.device, strip: bool = True, mod_pos_override=None):
        packed = motifs if isinstance(motifs, np.ndarray) else pack_motifs(list(motifs), strip, mod_pos_override)
        self.packed = packed
        self.n = len(packed)
        self.max_len = int(packed["len"].max()) if self.n else 1
        self.device = device
        with torch.cuda.device(device):
            self.motifs_d = _to_device(packed.view(np.uint8).reshape(-1), device)
            self.programs = torch.empty(max(1, self.n) * lib.nmb_program_bytes(), dtype=torch.uint8, device=device)
            # per motif: link to the previous motif and the parent program of a sibling run (nmb_compile_motifs_siblings)
            self.siblings = torch.empty(max(128, int(lib.nmb_sibling_bytes(self.n))), dtype=torch.uint8, device=device)
            self.compile()

    def compile(self) -> None:
        """(Re)run the motif compiler on the device-resident motif records (one small launch, no copies): the scan
        programs and the sibling words and parent programs of K2's sibling runs."""
        check(lib.nmb_compile_motifs_siblings(ptr(self.motifs_d), self.n, ptr(self.programs), ptr(self.siblings),
                                              _stream()), "nmb_compile_motifs_siblings")


class PreparedJobs:
    """A job table resident on the device (item offsets filled in), reusable across launches."""

    def __init__(self, jobs: np.ndarray, device: torch.device, motifs_per_item: int | None = None):
        self.mpi = motifs_per_item or choose_motifs_per_item(jobs, sm_count(device))
        jobs, self.n_items = self.finalize(jobs, self.mpi)
        self.n_jobs = len(jobs)
        with torch.cuda.device(device):
            self.jobs_d = _to_device(jobs.view(np.uint8).reshape(-1), device)

    @staticmethod
    def finalize(jobs: np.ndarray, mpi: int) -> tuple[np.ndarray, int]:
        """Copy of the table with item_offset filled in for `mpi` motifs per item, and the number of items."""
        jobs = jobs.copy()
        items = jobs["tile_count"].astype(np.int64) * (-(-jobs["motif_count"].astype(np.int64) // mpi))
        offs = np.zeros(len(jobs), dtype=np.int64)
        offs[1:] = np.cumsum(items)[:-1]
        n_items = int(items.sum())
        if n_items >= 2**31:
            raise ValueError("too many work items for one launch")
        jobs["item_offset"] = offs.astype(np.int32)
        return jobs, n_items

    @classmethod
    def many(cls, tables: Sequence[np.ndarray], device: torch.device, motifs_per_item: int | None = None) -> list:
        """Several job tables through ONE host-to-device copy (the tables of a streamed run's launches)."""
        out, parts = [], []
        for t in tables:
            p = cls.__new__(cls)
            p.mpi = motifs_per_item or choose_motifs_per_item(t, sm_count(device))
            fin, p.n_items = cls.finalize(t, p.mpi)
            p.n_jobs = len(fin)
            parts.append(fin)
            out.append(p)
        if not out:
            return out
        with torch.cuda.device(device):
            blob = _to_device(np.concatenate(parts).view(np.uint8).reshape(-1), device)
        at = 0
        for p, fin in zip(out, parts):
            p.jobs_d = blob[at:at + fin.nbytes]
            at += fin.nbytes
        return out


def scan_count(assembly: DeviceAssembly, pileup: DevicePileup, programs: MotifPrograms, jobs,
               n_out_rows: int, motifs_per_item: int | None = None, contig_group: torch.Tensor | None = None,
               grid_ctas: int = 0, out: torch.Tensor | None = None) -> torch.Tensor:
    """Launch K2 for a batch of jobs (a numpy job table, or PreparedJobs already on the device).  Returns the
    int64 device tensor [n_out_rows, 4] (n_mod '+', n_nomod '+', n_mod '-', n_nomod '-'); nothing is synchronised."""
    d = assembly.device
    with torch.cuda.device(d):
        prepared = jobs if isinstance(jobs, PreparedJobs) else PreparedJobs(jobs, d, motifs_per_item)
        if out is None:
            out = torch.zeros((n_out_rows, 4), dtype=torch.int64, device=d)
        view = assembly.view()
        if FAMILIES and prepared.mpi >= 2 and programs.n >= 2:  # sibling runs need blocks of two or more motifs
            check(
                lib.nmb_scan_count_siblings(C.byref(view), ptr(pileup.class_records), ptr(programs.programs),
                                            ptr(programs.siblings), programs.n, ptr(prepared.jobs_d), prepared.n_jobs,
                                            prepared.n_items, prepared.mpi, programs.max_len, ptr(contig_group),
                                            ptr(out), grid_ctas, ptr(_work_counter(d)) if BALANCED else None,
                                            _stream()),
                "nmb_scan_count_siblings",
            )
            return out
        if BALANCED:  # items drawn from a device counter (one pair per device and stream, re-armed by the kernel)
            check(
                lib.nmb_scan_count_balanced(C.byref(view), ptr(pileup.class_records), ptr(programs.programs),
                                            ptr(prepared.jobs_d), prepared.n_jobs, prepared.n_items, prepared.mpi,
                                            programs.max_len, ptr(contig_group), ptr(out), grid_ctas,
                                            ptr(_work_counter(d)), _stream()),
                "nmb_scan_count_balanced",
            )
            return out
        check(
            lib.nmb_scan_count(C.byref(view), ptr(pileup.class_records), ptr(programs.programs), ptr(prepared.jobs_d),
                               prepared.n_jobs, prepared.n_items, prepared.mpi, programs.max_len, ptr(contig_group),
                               ptr(out), grid_ctas, _stream()),
            "nmb_scan_count",
        )
        # a temporary job table goes back to torch's caching allocator; reuse is ordered on this same stream
    return out
