"""Loaders and pileup filters of the scoring path (mirror of nanomotif/dataload.py and fasta.py).

    load_pileup                              nanomotif/dataload.py:72-100
    filter_pileup                            nanomotif/dataload.py:191-200
    filter_pileup_minimummod_frequency       nanomotif/dataload.py:202-226
    filter_pileup_adjacency_filter           nanomotif/dataload.py:228-247
    load_fasta                               nanomotif/fasta.py:35-49

The text is parsed on the host (pyarrow CSV reader); the filters run as CUDA kernels on the columnar
arrays and return a filtered `PileupTable`.  Row order: the input order is kept (the reference returns
the adjacency-filtered rows grouped by (contig, strand) and sorted by position; nothing downstream
depends on that order).
"""
from __future__ import annotations

import numpy as np
import torch

from ._lib import check, lib, ptr
from .device import _require_cuda, _stream, _to_device, _to_device_narrow
from .pileup import PileupTable, strand_codes

# bedMethyl columns kept by the reference (1-based 1,2,4,6,10,11; dataload.py:84)
_BED_COLUMNS = {0: "contig", 1: "position", 3: "mod_type", 5: "strand", 9: "Nvalid_cov", 10: "percent_modified",
                11: "n_mod", 16: "n_diff"}


def load_pileup(path: str, with_counts: bool = False) -> PileupTable:
    """modkit pileup (18-column bedMethyl, tab separated, optionally gzip) -> PileupTable with
    fraction_mod = column 11 / 100 (dataload.py:85).  with_counts keeps n_mod (column 12) and n_diff
    (column 17) for the methylation-pattern table."""
    import pyarrow as pa
    import pyarrow.csv as pacsv

    names = [f"column_{i + 1}" for i in range(18)]
    types = {"column_1": pa.string(), "column_2": pa.int64(), "column_4": pa.string(), "column_6": pa.string(),
             "column_10": pa.int64(), "column_11": pa.float64(), "column_12": pa.int64(), "column_17": pa.int64()}
    keep = ["column_1", "column_2", "column_4", "column_6", "column_10", "column_11"]
    if with_counts:
        keep += ["column_12", "column_17"]
    table = pacsv.read_csv(
        path,
        read_options=pacsv.ReadOptions(column_names=names),
        parse_options=pacsv.ParseOptions(delimiter="\t"),
        convert_options=pacsv.ConvertOptions(column_types=types, include_columns=keep, null_values=["NA", "null"],
                                             strings_can_be_null=True),
    )
    if table.num_rows == 0:
        raise SystemExit("Pileup is empty after initial load")  # the reference prints and sys.exit(1)s
    col = lambda n: table.column(n).to_numpy(zero_copy_only=False)
    extra = {}
    if with_counts:
        extra = {"n_mod": col("column_12").astype(np.int64), "n_diff": col("column_17").astype(np.int64)}
    return PileupTable(col("column_1").astype(object), col("column_2").astype(np.int64), col("column_6").astype(object),
                       col("column_11").astype(np.float64) / 100, col("column_4").astype(object),
                       col("column_10").astype(np.int64), extra)


def load_fasta(path: str, trim_names: bool = False, trim_character: str = " ") -> dict[str, str]:
    """FASTA (optionally gzip) -> {name: upper-case sequence} (fasta.py:35-49 + seq.py:55)."""
    import gzip

    opener = gzip.open if str(path).endswith(".gz") else open
    out, name, parts = {}, None, []
    with opener(path, "rt") as f:
        for line in f:
            if line.startswith(">"):
                if name is not None:
                    out[name] = "".join(parts).upper()
                name = line[1:].strip()
                name = name.split(trim_character)[0] if trim_names else (name.split() or [""])[0]
                if name in out:
                    raise ValueError(f"duplicate contig name {name!r} in {path}")
                parts = []
            else:
                parts.append(line.strip())
    if name is not None:
        out[name] = "".join(parts).upper()
    return out


def _codes(values) -> tuple[np.ndarray, np.ndarray]:
    """Dense int32 codes (order of first appearance is irrelevant) and the unique values."""
    uniq, inv = np.unique(np.asarray(values).astype(str), return_inverse=True)
    return inv.astype(np.int32), uniq


def _mask_to_host(keep: torch.Tensor) -> np.ndarray:
    return keep.cpu().numpy().astype(bool)


def filter_pileup(pileup, min_modtype_fraction: float = 0.3, min_coverage: int = 5, device=None) -> PileupTable:
    """Keep positions with Nvalid_cov > min_coverage (dataload.py:191-200; min_modtype_fraction is
    accepted and ignored exactly like the reference)."""
    t = PileupTable.from_frame(pileup)
    d = _require_cuda(device)
    n = len(t)
    with torch.cuda.device(d):
        cov = _to_device(np.asarray(t.Nvalid_cov, dtype=np.int64), d)
        keep = torch.empty(n, dtype=torch.uint8, device=d)
        check(lib.nmb_filter_coverage(ptr(cov), n, int(min_coverage), ptr(keep), _stream()), "nmb_filter_coverage")
    return t.take(_mask_to_host(keep))


def filter_pileup_minimummod_frequency(pileup, methylation_threshold: float = 0.7, min_mod_frequency: float = 0.0001,
                                       min_mods_pr_contig: int = 50, device=None) -> PileupTable:
    """Keep contig_mods with enough methylated positions (dataload.py:202-226)."""
    t = PileupTable.from_frame(pileup)
    d = _require_cuda(device)
    n = len(t)
    cid, contigs = _codes(t.contig)
    mid, mods = _codes(t.mod_type)
    group = (cid.astype(np.int64) * len(mods) + mid).astype(np.int32)
    n_groups = max(1, len(contigs) * len(mods))
    with torch.cuda.device(d):
        g = _to_device(group, d)
        fr = _to_device(np.asarray(t.fraction_mod, dtype=np.float64), d)
        counts = torch.empty(2 * n_groups, dtype=torch.int64, device=d)
        keep = torch.empty(n, dtype=torch.uint8, device=d)
        check(lib.nmb_filter_min_mod_frequency(ptr(g), ptr(fr), n, n_groups, float(methylation_threshold),
                                               float(min_mod_frequency), int(min_mods_pr_contig), ptr(counts),
                                               ptr(keep), _stream()), "nmb_filter_min_mod_frequency")
    return t.take(_mask_to_host(keep))


def filter_pileup_adjacency_filter(pileup, methylation_threshold: float = 0.7, adjacency_distance: int = 8,
                                   device=None) -> PileupTable:
    """Drop a methylated position when a larger fraction exists within +-adjacency_distance on the
    same (contig, strand), over all mod types (dataload.py:228-247)."""
    t = PileupTable.from_frame(pileup)
    d = _require_cuda(device)
    n = len(t)
    cid, _ = _codes(t.contig) if t.contig is not None else (np.zeros(n, dtype=np.int32), None)
    pos = np.asarray(t.position, dtype=np.int64)
    order = None
    if n > 1 and not np.all((cid[1:] > cid[:-1]) | ((cid[1:] == cid[:-1]) & (pos[1:] >= pos[:-1]))):
        order = np.lexsort((pos, cid))  # the kernel needs (contig, position) order
    sel = (lambda a: a[order]) if order is not None else (lambda a: a)
    with torch.cuda.device(d):
        c_d = _to_device(sel(cid), d)
        p_d = _to_device(sel(pos), d)
        s_d = _to_device(sel(strand_codes(t.strand)), d)
        f_d = _to_device(sel(np.asarray(t.fraction_mod, dtype=np.float64)), d)
        keep = torch.empty(n, dtype=torch.uint8, device=d)
        flag = torch.zeros(1, dtype=torch.int32, device=d)
        check(lib.nmb_filter_adjacency(ptr(c_d), ptr(p_d), ptr(s_d), ptr(f_d), n, float(methylation_threshold),
                                       int(adjacency_distance), ptr(keep), ptr(flag), _stream()), "nmb_filter_adjacency")
        if int(flag.item()):
            raise RuntimeError("nmb_filter_adjacency: rows were not sorted by (contig, position)")
    k = _mask_to_host(keep)
    if order is not None:
        inv = np.empty(n, dtype=bool)
        inv[order] = k
        k = inv
    return t.take(k)


# ---------------------------------------------------------------------------------------------
# device ingest: bedMethyl text -> columns -> filters -> class planes without leaving the GPU (K6)
# ---------------------------------------------------------------------------------------------

_FNV_OFFSET, _FNV_PRIME, _U64 = 0xCBF29CE484222325, 0x100000001B3, (1 << 64) - 1


def _fnv1a64(b: bytes) -> int:
    h = _FNV_OFFSET
    for c in b:
        h = ((h ^ c) * _FNV_PRIME) & _U64
    return h


def _fnv1a64_many(enc) -> np.ndarray:
    """_fnv1a64 of every byte string of a list, one numpy pass per byte position instead of a Python step per byte
    (an assembly has tens of thousands of contig names; uint64 arithmetic wraps like the & _U64 above)."""
    n = len(enc)
    lens = np.fromiter((len(b) for b in enc), dtype=np.int64, count=n)
    h = np.full(n, _FNV_OFFSET, dtype=np.uint64)
    if n == 0 or int(lens.max()) == 0:
        return h
    start = np.zeros(n, dtype=np.int64)
    np.cumsum(lens[:-1], out=start[1:])
    flat = np.frombuffer(b"".join(enc), dtype=np.uint8)
    prime = np.uint64(_FNV_PRIME)
    for j in range(int(lens.max())):
        live = np.flatnonzero(lens > j)
        h[live] = (h[live] ^ flat[start[live] + j].astype(np.uint64)) * prime
    return h


def _name_table(names, device):
    """Device lookup table of nmb_bed_parse: hashes ascending, ids, name bytes by rank."""
    enc = [str(n).encode() for n in names]
    hashes = _fnv1a64_many(enc)
    order = np.argsort(hashes, kind="stable")
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    np.cumsum([len(enc[i]) for i in order], out=off[1:])
    blob = np.frombuffer(b"".join(enc[i] for i in order) or b"\0", dtype=np.uint8)
    return (_to_device(hashes[order].view(np.int64), device), _to_device(order.astype(np.int32), device),
            _to_device(off, device), _to_device(blob, device))


def _modtype_keys(mod_types) -> np.ndarray:
    keys = []
    for m in mod_types:
        b = str(m).encode()
        if not 1 <= len(b) <= 8:
            raise ValueError(f"mod type code {m!r} must be 1..8 bytes")
        keys.append(int.from_bytes(b, "big"))
    return np.array(keys, dtype=np.uint64)


class DeviceRows:
    """Pileup rows as device columns (what nmb_bed_parse writes).  contig_id indexes `contig_names`,
    mod_type indexes `mod_types`; strand 0 '+', 1 '-'."""

    COLUMNS = ("contig_id", "position", "strand", "mod_type", "Nvalid_cov", "fraction_mod", "percent_x100", "n_mod", "n_diff")

    def __init__(self, contig_names, mod_types, device, **cols):
        self.contig_names, self.mod_types, self.device = list(contig_names), tuple(mod_types), device
        for k in self.COLUMNS:
            setattr(self, k, cols.get(k))

    def __len__(self) -> int:
        return int(self.position.numel())

    def take_mask(self, keep: torch.Tensor) -> "DeviceRows":
        """Rows with keep == 1 (a 0/1 uint8 mask), in order (nmb_index_bytes + nmb_gather_rows)."""
        n = len(self)
        with torch.cuda.device(self.device):
            scratch = torch.empty((n + 4095) // 4096 + 2, dtype=torch.int64, device=self.device)
            n_out = torch.zeros(1, dtype=torch.int64, device=self.device)
            check(lib.nmb_index_bytes(ptr(keep), n, 1, ptr(scratch), None, 0, ptr(n_out), _stream()), "nmb_index_bytes")
            m = int(n_out.item())
            index = torch.empty(max(m, 1), dtype=torch.int64, device=self.device)
            if m:
                check(lib.nmb_index_bytes(ptr(keep), n, 1, ptr(scratch), ptr(index), m, ptr(n_out), _stream()),
                      "nmb_index_bytes")
            cols = {}
            for k in self.COLUMNS:
                src = getattr(self, k)
                if src is None:
                    continue
                dst = torch.empty(m, dtype=src.dtype, device=self.device)
                check(lib.nmb_gather_rows(ptr(src), src.element_size(), ptr(index), m, ptr(dst), _stream()),
                      "nmb_gather_rows")
                cols[k] = dst
        return DeviceRows(self.contig_names, self.mod_types, self.device, **cols)

    def to_table(self) -> PileupTable:
        """Host copy with names restored (parity checks, hand-over to host code)."""
        names = np.array(self.contig_names + ["?"], dtype=object)
        mods = np.array(list(self.mod_types) + ["?"], dtype=object)
        cid = self.contig_id.cpu().numpy()
        mt = self.mod_type.cpu().numpy().astype(np.int64)
        extra = {k: getattr(self, k).cpu().numpy() for k in ("n_mod", "n_diff", "percent_x100") if getattr(self, k) is not None}
        return PileupTable(names[np.where(cid >= 0, cid, len(self.contig_names))], self.position.cpu().numpy(),
                           np.array(["+", "-", "."], dtype=object)[self.strand.cpu().numpy()],
                           self.fraction_mod.cpu().numpy(), mods[np.minimum(mt, len(self.mod_types))],
                           self.Nvalid_cov.cpu().numpy(), extra)

    # ---- the three loader filters, device to device (dataload.py:191-247) ----
    def filter_coverage(self, min_coverage: int = 5) -> "DeviceRows":
        n = len(self)
        with torch.cuda.device(self.device):
            keep = torch.empty(n, dtype=torch.uint8, device=self.device)
            check(lib.nmb_filter_coverage(ptr(self.Nvalid_cov), n, int(min_coverage), ptr(keep), _stream()),
                  "nmb_filter_coverage")
        return self.take_mask(keep)

    def filter_min_mod_frequency(self, methylation_threshold: float = 0.7, min_mod_frequency: float = 0.0001,
                                 min_mods_pr_contig: int = 50) -> "DeviceRows":
        n, M = len(self), max(1, len(self.mod_types))
        n_groups = max(1, len(self.contig_names) * M)
        with torch.cuda.device(self.device):
            cid, mt = self.contig_id, self.mod_type.to(torch.int32)
            group = torch.where((cid >= 0) & (mt < M), cid * M + mt, torch.full_like(cid, -1))  # index arithmetic only
            counts = torch.empty(2 * n_groups, dtype=torch.int64, device=self.device)
            keep = torch.empty(n, dtype=torch.uint8, device=self.device)
            check(lib.nmb_filter_min_mod_frequency(ptr(group), ptr(self.fraction_mod), n, n_groups,
                                                   float(methylation_threshold), float(min_mod_frequency),
                                                   int(min_mods_pr_contig), ptr(counts), ptr(keep), _stream()),
                  "nmb_filter_min_mod_frequency")
        return self.take_mask(keep)

    def filter_adjacency(self, methylation_threshold: float = 0.7, adjacency_distance: int = 8) -> "DeviceRows":
        """Rows must be sorted by (contig, position), as modkit writes them."""
        n = len(self)
        with torch.cuda.device(self.device):
            keep = torch.empty(n, dtype=torch.uint8, device=self.device)
            flag = torch.zeros(1, dtype=torch.int32, device=self.device)
            check(lib.nmb_filter_adjacency(ptr(self.contig_id), ptr(self.position), ptr(self.strand), ptr(self.fraction_mod),
                                           n, float(methylation_threshold), int(adjacency_distance), ptr(keep), ptr(flag),
                                           _stream()), "nmb_filter_adjacency")
            if int(flag.item()):
                raise ValueError("filter_adjacency: rows are not sorted by (contig, position)")
        return self.take_mask(keep)

    def class_planes(self, assembly, low: float = 0.3, high: float = 0.7):
        """DevicePileup of these rows; `assembly.names` must be the `contig_names` the rows were parsed with."""
        from .device import DevicePileup

        if list(assembly.names) != self.contig_names:
            raise ValueError("rows were parsed against a different contig list than the assembly's")
        rows = self
        with torch.cuda.device(self.device):
            if bool((self.strand > 1).any()):
                rows = self.take_mask((self.strand < 2).to(torch.uint8))
        return DevicePileup.from_columns(assembly, rows.contig_id, rows.position, rows.strand, rows.fraction_mod, low, high,
                                         rows.mod_type, n_modtypes=max(1, len(self.mod_types)))



# ---------------------------------------------------------------------------------------------
# host TABLE -> device rows: the frames nanomotif hands to its workers (find_motifs_bin.py:399-427) are
# polars frames = Arrow buffers.  The numeric columns go to the device as they are, the three string
# columns (contig, strand, mod_type) as their raw offsets + bytes buffers and are resolved to ids by
# nmb_lookup_strings -- no per-row host work, no Python strings.
# ---------------------------------------------------------------------------------------------
def _frame_column(frame, name):
    """Column `name` of a pyarrow Table / polars / pandas frame / PileupTable / mapping, or None."""
    if isinstance(frame, PileupTable):
        return getattr(frame, name, None)
    if isinstance(frame, dict):
        return frame.get(name)
    cols = getattr(frame, "column_names", None) or getattr(frame, "columns", None)
    if cols is not None and name not in list(cols):
        return None
    if hasattr(frame, "get_column"):  # polars
        return frame.get_column(name)
    if hasattr(frame, "column") and hasattr(frame, "num_rows"):  # pyarrow.Table
        return frame.column(name)
    return frame[name]  # pandas


def _string_column(col, ints_are_codes: bool = True):
    """A string column as ("utf8", offsets int32/int64 [n + 1], bytes uint8) -- zero-copy views of Arrow buffers --
    or ("dict", codes int32 [n], [values]) for dictionary / categorical columns and for plain numpy / pandas object
    columns when pyarrow is not installed."""
    try:
        import pyarrow as pa
    except ImportError:  # pragma: no cover - pyarrow is in the image
        pa = None
    if pa is not None:
        if hasattr(col, "to_arrow"):  # polars Series
            col = col.to_arrow()
        if isinstance(col, pa.ChunkedArray):
            col = col.chunk(0) if col.num_chunks == 1 else col.combine_chunks()
        if not isinstance(col, pa.Array):
            a = col.to_numpy() if hasattr(col, "to_numpy") and not isinstance(col, np.ndarray) else np.asarray(col)
            if a.dtype.kind in "iub":
                if ints_are_codes:
                    return "codes", a, None
                uniq, inv = np.unique(a, return_inverse=True)
                return "dict", inv.astype(np.int32), [str(u) for u in uniq]
            try:
                col = pa.array(a, type=pa.large_string())
            except (pa.ArrowInvalid, pa.ArrowTypeError, pa.ArrowNotImplementedError):
                col = pa.array(a.astype(str).astype(object), type=pa.large_string())
        t = col.type
        if pa.types.is_dictionary(t):
            return "dict", col.indices.to_numpy(zero_copy_only=False).astype(np.int32), [str(v) for v in col.dictionary.to_pylist()]
        if not (pa.types.is_string(t) or pa.types.is_large_string(t)):
            col = col.cast(pa.large_string())  # string_view, ...
            t = col.type
        n = len(col)
        bufs = col.buffers()
        odt = np.int64 if pa.types.is_large_string(t) else np.int32
        off = np.frombuffer(bufs[1], dtype=odt)[col.offset:col.offset + n + 1] if n else np.zeros(1, odt)
        data = np.frombuffer(bufs[2], dtype=np.uint8) if bufs[2] is not None and bufs[2].size else np.zeros(1, np.uint8)
        lo, hi = int(off[0]), int(off[-1])
        if lo:  # a sliced array: rebase, ship only the bytes in use
            off = off - lo
        return "utf8", off, data[lo:max(hi, lo + 1)]
    a = np.asarray(col)
    if a.dtype.kind in "iub" and ints_are_codes:
        return "codes", a, None
    uniq, inv = np.unique(a.astype(str), return_inverse=True)
    return "dict", inv.astype(np.int32), [str(u) for u in uniq]


def _numeric_column(col, dtype):
    if hasattr(col, "to_arrow"):
        col = col.to_arrow()
    if hasattr(col, "combine_chunks") and hasattr(col, "num_chunks"):
        col = col.chunk(0) if col.num_chunks == 1 else col.combine_chunks()
    if hasattr(col, "to_numpy") and not isinstance(col, np.ndarray):
        try:
            col = col.to_numpy(zero_copy_only=False)
        except TypeError:
            col = col.to_numpy()
    return np.ascontiguousarray(np.asarray(col), dtype=dtype)


def _lookup_ids(kind, a, b, names, missing, out_dtype, device, table_cache=None):
    """Device ids of a string column (see _string_column) against `names`."""
    n_names = len(names)
    if kind == "codes":  # already integer codes (strand 0/1, mod type index)
        return _to_device(np.asarray(a).astype({torch.int32: np.int32, torch.uint8: np.uint8}[out_dtype], copy=False), device)
    if kind == "dict":
        index = {str(v): i for i, v in enumerate(names)}
        lut = np.array([index.get(v, missing) for v in b] + [missing], dtype=np.int64)
        codes = _to_device(a, device).long()
        codes = torch.where(codes < 0, torch.full_like(codes, len(b)), codes)  # null -> missing
        return torch.from_numpy(lut).to(device)[codes].to(out_dtype)
    key = ("names", tuple(names)) if table_cache is not None else None
    tab = table_cache.get(key) if table_cache is not None else None
    if tab is None:
        tab = _name_table(names, device)
        if table_cache is not None:
            table_cache[key] = tab
    h, ids, noff, blob = tab
    n = len(a) - 1
    off_d = None
    if a.dtype == np.int64 and n and int(a[-1]) < 2**31:  # large_utf8 offsets that fit int32: half the PCIe bytes
        off_d = _to_device_narrow(a, device)
    if off_d is None:
        off_d = _to_device(a, device)
    data_d = _to_device(b, device)
    out = torch.empty(n, dtype=out_dtype, device=device)
    check(lib.nmb_lookup_strings(ptr(data_d), ptr(off_d), off_d.element_size(), n, ptr(h), ptr(ids), ptr(noff), ptr(blob),
                                 n_names, missing, ptr(out), out.element_size(), _stream()), "nmb_lookup_strings")
    return out


def rows_from_table(frame, contig_names, mod_types=("a", "m", "21839"), device=None, table_cache=None,
                    with_coverage: bool = True) -> "DeviceRows":
    """A reference-shaped pileup table (columns contig: str, position: i64, strand: '+'/'-', mod_type: str,
    fraction_mod: f64 [, Nvalid_cov: i64]; pyarrow Table, polars / pandas frame, PileupTable or dict of arrays) ->
    DeviceRows.  contig_id = index into contig_names (-1 unknown), strand 0 '+' / 1 '-' / 2 anything else (modkit's
    '.'), mod_type = index into mod_types (255 unknown; a table without the column is all type 0)."""
    d = _require_cuda(device)
    contig_names = list(contig_names)
    with torch.cuda.device(d):
        pos_c, frac_c, strand_c = (_frame_column(frame, k) for k in ("position", "fraction_mod", "strand"))
        if pos_c is None:
            raise KeyError("pileup has no 'position' column")
        if strand_c is None or frac_c is None:
            raise KeyError("pileup needs 'strand' and 'fraction_mod' columns")
        pos_h = _numeric_column(pos_c, np.int64)
        pos = _to_device_narrow(pos_h, d)  # positions fit int32 (contig coordinates); widened again on the device
        pos = _to_device(pos_h, d) if pos is None else pos.to(torch.int64)
        frac = _to_device(_numeric_column(frac_c, np.float64), d)
        n = int(pos.numel())
        strand = _lookup_ids(*_string_column(strand_c), ["+", "-"], 2, torch.uint8, d, table_cache)
        contig_c = _frame_column(frame, "contig")
        if contig_c is None:
            if len(contig_names) != 1:
                raise KeyError("pileup has no 'contig' column but several contigs were given")
            cid = torch.zeros(n, dtype=torch.int32, device=d)
        else:
            cid = _lookup_ids(*_string_column(contig_c), contig_names, -1, torch.int32, d, table_cache)
        mt_c = _frame_column(frame, "mod_type")
        if mt_c is None:
            mt = torch.zeros(n, dtype=torch.uint8, device=d)
        else:
            # integer mod-type columns hold modkit codes such as 21839, not indices
            mt = _lookup_ids(*_string_column(mt_c, ints_are_codes=False), [str(m) for m in mod_types], 255, torch.uint8,
                             d, table_cache)
        cov_c = _frame_column(frame, "Nvalid_cov") if with_coverage else None
        cov = None if cov_c is None else _to_device(_numeric_column(cov_c, np.int64), d)
        for t in (frac, strand, cid, mt):
            if int(t.numel()) != n:
                raise ValueError("pileup columns differ in length")
    return DeviceRows(contig_names, mod_types, d, contig_id=cid, position=pos, strand=strand, mod_type=mt,
                      fraction_mod=frac, Nvalid_cov=cov)


def parse_bedmethyl(data, contig_names, mod_types=("a", "m", "21839"), with_counts: bool = False, device=None,
                    keep_unknown_contigs: bool = False) -> DeviceRows:
    """modkit bedMethyl TEXT (bytes, uint8 array / tensor on host or device) -> DeviceRows, parsed on the GPU.

    Same columns and arithmetic as load_pileup (dataload.py:72-100): contig, position, mod_type, strand,
    Nvalid_cov and fraction_mod = column 11 / 100.  Empty lines are skipped, lines with fewer than 18
    tab-separated fields raise.  Rows of contigs outside `contig_names` are dropped unless asked for."""
    d = _require_cuda(device)
    if isinstance(data, (bytes, bytearray, memoryview)):
        data = np.frombuffer(data, dtype=np.uint8)
    with torch.cuda.device(d):
        text = data.to(d, non_blocking=True) if isinstance(data, torch.Tensor) else _to_device(np.asarray(data, dtype=np.uint8), d)
        n_bytes = int(text.numel())
        scratch = torch.empty((n_bytes + 4095) // 4096 + 2, dtype=torch.int64, device=d)
        n_nl = torch.zeros(1, dtype=torch.int64, device=d)
        check(lib.nmb_index_bytes(ptr(text), n_bytes, 10, ptr(scratch), None, 0, ptr(n_nl), _stream()), "nmb_index_bytes")
        n_newlines = int(n_nl.item())
        newline_pos = torch.empty(max(n_newlines, 1), dtype=torch.int64, device=d)
        if n_newlines:
            check(lib.nmb_index_bytes(ptr(text), n_bytes, 10, ptr(scratch), ptr(newline_pos), n_newlines, ptr(n_nl),
                                      _stream()), "nmb_index_bytes")
        ends_with_newline = n_bytes > 0 and int(text[-1].item()) == 10
        n_lines = n_newlines + (1 if n_bytes > 0 and not ends_with_newline else 0)
        names = list(contig_names)
        h, ids, off, blob = _name_table(names, d)
        keys = _to_device(_modtype_keys(mod_types).view(np.int64), d) if len(mod_types) else None
        new = lambda dt: torch.empty(n_lines, dtype=dt, device=d)
        cols = dict(contig_id=new(torch.int32), position=new(torch.int64), strand=new(torch.uint8), mod_type=new(torch.uint8),
                    Nvalid_cov=new(torch.int64), fraction_mod=new(torch.float64), percent_x100=new(torch.uint16))
        if with_counts:
            cols.update(n_mod=new(torch.int64), n_diff=new(torch.int64))
        status = torch.zeros(4, dtype=torch.int32, device=d)
        check(lib.nmb_bed_parse(ptr(text), n_bytes, ptr(newline_pos), n_lines, ptr(h), ptr(ids), ptr(off), ptr(blob),
                                len(names), ptr(keys), len(mod_types), ptr(cols["contig_id"]), ptr(cols["position"]),
                                ptr(cols["strand"]), ptr(cols["mod_type"]), ptr(cols["Nvalid_cov"]), ptr(cols["fraction_mod"]),
                                ptr(cols["percent_x100"]), ptr(cols.get("n_mod")), ptr(cols.get("n_diff")), ptr(status),
                                _stream()), "nmb_bed_parse")
        malformed, empty, _notnum, unknown = (int(v) for v in status.cpu().tolist())
        if malformed:
            raise ValueError(f"bedMethyl: {malformed} line(s) with fewer than 18 tab-separated columns")
        rows = DeviceRows(names, mod_types, d, **cols)
        if empty or (unknown and not keep_unknown_contigs):
            floor = -1 if keep_unknown_contigs else 0
            rows = rows.take_mask((rows.contig_id >= floor).to(torch.uint8))
    return rows


def bgzf_blocks(data) -> dict | None:
    """Block table of a BGZF file (SAM spec 4.1: gzip members whose extra field carries 'BC' + BSIZE), or None
    when `data` is not BGZF (plain gzip, text).  Only the 18-byte headers and 8-byte trailers are read."""
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    n = len(buf)
    in_off, in_len, out_len, crc = [], [], [], []
    at = 0
    while at < n:
        if at + 18 > n or buf[at] != 31 or buf[at + 1] != 139 or buf[at + 2] != 8 or not (buf[at + 3] & 4):
            return None
        xlen = int(buf[at + 10]) | (int(buf[at + 11]) << 8)
        bsize, x = None, at + 12
        while x + 4 <= at + 12 + xlen:  # extra subfields: SI1 SI2 SLEN(2) data
            slen = int(buf[x + 2]) | (int(buf[x + 3]) << 8)
            if buf[x] == 66 and buf[x + 1] == 67 and slen == 2:
                bsize = (int(buf[x + 4]) | (int(buf[x + 5]) << 8)) + 1
            x += 4 + slen
        if bsize is None or at + bsize > n or bsize < 12 + xlen + 8:
            return None
        tail = at + bsize - 8
        in_off.append(at + 12 + xlen)
        in_len.append(tail - (at + 12 + xlen))
        crc.append(int.from_bytes(buf[tail:tail + 4].tobytes(), "little"))
        out_len.append(int.from_bytes(buf[tail + 4:tail + 8].tobytes(), "little"))
        at += bsize
    out_off = np.zeros(len(out_len) + 1, dtype=np.int64)
    np.cumsum(out_len, out=out_off[1:])
    return dict(in_off=np.array(in_off, dtype=np.int64), in_len=np.array(in_len, dtype=np.int32),
                out_off=out_off[:-1].copy(), out_len=np.array(out_len, dtype=np.int32),
                crc=np.array(crc, dtype=np.uint32), total=int(out_off[-1]))


def inflate_bgzf_device(data, device=None, verify_crc: bool = True) -> torch.Tensor:
    """The inflated bytes of a BGZF file as a device uint8 tensor (K7: one thread per 64 KB block)."""
    d = _require_cuda(device)
    blocks = bgzf_blocks(data)
    if blocks is None:
        raise ValueError("not a BGZF file (no 'BC' extra subfield); use gzip on the host")
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    nb = len(blocks["in_len"])
    with torch.cuda.device(d):
        comp = _to_device(buf, d)
        out = torch.empty(max(1, blocks["total"]), dtype=torch.uint8, device=d)
        status = torch.zeros(max(1, nb), dtype=torch.int32, device=d)
        crc = _to_device(blocks["crc"].view(np.int32), d) if verify_crc else None
        # named, so that the block table stays allocated until the launch has been enqueued
        in_off, in_len = _to_device(blocks["in_off"], d), _to_device(blocks["in_len"], d)
        out_off, out_len = _to_device(blocks["out_off"], d), _to_device(blocks["out_len"], d)
        check(lib.nmb_bgzf_inflate(ptr(comp), ptr(in_off), ptr(in_len), ptr(out_off), ptr(out_len), ptr(crc),
                                   nb, ptr(out), ptr(status), _stream()), "nmb_bgzf_inflate")
        bad = torch.nonzero(status[:nb]).view(-1)
        if int(bad.numel()):
            b = int(bad[0].item())
            raise ValueError(f"BGZF block {b} of {nb} failed to inflate (status {int(status[b].item())})")
    return out[:blocks["total"]]


def load_pileup_device(path: str, contig_names, mod_types=("a", "m", "21839"), with_counts: bool = False, device=None,
                       keep_unknown_contigs: bool = False) -> DeviceRows:
    """load_pileup with inflate and parse on the GPU: a bgzip-compressed pileup goes to the device compressed
    (K7), plain text as it is; only a non-BGZF gzip file is inflated on the host."""
    with open(path, "rb") as f:
        data = f.read()
    if data[:2] == b"\x1f\x8b":
        if bgzf_blocks(data) is not None:
            data = inflate_bgzf_device(data, device)
        else:
            import gzip

            data = gzip.decompress(data)
    if len(data) == 0:
        raise SystemExit("Pileup is empty after initial load")  # dataload.py:89-91
    return parse_bedmethyl(data, contig_names, mod_types, with_counts, device, keep_unknown_contigs)


def load_contigs_pileup_bgzip(path: str, contigs, mod_types=("a", "m", "21839"), with_counts: bool = False,
                              device=None) -> DeviceRows:
    """dataload.load_contigs_pileup_bgzip (dataload.py:102-152) = epymetheus.query_pileup_records on a bgzip + tabix
    pileup: ONLY the BGZF members that hold the requested contigs are read from disk (virtual offsets of the .tbi),
    inflated (K7) and parsed (K6) on the device.  Rows come back with contig_id indexing `contigs`; contigs that are
    not in the index contribute nothing (the reference logs a warning and returns an empty frame when nothing is found).
    A bin's pileup therefore costs its own share of the file, not the whole file (cfg 3: > 100 GB of text)."""
    from .bgzf import TabixIndex, fetch_contigs_device

    contigs = list(contigs)
    d = _require_cuda(device)
    index = TabixIndex.read(path + ".tbi")
    text, _ = fetch_contigs_device(path, contigs, d, index)
    if int(text.numel()) == 0:
        new = lambda dt: torch.empty(0, dtype=dt, device=d)
        counts = dict(n_mod=new(torch.int64), n_diff=new(torch.int64)) if with_counts else {}
        return DeviceRows(contigs, mod_types, d, contig_id=new(torch.int32), position=new(torch.int64), strand=new(torch.uint8),
                          mod_type=new(torch.uint8), Nvalid_cov=new(torch.int64), fraction_mod=new(torch.float64),
                          percent_x100=new(torch.uint16), **counts)
    # merged block ranges may carry neighbouring contigs (two requested contigs with others between them never do:
    # ranges are per contig span); rows of unknown contigs are dropped by the parser
    return parse_bedmethyl(text, contigs, mod_types, with_counts, d)


def parse_fasta_device(data, trim_names: bool = False, trim_character: str = " ", device=None):
    """FASTA TEXT (bytes / uint8 array / tensor, host or device) -> DeviceAssembly, parsed on the GPU: the sequence lines
    of every record are concatenated on the device and packed (nmb_fasta_lines / nmb_fasta_copy / nmb_pack_sequence);
    only the header lines come back to the host, for the names.  Same names and sequences as load_fasta
    (fasta.py:35-49 + the upper-casing of seq.py:55, done by the packer)."""
    from .device import DeviceAssembly

    d = _require_cuda(device)
    if isinstance(data, (bytes, bytearray, memoryview)):
        data = np.frombuffer(data, dtype=np.uint8)
    with torch.cuda.device(d):
        text = data.to(d, non_blocking=True) if isinstance(data, torch.Tensor) else _to_device(np.asarray(data, dtype=np.uint8), d)
        n_bytes = int(text.numel())
        scratch = torch.empty((n_bytes + 4095) // 4096 + 2, dtype=torch.int64, device=d)
        n_nl = torch.zeros(1, dtype=torch.int64, device=d)
        check(lib.nmb_index_bytes(ptr(text), n_bytes, 10, ptr(scratch), None, 0, ptr(n_nl), _stream()), "nmb_index_bytes")
        n_newlines = int(n_nl.item())
        newline_pos = torch.empty(max(n_newlines, 1), dtype=torch.int64, device=d)
        if n_newlines:
            check(lib.nmb_index_bytes(ptr(text), n_bytes, 10, ptr(scratch), ptr(newline_pos), n_newlines, ptr(n_nl),
                                      _stream()), "nmb_index_bytes")
        n_lines = n_newlines + (1 if n_bytes > 0 and int(text[-1].item()) != 10 else 0)
        if n_lines == 0:
            raise ValueError("empty FASTA")
        kind = torch.empty(n_lines, dtype=torch.uint8, device=d)
        total = torch.zeros(1, dtype=torch.int64, device=d)

        def copy_pass(want_headers: int):
            payload = torch.empty(n_lines + 1, dtype=torch.int64, device=d)
            payload[n_lines] = 0
            check(lib.nmb_fasta_lines(ptr(text), n_bytes, ptr(newline_pos), n_newlines, n_lines, want_headers, ptr(kind),
                                      ptr(payload), _stream()), "nmb_fasta_lines")
            check(lib.nmb_exclusive_scan_i64(ptr(payload), n_lines + 1, ptr(total), _stream()), "nmb_exclusive_scan_i64")
            n_out = int(total.item())
            out = torch.empty(max(n_out, 1), dtype=torch.uint8, device=d)
            check(lib.nmb_fasta_copy(ptr(text), n_bytes, ptr(newline_pos), n_newlines, n_lines, want_headers, ptr(payload),
                                     ptr(out), _stream()), "nmb_fasta_copy")
            return payload, out[:n_out]

        seq_off, seq = copy_pass(0)  # seq_off[r] = sequence bytes before line r
        # header lines: their line numbers (ascending) through the generic byte index
        n_hdr = torch.zeros(1, dtype=torch.int64, device=d)
        scratch2 = torch.empty((n_lines + 4095) // 4096 + 2, dtype=torch.int64, device=d)
        check(lib.nmb_index_bytes(ptr(kind), n_lines, 1, ptr(scratch2), None, 0, ptr(n_hdr), _stream()), "nmb_index_bytes")
        n_contigs = int(n_hdr.item())
        if n_contigs == 0:
            raise ValueError("FASTA without a header line")
        hdr_lines = torch.empty(n_contigs, dtype=torch.int64, device=d)
        check(lib.nmb_index_bytes(ptr(kind), n_lines, 1, ptr(scratch2), ptr(hdr_lines), n_contigs, ptr(n_hdr), _stream()),
              "nmb_index_bytes")
        starts = seq_off[hdr_lines].cpu().numpy()  # a header line carries no sequence bytes: the offset of its record
        hdr_off, hdr = copy_pass(1)
        hdr_starts = hdr_off[hdr_lines].cpu().numpy()
        hdr_bytes = hdr.cpu().numpy().tobytes()
    ends = np.append(starts[1:], int(seq.numel()))
    hdr_ends = np.append(hdr_starts[1:], len(hdr_bytes))
    names = []
    for b, e in zip(hdr_starts, hdr_ends):
        name = hdr_bytes[b:e].decode().strip()
        names.append(name.split(trim_character)[0] if trim_names else (name.split()[0] if name.split() else ""))
    lengths = (ends - starts).astype(np.int64)
    return DeviceAssembly(names, lengths, seq if int(seq.numel()) else torch.zeros(1, dtype=torch.uint8, device=d),
                          starts.astype(np.int64), d)


def load_fasta_device(path: str, trim_names: bool = False, trim_character: str = " ", device=None):
    """load_fasta with the parse and the 2-bit packing on the GPU (bgzip files are inflated there as well)."""
    with open(path, "rb") as f:
        data = f.read()
    if data[:2] == b"\x1f\x8b":
        if bgzf_blocks(data) is not None:
            data = inflate_bgzf_device(data, device)
        else:
            import gzip

            data = gzip.decompress(data)
    return parse_fasta_device(data, trim_names, trim_character, device)
