"""ctypes binding of libnmb200.so (the C ABI declared in include/nmb200.h).

The product path has no CPU fallback: if the shared library is missing or does not export the
declared ABI, importing this module raises.  Nothing here touches ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnmb200.so")

# ---- constants mirrored from include/nmb200.h -------------------------------------------------
ABI_VERSION = 10
CHUNK_WORDS = 16
CHUNK_BP = 512
TILE_WORDS = 2048
TILE_BP = 65536
TILE_CHUNKS = 128
HALO_WORDS = 4
SEQ_PLANE_WORDS = TILE_WORDS + 2 * HALO_WORDS
SEQ_REC_WORDS = 2 * SEQ_PLANE_WORDS + TILE_CHUNKS
CLS_REC_WORDS = 4 * TILE_WORDS
# lane-interleaved planes (nmb200.h NMB_WORD_SLOT): WORD_SLOT[w] = slot of tile word w, so
# `plane_in_slot_order[..., WORD_SLOT]` is the plane in natural word order
_w = np.arange(TILE_WORDS)
WORD_SLOT = ((_w & 12) << 7) | ((_w >> 4) << 2) | (_w & 3)
SLOT_WORD = np.argsort(WORD_SLOT)  # inverse: natural_plane[..., SLOT_WORD] is the plane in slot order
del _w
MIN_GAP_BP = 64
MAX_MOTIF_LEN = 62
MAX_WINDOW = 61
MAX_MOTIFS_PER_ITEM = 32


class NmbError(RuntimeError):
    """A libnmb200 entry point returned a negative status."""


class NmbAssembly(C.Structure):
    _fields_ = [
        ("seq_records", C.c_void_p),
        ("nonacgt", C.c_void_p),
        ("contig_start", C.c_void_p),
        ("contig_len", C.c_void_p),
        ("n_contigs", C.c_int32),
        ("n_tiles", C.c_int32),
    ]


class NmbMT19937(C.Structure):
    _fields_ = [("key", C.c_uint32 * 624), ("pos", C.c_int32)]


MOTIF_DTYPE = np.dtype([("allowed", np.uint8, (MAX_MOTIF_LEN,)), ("len", np.uint8), ("mod_pos", np.uint8)])
assert MOTIF_DTYPE.itemsize == 64

JOB_DTYPE = np.dtype(
    [
        ("motif_begin", np.int32),
        ("motif_count", np.int32),
        ("modtype", np.int32),
        ("tile_begin", np.int32),
        ("tile_count", np.int32),
        ("contig_begin", np.int32),
        ("contig_end", np.int32),
        ("group_mode", np.int32),
        ("n_groups", np.int32),
        ("item_offset", np.int32),
        ("out_base", np.int64),
    ],
    align=True,
)
assert JOB_DTYPE.itemsize == 48

SWEEP_HIT_DTYPE = np.dtype([("slot", np.int32), ("index", np.uint32), ("n_mod", np.uint32), ("n_nomod", np.uint32)])
assert SWEEP_HIT_DTYPE.itemsize == 16

SWEEP_QUERY_DTYPE = np.dtype(
    [
        ("kind", np.int32),
        ("n_pos", np.int32),
        ("base", np.int64),
        ("class_step", np.int32),
        ("n_states", np.uint8, (7,)),
        ("reserved", np.uint8),
        ("offset", np.int32, (7, 5)),
    ],
    align=True,
)
assert SWEEP_QUERY_DTYPE.itemsize == 168

_P = C.c_void_p
_I32 = C.c_int32
_I64 = C.c_int64
_F64 = C.c_double

# name -> (restype, argtypes); every symbol declared in include/nmb200.h
SIGNATURES = {
    "nmb_abi_version": (C.c_int, []),
    "nmb_last_error": (C.c_char_p, []),
    "nmb_device_sm_count": (C.c_int, []),
    "nmb_program_bytes": (C.c_int, []),
    "nmb_pack_sequence": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _P, _P, _P]),
    "nmb_build_class_planes": (C.c_int, [_P, _P, _P, _P, _P, _I64, _F64, _F64, C.POINTER(NmbAssembly), _I32, _P, _P]),
    "nmb_add_class_planes": (C.c_int, [_P, _P, _P, _P, _P, _I64, _F64, _F64, C.POINTER(NmbAssembly), _I32, _P, _P, _P]),
    "nmb_lookup_strings": (C.c_int, [_P, _P, _I32, _I64, _P, _P, _P, _P, _I32, _I32, _P, _I32, _P]),
    "nmb_build_class_planes_compact": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _I32, C.POINTER(NmbAssembly), _I32, _P, _P]),
    "nmb_clear_class_planes": (C.c_int, [C.POINTER(NmbAssembly), _I32, _P, _P]),
    "nmb_index_bytes": (C.c_int, [_P, _I64, _I32, _P, _P, _I64, _P, _P]),
    "nmb_bed_parse": (C.c_int, [_P, _I64, _P, _I64, _P, _P, _P, _P, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "nmb_fasta_lines": (C.c_int, [_P, _I64, _P, _I64, _I64, _I32, _P, _P, _P]),
    "nmb_fasta_copy": (C.c_int, [_P, _I64, _P, _I64, _I64, _I32, _P, _P, _P]),
    "nmb_exclusive_scan_i64": (C.c_int, [_P, _I64, _P, _P]),
    "nmb_gather_rows": (C.c_int, [_P, _I32, _P, _I64, _P, _P]),
    "nmb_bgzf_inflate": (C.c_int, [_P, _P, _P, _P, _P, _P, _I32, _P, _P, _P]),
    "nmb_sweep_hist_size": (C.c_int64, []),
    "nmb_sweep_hist": (C.c_int, [C.POINTER(NmbAssembly), _P, _I32, _I32, _I32, _I32, _P, _I32, _P, _P]),
    "nmb_sweep_finalize": (C.c_int, [_P, _I32, _P]),
    "nmb_sweep_bipartite_size": (C.c_int64, []),
    "nmb_sweep_bipartite": (C.c_int, [C.POINTER(NmbAssembly), _P, _I32, _I32, _I32, _I32, _P, _I32, _P, _P]),
    "nmb_sweep_bipartite_finalize": (C.c_int, [_P, _I32, _P]),
    "nmb_sweep_slice": (C.c_int, [_P, _I64, _I32, _P, _I64, _I64, _I32, _P]),
    "nmb_sweep_expand": (C.c_int, [_P, _P, _I64, _I64, _P]),
    "nmb_sweep_filter": (C.c_int, [_P, _P, _I64, _F64, _I64, _P, _I64, _P, _P]),
    "nmb_sweep_expand_filter": (C.c_int, [_P, _P, _I64, _I64, _I32, _I32, _F64, _I64, _I32, _P, _I64, _P, _P]),
    "nmb_sweep_bipartite_filter": (C.c_int, [_P, _I32, _I32, _F64, _I64, _I32, _P, _I64, _P, _P]),
    "nmb_sweep_bip_iupac_slice": (C.c_int, [_P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P]),
    "nmb_sweep_bip_iupac_expand": (C.c_int, [_P, _P, _I64, _I64, _P]),
    "nmb_sweep_bip_iupac_expand_filter": (C.c_int, [_P, _P, _I64, _I64, _F64, _I64, _I32, _P, _I64, _P, _P]),
    "nmb_sweep_prune_lattice": (C.c_int, [_I32, _P, _P, _P]),
    "nmb_sweep_lookup": (C.c_int, [_P, _P, _P, _I32, _P, _I64, _P, _P]),
    "nmb_add_class_planes_compact": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _I32, C.POINTER(NmbAssembly), _I32, _P, _P]),
    "nmb_filter_coverage": (C.c_int, [_P, _I64, _I64, _P, _P]),
    "nmb_filter_min_mod_frequency": (C.c_int, [_P, _P, _I64, _I32, _F64, _F64, _I64, _P, _P, _P]),
    "nmb_filter_adjacency": (C.c_int, [_P, _P, _P, _P, _I64, _F64, _I32, _P, _P, _P]),
    "nmb_compile_motifs": (C.c_int, [_P, _I32, _P, _P]),
    "nmb_scan_count": (C.c_int, [C.POINTER(NmbAssembly), _P, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _I32, _P]),
    "nmb_scan_count_balanced": (C.c_int, [C.POINTER(NmbAssembly), _P, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _I32, _P, _P]),
    "nmb_sibling_bytes": (C.c_int64, [_I32]),
    "nmb_compile_motifs_siblings": (C.c_int, [_P, _I32, _P, _P, _P]),
    "nmb_scan_count_siblings": (C.c_int, [C.POINTER(NmbAssembly), _P, _P, _P, _I32, _P, _I32, _I32, _I32, _I32, _P, _P, _I32, _P, _P]),
    "nmb_match_plane": (C.c_int, [C.POINTER(NmbAssembly), _P, _I32, _I32, _I32, _I32, _I32, _P, _P]),
    "nmb_letter_plane": (C.c_int, [_P, _I64, _I32, _I64, _P, _I64, _P]),
    "nmb_compact_positions": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _I64, _P, _P]),
    "nmb_test_positions": (C.c_int, [_P, _I64, _I64, _P, _I64, _P, _P]),
    "nmb_extract_windows": (C.c_int, [C.POINTER(NmbAssembly), _P, _P, _I64, _I32, _P, _P]),
    "nmb_window_hist": (C.c_int, [_P, _P, _I64, _I32, _P, _I32, _I32, _P, _P, _P, _P]),
    "nmb_window_hist_ranges": (C.c_int, [_P, _P, _I64, _I32, _P, _I32, _P, _P, _I64, _I32, _P, _P, _P, _P]),
    "nmb_pattern_stats": (C.c_int, [_P, _P, _P, _P, _P, _I64, _P, _P, _I32, _P, _P, _P, _P]),
    "nmb_pattern_median": (C.c_int, [_P, _P, _P, _P, _P, _I64, _P, _P, _I32, _P, _P, _P, _P, _P]),
    "nmb_pattern_index_build": (C.c_int, [C.POINTER(NmbAssembly), _P, _P, _P, _P, _I32, _P, _P, _P, _I64, _I64, _F64, _P, _P, _P, _P, _P, _P]),
    "nmb_pattern_scan": (C.c_int, [C.POINTER(NmbAssembly), _P, _P, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _I32, _P]),
    "nmb_pattern_scan_balanced": (C.c_int, [C.POINTER(NmbAssembly), _P, _P, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _I32, _P, _P]),
    "nmb_segment_offsets": (C.c_int, [_P, _I64, _P, _P, _P]),
    "nmb_segment_median": (C.c_int, [_P, _P, _I64, _P, _P]),
    "nmb_mt_sample": (C.c_int, [_P, _I64, _I64, _P]),
    "nmb_mt_sample_many": (C.c_int, [_P, _P, _P, _I64, _P]),
    "nmb_pack_motifs": (C.c_int, [_P, _P, _P, _I32, _I32, _I32, _P, _P]),
    "nmb_stager_create": (C.c_int, [_I64, _I32, C.POINTER(_P)]),
    "nmb_stager_copy": (C.c_int, [_P, _P, _P, _I64, _P]),
    "nmb_stager_copy_narrow": (C.c_int, [_P, _P, _P, _I64, C.POINTER(C.c_int32), _P]),
    "nmb_stager_gather": (C.c_int, [_P, _P, _P, _P, _I64, _P]),
    "nmb_stager_destroy": (C.c_int, [_P]),
    "nmb_bin_means": (C.c_int, [_P, _P, _I32, _I32, _P, _P, _I32, _F64, _P, _P, _P, _P, _P]),
    "nmb_bin_matrix": (C.c_int, [_P, _P, _P, _P, _P, _P, _I32, _I32, _P, _I64, _P, _I32, _P, _P]),
    "nmb_pssm_kl": (C.c_int, [_P, _P, _I32, _I32, _P, _P, _P, _P]),
}


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python nanomotif_b200/build.py` "
            "(nvcc, sm_100a). nanomotif_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:  # pragma: no cover - ABI mismatch
            raise ImportError(f"{LIB_PATH} does not export {name}; rebuild it with `python nanomotif_b200/build.py`") from exc
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.nmb_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.nmb_abi_version()} != {ABI_VERSION}; rebuild it")
    return lib


lib = _load()


def check(status: int, what: str = "libnmb200") -> None:
    if status < 0:
        msg = lib.nmb_last_error()
        raise NmbError(f"{what} failed with status {status}: {msg.decode(errors='replace') if msg else ''}")


def ptr(t) -> int | None:
    """Device (or host) address of a torch tensor / numpy array; None passes NULL."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()
