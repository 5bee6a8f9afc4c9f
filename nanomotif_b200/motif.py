"""Motif value type of the scoring path and its compilation to device masks.

Mirrors the part of the reference's ``nanomotif.motif.Motif`` (nanomotif/motif.py:18-359) that the
hot path consumes: a regex-subset string over ``A C G T . [..]`` plus the 0-based index of the
modified base.  The string algebra stays on the host; what the GPU sees is one 4-bit allowed-set per
motif position (bit0=A bit1=T bit2=G bit3=C, the order of nanomotif/constants.py:21-28).

Any object with ``str(obj)`` = motif string and an integer ``mod_position`` attribute (e.g. the
reference's own ``Motif``) is accepted wherever this module takes a motif.
"""
from __future__ import annotations

import numpy as np

from . import _lib

BASES = ("A", "T", "G", "C")  # nanomotif/constants.py:1 -- PSSM row order and bit order
_BIT = {"A": 1, "T": 2, "G": 4, "C": 8}
_WILD = 0xF
_COMP_BASE = {"A": "T", "T": "A", "G": "C", "C": "G", ".": ".", "N": "N"}
_IUPAC_SETS = {
    "A": "A", "C": "C", "G": "G", "T": "T", "R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT",
    "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT",
}
_SET_TO_IUPAC = {frozenset(v): k for k, v in _IUPAC_SETS.items()}


def tokenize(motif_string: str) -> list[str]:
    """Split into per-position tokens, keeping bracket classes together (motif.py:226-245)."""
    if "[" not in motif_string:  # the common case in the search: one token per character
        return list(motif_string)
    out, i, n = [], 0, len(motif_string)
    while i < n:
        ch = motif_string[i]
        if ch == "[":
            j = motif_string.find("]", i)
            if j < 0:
                raise ValueError("Unmatched bracket")
            out.append(motif_string[i : j + 1])
            i = j + 1
        else:
            out.append(ch)
            i += 1
    return out


def token_mask(token: str) -> int:
    """Allowed-set of one token under *regex* semantics (what utils.subseq_indices matches)."""
    if token == ".":
        return _WILD
    letters = token[1:-1] if token.startswith("[") else token
    m = 0
    for ch in letters:
        if ch not in _BIT:
            raise ValueError(f"motif token {token!r}: only A, C, G, T, '.' and [..] classes are supported")
        m |= _BIT[ch]
    if m == 0:
        raise ValueError(f"empty motif token {token!r}")
    return m


class Motif(str):
    """``Motif("G[AG].GAAG[CT]", 5)`` -- same constructor and attributes as the reference type."""

    def __new__(cls, motif_string, *args, **kwargs):
        return str.__new__(cls, motif_string)

    def __init__(self, _motif_string, mod_position):
        self.mod_position = mod_position
        self.string = str.__str__(self)

    # value semantics identical to motif.py:26-36
    def __eq__(self, other):
        return (
            hasattr(other, "mod_position")
            and isinstance(other, str)
            and str.__str__(self) == str.__str__(other)
            and self.mod_position == other.mod_position
        )

    # no __ne__: like the reference type (motif.py:26-36 defines __eq__ only), `!=` is str's -- it compares the strings
    # and ignores mod_position.  Its one use on the path (find_motifs_bin.py:780) compares motifs of equal position.

    def __hash__(self):
        return hash((self.string, self.mod_position))

    def __repr__(self):
        return f"Motif({self.string!r}, pos={self.mod_position})"

    def split(self) -> list[str]:  # type: ignore[override]
        return tokenize(self.string)

    def length(self) -> int:
        return len(self.split())

    def new_stripped_motif(self, character: str = ".") -> "Motif":
        """Drop flanking wildcards and re-base mod_position (motif.py:213-224)."""
        s = self.string
        lead = len(s) - len(s.lstrip(character))
        if lead == len(s):  # nothing but wildcards: returned unchanged, like the reference
            return self
        return Motif(s.strip(character), self.mod_position - lead)

    def reverse_compliment(self) -> "Motif":
        """Reverse complement; bracket classes stay well formed (motif.py:260-266)."""
        toks = self.split()
        out = []
        for tok in reversed(toks):
            if tok.startswith("["):
                out.append("[" + "".join(_COMP_BASE[c] for c in reversed(tok[1:-1])) + "]")
            else:
                out.append(_COMP_BASE[tok])
        return Motif("".join(out), len(toks) - self.mod_position - 1)

    def one_hot(self) -> np.ndarray:
        """(length, 4) 0/1 matrix in A,T,G,C column order (motif.py:247-258)."""
        toks = self.split()
        arr = np.zeros((len(toks), 4), dtype=int)
        for i, tok in enumerate(toks):
            m = _WILD if tok in (".", "N") else token_mask(tok)
            for b in range(4):
                arr[i, b] = (m >> b) & 1
        return arr

    def count_isolated_bases(self, isolation_size: int = 2) -> int:
        """Constrained positions whose neighbourhood of +-isolation_size holds only wildcards.  Keeps the
        reference's right-edge quirk: the window is clipped at len-1, not len (motif.py:178-194)."""
        toks = self.split()
        n = 0
        for pos, tok in enumerate(toks):
            if tok == ".":
                continue
            lo = max(pos - isolation_size, 0)
            hi = min(pos + isolation_size + 1, len(toks) - 1)
            around = set(toks[lo:pos] + toks[pos + 1 : hi])
            n += (around == {"."}) + (around == {"N"})
        return n

    def sub_motif_of(self, other) -> bool:
        """True when every occurrence of self is an occurrence of `other` aligned at the modified base
        (motif.py:54-88, including its early exits)."""
        other = as_motif(other)
        if self.string == other.string:
            return False
        a, b = self.new_stripped_motif(), other.new_stripped_motif()
        if a.length() < b.length():
            return False
        sa, sb = a.split(), b.split()
        off = b.mod_position - a.mod_position
        if off > 0:
            return False
        for i, base in enumerate(sa):
            j = i + off
            if j < 0:
                continue
            if j >= len(sb):
                return True
            if sb[j] != "." and not set(base) <= set(sb[j]):
                return False
        return True

    def sub_motif_of_any(self, others) -> bool:
        return any(self.sub_motif_of(o) for o in others)

    def iupac(self) -> str:
        out = []
        for tok in self.split():
            if tok == ".":
                out.append("N")
            else:
                letters = tok[1:-1] if tok.startswith("[") else tok
                out.append(_SET_TO_IUPAC.get(frozenset(letters), ""))
        return "".join(out)

    def from_iupac(self) -> "Motif":
        out = []
        for ch in self.string:
            s = _IUPAC_SETS[ch]
            out.append("." if len(s) == 4 else (s if len(s) == 1 else "[" + s + "]"))
        return Motif("".join(out), self.mod_position)


def as_motif(motif) -> Motif:
    if isinstance(motif, Motif):
        return motif
    if not hasattr(motif, "mod_position"):
        raise TypeError("Motif is not a Motif type")  # same message as find_motifs_bin.py:1253
    return Motif(str.__str__(motif), int(motif.mod_position))


_PLAIN_TABLE = bytes(_BIT.get(chr(c), _WILD if chr(c) == "." else 0) for c in range(256))  # 0 = not a plain token


def motif_masks(motif) -> tuple[np.ndarray, int]:
    """(allowed-set per position as uint8 array, mod_position) of the motif as given (not stripped)."""
    m = as_motif(motif)
    s = m.string
    if "[" not in s:  # one token per character (what the search generates): one table lookup for the whole motif
        masks = np.frombuffer(s.encode("latin-1", "replace").translate(_PLAIN_TABLE), dtype=np.uint8)
        if masks.size and masks.min() == 0:
            bad = s[int(np.argmin(masks))]
            raise ValueError(f"motif token {bad!r}: only A, C, G, T, '.' and [..] classes are supported")
        return masks, int(m.mod_position)
    toks = m.split()
    return np.fromiter((token_mask(t) for t in toks), dtype=np.uint8, count=len(toks)), int(m.mod_position)


_PLAIN_LUT = np.full(256, 0xFF, dtype=np.uint8)  # byte -> allowed-set; 0xFF = not a plain motif character
for _ch, _m in _BIT.items():
    _PLAIN_LUT[ord(_ch)] = _m
_PLAIN_LUT[ord(".")] = _WILD
_PLAIN_LUT[0] = 0  # padding


def _pack_one(out, i, m, strip, mod_pos_override):
    if strip:
        m = m.new_stripped_motif()
    masks, mp = motif_masks(m)
    n = len(masks)
    if n == 0:
        raise ValueError("Motif is empty")
    if n > _lib.MAX_MOTIF_LEN:
        raise ValueError(f"motif {m!r}: stripped length {n} exceeds {_lib.MAX_MOTIF_LEN}")
    if int(masks.min()) == _WILD:
        raise ValueError(f"motif {m!r} has no constrained position")
    if mod_pos_override is not None:
        mp = mod_pos_override
    if not (0 <= mp < n):
        raise ValueError(f"motif {m!r}: mod_position {mp} outside the stripped motif")
    out["allowed"][i, :n] = masks
    out["len"][i] = n
    out["mod_pos"][i] = mp


def pack_motifs(motifs, strip: bool = True, mod_pos_override: int | None = None) -> np.ndarray:
    """Compile motifs to an array of ``nmb_motif`` records (include/nmb200.h).

    strip=True applies new_stripped_motif first, as motif_model_contig does
    (find_motifs_bin.py:1307).  Raises ValueError for motifs the device path cannot represent.
    The whole batch goes through ONE native call (nmb_pack_motifs, host code of libnmb200: strip, split, allowed sets):
    ~0.15 us per motif instead of ~2 us for the numpy version below and ~6 us motif by motif -- a frontier round of a
    lock-step search packs the <= 4 children of every (bin, mod type) search, and this was half of a round's host
    time.  Motifs the native packer refuses go through `_pack_one`, which raises the precise error.
    """
    motifs = motifs if isinstance(motifs, (list, tuple)) else list(motifs)
    n_motifs = len(motifs)
    if n_motifs == 0:
        return np.zeros(0, dtype=_lib.MOTIF_DTYPE)
    try:
        text = "".join(motifs)
    except TypeError:
        text = None  # not strings: the loop below raises the reference's TypeError
    if text is None or not text.isascii():
        return _pack_motifs_numpy(motifs, strip, mod_pos_override)
    try:
        mods32 = np.fromiter((mo.mod_position for mo in motifs), dtype=np.int32, count=n_motifs)
    except AttributeError:
        raise TypeError("Motif is not a Motif type") from None  # same message as find_motifs_bin.py:1253
    except (TypeError, ValueError, OverflowError):  # None, floats, huge values: the slow path says what is wrong
        return _pack_motifs_numpy(motifs, strip, mod_pos_override)
    if mod_pos_override is not None and not 0 <= mod_pos_override < 2**31:
        return _pack_motifs_numpy(motifs, strip, mod_pos_override)
    off = np.zeros(n_motifs + 1, dtype=np.int64)
    np.cumsum(np.fromiter(map(len, motifs), dtype=np.int64, count=n_motifs), out=off[1:])
    out = np.zeros(n_motifs, dtype=_lib.MOTIF_DTYPE)
    status = np.empty(n_motifs, dtype=np.uint8)
    _lib.check(_lib.lib.nmb_pack_motifs(text.encode("ascii"), off.ctypes.data, mods32.ctypes.data, n_motifs, 1 if strip else 0,
                                        -1 if mod_pos_override is None else int(mod_pos_override), out.ctypes.data,
                                        status.ctypes.data), "nmb_pack_motifs")
    if status.any():
        for i in np.flatnonzero(status).tolist():
            _pack_one(out, i, as_motif(motifs[i]), strip, mod_pos_override)  # raises the precise error
    return out


def _pack_motifs_numpy(motifs, strip: bool = True, mod_pos_override: int | None = None) -> np.ndarray:
    """pack_motifs without the native helper: motifs without bracket classes are packed together with one bytes join
    and one table lookup, the others one by one.  Kept for inputs the native call does not take (non-ASCII text, odd
    mod positions -- they end in the precise error) and as the independent implementation the tests hold it against."""
    n_motifs = len(motifs)
    out = np.zeros(n_motifs, dtype=_lib.MOTIF_DTYPE)
    W = _lib.MAX_MOTIF_LEN
    plain_idx, parts, mods, slow = [], [], [], []
    for i, mo in enumerate(motifs):
        st = str.__str__(mo)
        if "[" in st:
            slow.append(i)
            continue
        mp = mo.mod_position if hasattr(mo, "mod_position") else None
        if mp is None:
            raise TypeError("Motif is not a Motif type")
        if strip:
            core = st.lstrip(".")
            lead = len(st) - len(core)
            if core:  # an all-wildcard motif is returned unchanged by new_stripped_motif (and rejected below)
                st, mp = core.rstrip("."), mp - lead
        if len(st) > W or not st.isascii():
            slow.append(i)  # raises the precise error
            continue
        plain_idx.append(i)
        parts.append(st.ljust(W, "\0"))
        mods.append(mp)
    if plain_idx:
        idx = np.asarray(plain_idx, dtype=np.int64)
        codes = np.frombuffer("".join(parts).encode("latin-1"), dtype=np.uint8).reshape(len(parts), W)
        masks = _PLAIN_LUT[codes]
        lens = (codes != 0).sum(axis=1)
        mp = np.asarray(mods, dtype=np.int64) if mod_pos_override is None else np.full(len(parts), mod_pos_override, dtype=np.int64)
        ok = (masks != 0xFF).all(axis=1) & (lens > 0) & (mp >= 0) & (mp < lens)
        ok &= ((masks != _WILD) & (masks != 0)).any(axis=1)
        if not ok.all():
            slow.extend(idx[~ok].tolist())  # the slow path raises the precise error
            idx, masks, lens, mp = idx[ok], masks[ok], lens[ok], mp[ok]
        out["allowed"][idx] = masks
        out["len"][idx] = lens
        out["mod_pos"][idx] = mp
    for i in slow:
        _pack_one(out, i, as_motif(motifs[i]), strip, mod_pos_override)
    return out


SIB_SAME, SIB_DIFF = 1, 2  # sibling link kinds (csrc/scan.cu)


def sibling_links(packed: np.ndarray) -> np.ndarray:
    """Sibling word of every packed motif, as the device motif compiler writes it (nmb_compile_motifs_siblings): the
    link to the previous motif -- same len and mod_pos and the same allowed set at every position but at most one j,
    where both sets are non-empty -- as j | kind << 6 | own set at j << 8 | previous motif's set at j << 12."""
    out = np.zeros(len(packed), dtype=np.uint32)
    for i in range(1, len(packed)):
        a, b = packed[i - 1], packed[i]
        la, lb = int(a["len"]), int(b["len"])
        ok = all(1 <= int(m["len"]) <= _lib.MAX_MOTIF_LEN and int(m["mod_pos"]) < int(m["len"]) for m in (a, b))
        if not ok or la != lb or a["mod_pos"] != b["mod_pos"]:
            continue
        sa, sb = a["allowed"][:la] & 0xF, b["allowed"][:lb] & 0xF
        d = np.flatnonzero(sa != sb)
        if len(d) == 0:
            out[i] = SIB_SAME << 6
        elif len(d) == 1 and sa[d[0]] and sb[d[0]]:
            j = int(d[0])
            out[i] = j | SIB_DIFF << 6 | int(sb[j]) << 8 | int(sa[j]) << 12
    return out


def sibling_runs(links: np.ndarray, begin: int, count: int) -> list[tuple[int, int, int]]:
    """The sibling runs K2 scores inside the motif block [begin, begin + count), from sibling_links: (first motif,
    members, split position j) per run of >= 2 members, left to right.  A run takes the following motifs while they
    are linked to their left neighbour and any differing link is at the run's j; identical motifs alone form no run."""
    kind = (links[begin:begin + count] >> 6) & 3
    jj = links[begin:begin + count] & 63
    runs, a = [], 0
    while a < count:
        e = a + 1
        while e < count and kind[e]:
            e += 1
        diff = [i for i in range(a + 1, e) if kind[i] == SIB_DIFF]
        if not diff:
            a += 1
            continue
        j = int(jj[diff[0]])
        end = a + 1
        while end < e and not (kind[end] == SIB_DIFF and jj[end] != j):
            end += 1
        runs.append((begin + a, end - a, j))
        a = end
    return runs


def window_masks(motifs, width: int) -> np.ndarray:
    """Full-width (not stripped) masks for the window filter (DNAarray.filter_sequence_matches)."""
    out = np.zeros(len(motifs), dtype=_lib.MOTIF_DTYPE)
    for i, mo in enumerate(motifs):
        toks = as_motif(mo).split()
        if len(toks) != width:
            raise AssertionError("Sequence must have the same length as sequences in the array")  # seq.py:516
        # one_hot semantics (motif.py:247-258): 'N' and '.' are all-ones
        out["allowed"][i, :width] = [(_WILD if t in (".", "N") else token_mask(t)) for t in toks]
        out["len"][i] = width
        out["mod_pos"][i] = min(int(getattr(mo, "mod_position", 0)), width - 1)
    return out
