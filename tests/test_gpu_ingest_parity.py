"""The pileup ingest chain row by row against plain references, at the places where its kernels could be subtly wrong:

    nmb_index_bytes          byte positions vs np.flatnonzero: unaligned sources, 16- and 4096-byte edges, > 1024 blocks,
                             capacity smaller than the count; the '\\n' index of the parser and the keep masks of take_mask
    nmb_bed_parse            every kept column vs oracle/restate.py::load_pileup_text on text that puts number, name, mod code
                             and strand edges at line starts, line ends and block boundaries; the status counters
    the three filters        DeviceRows.filter_* and dataload.filter_pileup* vs the oracle: interleaved and invalid groups,
                             values equal to every threshold, ties, NaN rows, contig changes, distances 0 / 1 / 8 / 1000
    class planes             class records decoded on the host vs a numpy restatement of find_motifs_bin.py:1308-1314, from
                             float rows (from_columns) and from compact rows (from_compact); dup_count vs numpy.unique
    end to end               text (plain and BGZF) -> parse -> filters -> class planes == load_pileup_text -> oracle filters ->
                             oracle classification

Every comparison is exact."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O

MOD_TYPES = ("a", "m", "21839", "ABCDEFGH")  # the last one is a code of exactly 8 bytes, the longest the parser keys


@pytest.fixture(scope="module")
def dl():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from nanomotif_b200 import dataload

    return dataload


def _stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


# ---------------------------------------------------------------------------------------------------------------------
# nmb_index_bytes
# ---------------------------------------------------------------------------------------------------------------------
SENTINEL = -7


def index_bytes(src, value, capacity, out_len):
    """(count, out as numpy) of one nmb_index_bytes call on the device uint8 tensor `src`; out starts as SENTINEL."""
    import torch

    from nanomotif_b200._lib import check, lib, ptr

    n = int(src.numel())
    scratch = torch.empty((n + 4095) // 4096 + 1, dtype=torch.int64, device=src.device)
    n_out = torch.full((1,), -1, dtype=torch.int64, device=src.device)
    out = torch.full((max(out_len, 1),), SENTINEL, dtype=torch.int64, device=src.device)
    check(lib.nmb_index_bytes(ptr(src), n, value, ptr(scratch), ptr(out), capacity, ptr(n_out), _stream()), "nmb_index_bytes")
    return int(n_out.item()), out.cpu().numpy()


def test_byte_index_against_flatnonzero(dl):
    import torch

    rng = np.random.default_rng(101)
    big = 1024 * 4096 + 3 * 4096 + 17  # 1028 blocks: the one-CTA scan takes two blocks per thread
    host = np.zeros(big + 64, dtype=np.uint8)
    dev = torch.empty(big + 64, dtype=torch.uint8, device="cuda")
    assert dev.data_ptr() % 256 == 0
    for value, fill in ((10, "random"), (1, "random"), (10, "all"), (1, "none"), (1, "mask")):
        if fill == "random":  # text-like bytes, the value about once in 16
            host[:] = rng.integers(0, 256, host.size, dtype=np.uint8)
            host[rng.random(host.size) < 1 / 16] = value
        elif fill == "all":
            host[:] = value
        elif fill == "none":
            host[:] = rng.integers(2, 256, host.size, dtype=np.uint8)
        else:  # a keep mask
            host[:] = rng.random(host.size) < 0.5
        # the value on every 16- and 4096-byte edge (and one before / after), where the vector and scalar paths meet
        if fill in ("random", "mask"):
            for b in range(0, host.size, 4096):
                host[[x for x in (b - 1, b, b + 15, b + 16) if 0 <= x < host.size]] = value
        dev.copy_(torch.from_numpy(host))
        for n in (0, 1, 15, 16, 17, 31, 4095, 4096, 4097, 5 * 4096 + 1, big):
            offsets = range(16) if n < big else (0, 1, 8, 15)
            for off in offsets:
                want = np.flatnonzero(host[off:off + n] == value)
                src = dev[off:off + n]
                count, _ = index_bytes(src, value, 0, 4)
                assert count == len(want), (value, fill, n, off)
                count, got = index_bytes(src, value, len(want), len(want) + 3)
                assert count == len(want)
                np.testing.assert_array_equal(got[:len(want)], want)
                assert (got[len(want):] == SENTINEL).all()
                if len(want) and off in (0, 3, 15):  # capacity below the count: a correct prefix, nothing past it
                    for cap in sorted({1, len(want) // 2, len(want) - 1} - {0}):
                        count, got = index_bytes(src, value, cap, len(want) + 3)
                        assert count == len(want)
                        np.testing.assert_array_equal(got[:cap], want[:cap])
                        assert (got[cap:] == SENTINEL).all(), (value, fill, n, off, cap)


def test_take_mask_gathers_the_kept_rows(dl):
    import torch

    rng = np.random.default_rng(102)
    for n in (1, 31, 33, 257, 4096, 4097, 70001):
        for p in (0.0, 0.5, 1.0):
            keep = (rng.random(n) < p).astype(np.uint8)
            cols = dict(contig_id=rng.integers(-2, 5, n).astype(np.int32), position=rng.integers(-1, 2**40, n),
                        strand=rng.integers(0, 3, n).astype(np.uint8), mod_type=rng.integers(0, 256, n).astype(np.uint8),
                        Nvalid_cov=rng.integers(0, 99, n), fraction_mod=rng.random(n),
                        percent_x100=rng.integers(0, 2**16, n).astype(np.uint16))
            rows = dl.DeviceRows(["x"], MOD_TYPES, torch.device("cuda"),
                                 **{k: torch.from_numpy(v).cuda() for k, v in cols.items()})
            # the mask as a slice at an odd byte offset of a larger buffer
            buf = torch.zeros(n + 5, dtype=torch.uint8, device="cuda")
            buf[3:3 + n] = torch.from_numpy(keep).cuda()
            got = rows.take_mask(buf[3:3 + n])
            assert len(got) == int(keep.sum())
            for k, v in cols.items():
                assert getattr(got, k).cpu().numpy().tobytes() == v[keep == 1].tobytes(), (n, p, k)


# ---------------------------------------------------------------------------------------------------------------------
# nmb_bed_parse
# ---------------------------------------------------------------------------------------------------------------------
NAMES = ["c10", "c", "c1", "NODE_1_length_5_cov_2.5", "c", "c100"]  # prefixes of each other, and "c" twice
PCT_EDGES = ["0", "0.00", "100", "100.00", "100.01", "100.000", "5.", ".5", "-0.00", "-0", "-5.25", "-.5", "33.33", "66.67",
             "0.125", "99.999", "000.10", "007.50", "70", "30", "70.00", "30.00",
             "123456789012345", "1.23456789012345", ".000000000000001", "99.9999999999999",   # 15 significant digits
             "1234567890123456", "1.234567890123456", "0.000000000000001",                    # 16: outside the grammar
             "NA", "null", "", "1e1", "+5", "nan"]
PCT_GARBAGE = ["5-", "--5", ".", "-", "1.2.3", "5 ", "0x10"]  # text the oracle's float() refuses: not a number here
INT_EDGES = ["0", "7", "-0", "-5", "123456789012345678", "1234567890123456789", "NA", "", "+5"]  # 18 digits in, 19 out
MOD_EDGES = ["a", "m", "21839", "ABCDEFGH", "ABCDEFGHI", "ABCDEFG", "h", "", "M"]
STRAND_EDGES = ["+", "-", ".", "+-", "--", "", "++"]


def dev_int(s):
    """What nmb_bed_parse reads from an integer field (position, Nvalid_cov, n_mod, n_diff): the value of an optional
    '-' and 1..18 digits, else None (written as -1 and counted as not a number)."""
    return int(s) if re.fullmatch(r"-?\d{1,18}", s) else None


def dev_pct(s):
    """Column 11 as nmb_bed_parse reads it: an optional '-', digits and at most one '.', 1..15 digits in all; the value is
    then the correctly rounded double of the text, i.e. float(s).  Anything else (NA, exponents, a 16th digit) -> None."""
    m = re.fullmatch(r"-?(\d*)\.?(\d*)", s)
    if not m or not 1 <= len(m[1]) + len(m[2]) <= 15:
        return None
    return float(s)


def host_key(s):
    """percent_x100 from the text: hundredths of a percent when the text is unsigned, has at most two decimals and lies
    in 0..100, else 0xFFFF."""
    m = re.fullmatch(r"(\d*)(?:\.(\d{0,2}))?", s)
    if not m or dev_pct(s) is None:
        return 0xFFFF
    k = int(m[1] or 0) * 100 + int((m[2] or "").ljust(2, "0"))
    return k if k <= 10000 else 0xFFFF


def edge_lines(rng, n_lines):
    """Fields of bedMethyl lines (18 or more) whose kept columns are drawn from the edge lists; column 18 is padding."""
    known = sorted(set(NAMES)) + ["c2", "C", "c1000", "NODE_1_length_5_cov_2.50"]
    out = []
    for i in range(n_lines):
        pick = lambda xs: xs[int(rng.integers(len(xs)))]
        f = [pick(known), pick(INT_EDGES[:5]) if rng.random() < 0.8 else pick(INT_EDGES), "0", pick(MOD_EDGES), "9",
             pick(STRAND_EDGES) if rng.random() < 0.3 else pick(["+", "-"]), "0", "1", "255,0,0",
             pick(INT_EDGES[:4]) if rng.random() < 0.8 else pick(INT_EDGES), pick(PCT_EDGES),
             pick(INT_EDGES), "0", "0", "0", "0", pick(INT_EDGES), "0"]
        if i % 7 == 3:
            f += ["extra"] * int(rng.integers(1, 4))  # more than 18 fields: accepted, ignored
        if i % 11 == 5:
            f[17] = "x\ry"  # a '\r' inside column 18 ends the line there; the columns before it are all in
        out.append(f)
    return out


def place_on_block_edges(lines, eols):
    """Text of the lines, padding column 18 of the line before each 4096-byte edge so that the edge falls on that
    line's newline, one byte before it or one byte after it (in turn)."""
    text = bytearray()
    boundary, turn = 4096, 0
    for f, eol in zip(lines, eols):
        line = "\t".join(f).encode()
        end = len(text) + len(line) + len(eol) - 1  # index of the newline
        target = boundary - 1 + turn % 3
        if end <= target < end + 200:
            f = list(f)
            f[17] = f[17] + "p" * (target - end)
            line = "\t".join(f).encode()
            end = target
            turn += 1
        if end >= boundary - 1:
            boundary += 4096
        text += line + eol.encode()
    return bytes(text)


def raw_parse(dl, text, names, mod_types, with_counts=True):
    """nmb_bed_parse on the device text (a tensor, possibly an unaligned slice): every line's columns, dropped lines
    included, and the four status counters."""
    import torch

    from nanomotif_b200._lib import check, lib, ptr

    d = text.device
    n_bytes = int(text.numel())
    scratch = torch.empty((n_bytes + 4095) // 4096 + 1, dtype=torch.int64, device=d)
    n_nl = torch.zeros(1, dtype=torch.int64, device=d)
    check(lib.nmb_index_bytes(ptr(text), n_bytes, 10, ptr(scratch), None, 0, ptr(n_nl), _stream()), "nmb_index_bytes")
    n_newlines = int(n_nl.item())
    newline_pos = torch.empty(max(n_newlines, 1), dtype=torch.int64, device=d)
    check(lib.nmb_index_bytes(ptr(text), n_bytes, 10, ptr(scratch), ptr(newline_pos), n_newlines, ptr(n_nl), _stream()),
          "nmb_index_bytes")
    n_lines = n_newlines + (1 if n_bytes and int(text[-1].item()) != 10 else 0)
    h, ids, off, blob = dl._name_table(names, d)
    keys = torch.from_numpy(dl._modtype_keys(mod_types).view(np.int64)).to(d)
    new = lambda dt: torch.full((max(n_lines, 1),), 99, dtype=dt, device=d)
    cols = dict(contig_id=new(torch.int32), position=new(torch.int64), strand=new(torch.uint8), mod_type=new(torch.uint8),
                Nvalid_cov=new(torch.int64), fraction_mod=new(torch.float64), percent_x100=new(torch.uint16),
                n_mod=new(torch.int64) if with_counts else None, n_diff=new(torch.int64) if with_counts else None)
    status = torch.full((4,), -1, dtype=torch.int32, device=d)
    check(lib.nmb_bed_parse(ptr(text), n_bytes, ptr(newline_pos), n_lines, ptr(h), ptr(ids), ptr(off), ptr(blob), len(names),
                            ptr(keys), len(mod_types), ptr(cols["contig_id"]), ptr(cols["position"]), ptr(cols["strand"]),
                            ptr(cols["mod_type"]), ptr(cols["Nvalid_cov"]), ptr(cols["fraction_mod"]),
                            ptr(cols["percent_x100"]), ptr(cols["n_mod"]), ptr(cols["n_diff"]), ptr(status), _stream()),
          "nmb_bed_parse")
    out = {k: v[:n_lines].cpu().numpy() for k, v in cols.items() if v is not None}
    return out, status.cpu().tolist()


def expected_rows(text, names, mod_types):
    """Per non-empty line, what the parser writes: the oracle's value (load_pileup_text) of every field inside the
    parser's grammar, -1 / NaN for the rest (documented differences: the oracle's int() / float() also read 19+ digit
    integers, 16+ digit decimals, exponents and a leading '+'), plus the status counters."""
    want = O.load_pileup_text(text)
    fields = [ln.split("\r")[0].split("\t") for ln in text.split("\n")]
    fields = [f for f in fields if f != [""]]
    assert len(fields) == len(want["contig"])
    idx = {}
    for i, nm in enumerate(names):
        idx.setdefault(nm, i)  # a repeated name resolves to its first id
    e = {k: [] for k in ("contig_id", "position", "strand", "mod_type", "Nvalid_cov", "fraction_mod", "percent_x100",
                         "n_mod", "n_diff")}
    notnum = unknown = 0
    for i, f in enumerate(fields):
        assert f[0] == want["contig"][i] and f[3] == want["mod_type"][i] and f[5] == want["strand"][i]
        e["contig_id"].append(idx.get(f[0], -1))
        unknown += f[0] not in idx
        for col, k, oracle_key in (("position", 1, "position"), ("Nvalid_cov", 9, "Nvalid_cov"), ("n_mod", 11, "n_mod"),
                                   ("n_diff", 16, "n_diff")):
            v = dev_int(f[k])
            if v is None:
                notnum += 1
                e[col].append(-1)
            else:
                assert v == want[oracle_key][i]
                e[col].append(v)
        p = dev_pct(f[10])
        if p is None:
            notnum += 1
            e["fraction_mod"].append(np.nan)
        else:
            assert want["fraction_mod"][i] is not None and np.float64(p / 100).tobytes() == np.float64(want["fraction_mod"][i]).tobytes()
            e["fraction_mod"].append(want["fraction_mod"][i])
        e["percent_x100"].append(host_key(f[10]))
        e["strand"].append({"+": 0, "-": 1}.get(f[5], 2))
        e["mod_type"].append(mod_types.index(f[3]) if f[3] in mod_types else 255)
    dt = dict(contig_id=np.int32, strand=np.uint8, mod_type=np.uint8, fraction_mod=np.float64, percent_x100=np.uint16)
    return {k: np.array(v, dtype=dt.get(k, np.int64)) for k, v in e.items()}, notnum, unknown


def check_parse(got, status, text, names, mod_types, n_empty):
    want, notnum, unknown = expected_rows(text, names, mod_types)
    live = got["contig_id"] != -2
    assert int((~live).sum()) == n_empty
    assert status == [0, n_empty, notnum, unknown]
    for k, v in want.items():
        assert got[k][live].tobytes() == v.tobytes(), k  # fraction_mod bit for bit, NaN where the oracle has None


def test_parser_edges_against_oracle(dl):
    import torch

    rng = np.random.default_rng(103)
    lines = edge_lines(rng, 1500)
    # the pct edges also at the first and the last line
    lines[0][10], lines[-1][10] = "-0.00", "100.01"
    eols = [("\n", "\r\n", "\n\n", "\r\n\r\n")[int(rng.choice(4, p=[0.7, 0.2, 0.05, 0.05]))] for _ in lines]
    text = place_on_block_edges(lines, eols)
    assert len(text) > 6 * 4096
    n_empty = sum(e.count("\n") - 1 for e in eols)
    buf = torch.zeros(len(text) + 32, dtype=torch.uint8, device="cuda")
    for variant, body in (("newline at the end", text), ("last line without newline", text.rstrip(b"\r\n"))):
        n_empty_v = n_empty if variant == "newline at the end" else n_empty - (eols[-1].count("\n") - 1)
        for off in (0, 1, 7, 13):  # the text as an unaligned slice
            buf[off:off + len(body)] = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
            got, status = raw_parse(dl, buf[off:off + len(body)], NAMES, MOD_TYPES)
            check_parse(got, status, body.decode(), NAMES, MOD_TYPES, n_empty_v)
    # the newline index really sat on the 4096-byte edges: lines ending at, just before and just after each
    nl = np.flatnonzero(np.frombuffer(text, dtype=np.uint8) == 10)
    for r in (-1, 0, 1):
        assert np.isin(np.arange(1, len(text) // 4096) * 4096 + r, nl).sum() >= 1
    # what parse_bedmethyl keeps: known contigs only, in order; rows the parser could not place are not dropped
    rows = dl.parse_bedmethyl(text, NAMES, MOD_TYPES, with_counts=True)
    want, _, _ = expected_rows(text.decode(), NAMES, MOD_TYPES)
    keep = want["contig_id"] >= 0
    assert len(rows) == int(keep.sum())
    for k in ("contig_id", "position", "fraction_mod", "percent_x100", "n_diff"):
        assert getattr(rows, k).cpu().numpy().tobytes() == want[k][keep].tobytes(), k


def test_parser_status_on_malformed_text(dl):
    """Lines the oracle refuses (it raises on fewer than 18 columns and on numbers float() cannot read), against the
    parser's documented rules: a line ends at '\\n' or at its first '\\r'; nothing before its end -> empty; fewer than 18
    fields -> malformed (contig id -2, no other counter); else fields outside the number grammar count as not a number."""
    import torch

    rng = np.random.default_rng(110)
    base = ["c1", "5", "6", "a", "9", "+", "0", "1", "0", "9", "50.00", "4", "0", "0", "0", "0", "1", "0"]
    lines = []
    for i in range(400):
        f = list(base)
        f[1] = str(i)
        kind = i % 8
        if kind == 0:
            f[10] = PCT_GARBAGE[i // 8 % len(PCT_GARBAGE)]
        elif kind == 1:
            f = f[:int(rng.integers(1, 18))]  # 1..17 fields
        elif kind == 2:
            j = int(rng.integers(0, 17))
            f[j] = f[j][:1] + "\r" + f[j][1:]  # a '\r' before column 18 cuts the line short
        elif kind == 3:
            f = [""] * 18  # 18 empty fields: not an empty line, an unknown (empty) contig name and five non-numbers
        elif kind == 4:
            f = ["\r"] + f[1:]  # ends before anything: an empty line
        elif kind == 5:
            f[int(rng.choice([1, 9, 11, 16]))] = rng.choice(["1x", "x", "5.5", "--1", "1-"])
        lines.append("\t".join(f))
    text = "\n".join(lines)  # no final newline
    malformed = empty = notnum = unknown = 0
    want_cid, want_pos, want_frac = [], [], []
    for ln in lines:
        f = ln.split("\r")[0].split("\t")
        if f == [""]:
            empty += 1
            want_cid.append(-2)
        elif len(f) < 18:
            malformed += 1
            want_cid.append(-2)
        else:
            unknown += f[0] not in NAMES
            want_cid.append(NAMES.index(f[0]) if f[0] in NAMES else -1)
            notnum += sum(dev_int(f[k]) is None for k in (1, 9, 11, 16)) + (dev_pct(f[10]) is None)
            want_pos.append(-1 if dev_int(f[1]) is None else dev_int(f[1]))
            want_frac.append(np.nan if dev_pct(f[10]) is None else dev_pct(f[10]) / 100)
    assert malformed > 40 and empty > 40 and unknown > 40 and notnum > 300
    got, status = raw_parse(dl, torch.frombuffer(bytearray(text.encode()), dtype=torch.uint8).cuda(), NAMES, MOD_TYPES)
    assert status == [malformed, empty, notnum, unknown]
    assert got["contig_id"].tolist() == want_cid
    ok = got["contig_id"] != -2
    assert got["position"][ok].tolist() == want_pos
    assert got["fraction_mod"][ok].tobytes() == np.array(want_frac).tobytes()
    with pytest.raises(ValueError, match="fewer than 18"):
        dl.parse_bedmethyl(text.encode(), NAMES, MOD_TYPES)


def test_parser_keys_feed_the_compact_builder(dl):
    """percent_x100 of the parser straight into from_compact: keys on the grid classify like the float rows, 0xFFFF keys
    (off the grid, not a number) are neither class."""
    from nanomotif_b200.device import DeviceAssembly, DevicePileup

    pcts = PCT_EDGES + ["%.2f" % (k / 100) for k in range(0, 10001, 97)] + ["69.99", "70.00", "70.01", "29.99", "30.01"]
    L = len(pcts) + 3
    text = "".join("\t".join(["c", str(i), "0", "a", "9", "+-"[i % 2], "0", "1", "0", "9", p] + ["0"] * 7) + "\n"
                   for i, p in enumerate(pcts))
    rows = dl.parse_bedmethyl(text.encode(), ["c"], ("a",))
    key = rows.percent_x100.cpu().numpy()
    assert (key == 0xFFFF).sum() > 20 and (key <= 10000).sum() > 100
    asm = DeviceAssembly.from_sequences({"c": "A" * L})
    pos, strand = rows.position.cpu().numpy(), rows.strand.cpu().numpy()
    frac = rows.fraction_mod.cpu().numpy()
    for low, high in ((0.3, 0.7), (0.5, 0.5), (0.0, 1.0), (0.7, 0.3)):
        got = decode(DevicePileup.from_compact(asm, pos, strand, key, [0, len(pos)], low, high))
        # the float classification of the rows whose key is on the grid (the others are NaN or off the grid)
        on = key <= 10000
        want = oracle_classes(np.zeros(on.sum(), np.int64), pos[on], strand[on], np.zeros(on.sum(), np.int64), frac[on],
                              [L], 1, low, high)
        assert got == want, (low, high)


# ---------------------------------------------------------------------------------------------------------------------
# class planes: host decoder and the numpy restatement of find_motifs_bin.py:1308-1314
# ---------------------------------------------------------------------------------------------------------------------
def decode(pileup):
    """{(mod type, contig, position, strand, class)} of every set bit of the class records (class 0 methylated,
    1 unmethylated); a bit outside every contig decodes to a position >= the contig's length."""
    from nanomotif_b200 import _lib as L

    asm = pileup.assembly
    rec = pileup.class_records.cpu().numpy().view(np.uint32).reshape(pileup.n_modtypes, asm.n_tiles, 4, L.TILE_WORDS)
    natural = np.ascontiguousarray(rec[..., L.WORD_SLOT])  # slot order -> tile word order
    bits = np.unpackbits(natural.view(np.uint8), axis=-1, bitorder="little")  # bit b of word w at w * 32 + b
    mt, tile, plane, off = np.nonzero(bits)
    g = tile.astype(np.int64) * L.TILE_BP + off
    c = np.searchsorted(asm.starts, g, side="right") - 1
    assert (c >= 0).all()
    p = g - asm.starts[c]
    return set(zip(mt.tolist(), c.tolist(), p.tolist(), (plane >> 1).tolist(), (plane & 1).tolist()))


def oracle_classes(contig_id, position, strand, mod_type, fraction_mod, lengths, n_modtypes, low, high):
    """find_motifs_bin.py:1308-1314 per (mod type, contig): fraction >= high -> methylated, <= low -> unmethylated, on
    the '+' / '-' strand; rows of unknown contigs, mod types or strands take no part, and positions outside the contig
    never meet a motif occurrence (np.isin against indices inside the contig)."""
    cid = np.asarray(contig_id, dtype=np.int64)
    pos = np.asarray(position, dtype=np.int64)
    st = np.asarray(strand, dtype=np.int64)
    mt = np.asarray(mod_type, dtype=np.int64)
    f = np.asarray(fraction_mod, dtype=np.float64)
    lengths = np.asarray(lengths, dtype=np.int64)
    ok = (cid >= 0) & (cid < len(lengths)) & (mt >= 0) & (mt < n_modtypes) & (st >= 0) & (st <= 1)
    ok &= (pos >= 0) & (pos < lengths[np.clip(cid, 0, len(lengths) - 1)])
    out = set()
    for cls, sel in ((0, f >= high), (1, f <= low)):
        i = np.flatnonzero(ok & sel)
        out |= set(zip(mt[i].tolist(), cid[i].tolist(), pos[i].tolist(), st[i].tolist(), [cls] * len(i)))
    return out


# contig ends on word (32), chunk (512) and tile (65536) edges, one position either side, and a 1-bp contig
EDGE_LENGTHS = [65536, 1, 31, 32, 33, 511, 512, 513, 65535, 65537, 3000, 64 * 1024 * 2 + 5]


def edge_rows(rng, lengths, n_modtypes, grid=False):
    """Rows at every edge position of every contig (-1, 0, 1, bits 0 / 31 of words, chunk and tile edges, the contig's
    last tile, len - 1, len, len + 1) plus random ones, with out-of-range ids, mod types and strands mixed in.
    Fractions: the thresholds themselves, their float neighbours, 0, 1, NaN, random; on the percent grid if `grid`."""
    from nanomotif_b200.device import plan_layout

    starts, _ = plan_layout(lengths)
    cid, pos = [], []
    for c, L in enumerate(lengths):
        ps = {-1, 0, 1, 30, 31, 32, 33, 63, 64, 511, 512, 513, L - 33, L - 32, L - 31, L - 2, L - 1, L, L + 1}
        for t in range(int(starts[c]) // 65536, (int(starts[c]) + L) // 65536 + 1):  # tile edges inside the contig
            ps |= {t * 65536 - int(starts[c]) + d for d in (-1, 0, 1)}
        ps |= set(rng.integers(0, L, 40).tolist())
        ps = sorted(p for p in ps if -1 <= p <= L + 1)
        cid += [c] * len(ps)
        pos += ps
    # every position on both strands and '.', under every mod type, one past the last and 255
    combos = np.array([(s, m) for s in (0, 1, 2) for m in list(range(n_modtypes + 1)) + [255]])
    cid, pos = np.repeat(cid, len(combos)), np.repeat(pos, len(combos))
    n = len(pos)
    strand, mt = np.tile(combos[:, 0], n // len(combos)), np.tile(combos[:, 1], n // len(combos))
    cid = np.where(rng.random(n) < 0.05, rng.choice([-1, len(lengths), 1000], n), cid)
    if grid:
        keys = rng.choice([0, 1, 2999, 3000, 3001, 4999, 5000, 5001, 6999, 7000, 7001, 9999, 10000], n)
        keys = np.where(rng.random(n) < 0.3, rng.integers(0, 10001, n), keys)
        frac = (keys / 100.0) / 100.0
    else:
        special = np.array([0.0, 1.0, 0.3, 0.7, 0.5, np.nextafter(0.3, 1), np.nextafter(0.3, 0), np.nextafter(0.7, 1),
                            np.nextafter(0.7, 0), np.nan, -0.0, 0.0001])
        frac = np.where(rng.random(n) < 0.6, special[rng.integers(0, len(special), n)], rng.random(n))
    return cid, pos, strand, mt, frac


def unique_rows(cid, pos, strand, mt, *rest):
    """The first row of each (contig, position, strand, mod type): the class records need unique rows."""
    _, first = np.unique(np.stack([cid, pos, strand, mt]), axis=1, return_index=True)
    first = np.sort(first)
    return (cid[first], pos[first], strand[first], mt[first]) + tuple(a[first] for a in rest)


def test_class_planes_from_columns_at_contig_edges(dl):
    from nanomotif_b200.device import DeviceAssembly, DevicePileup

    rng = np.random.default_rng(104)
    lengths = EDGE_LENGTHS
    asm = DeviceAssembly.from_sequences({f"c{i}": "ACGT" * (L // 4) + "A" * (L % 4) for i, L in enumerate(lengths)})
    assert asm.n_tiles >= 5
    cid, pos, strand, mt, frac = unique_rows(*edge_rows(rng, lengths, 3))
    for low, high in ((0.3, 0.7), (0.5, 0.5), (0.0, 1.0), (0.7, 0.3)):
        p = DevicePileup.from_columns(asm, cid.astype(np.int32), pos, strand, frac, low, high, mt, 3)
        got = decode(p)
        want = oracle_classes(cid, pos, strand, mt, frac, lengths, 3, low, high)
        assert got == want, (low, high, sorted(got ^ want)[:10])
        assert p.duplicate_rows == 0
    # the rows reach every edge: both ends of each contig, bits 0 and 31 of a word, both planes of both strands
    want = oracle_classes(cid, pos, strand, mt, frac, lengths, 3, 0.5, 0.5)
    assert {(q[1], q[2]) for q in want} >= {(c, 0) for c in range(len(lengths))} | {(c, L - 1) for c, L in enumerate(lengths)}
    assert {q[2] % 32 for q in want} >= {0, 31} and {(q[3], q[4]) for q in want} == {(0, 0), (0, 1), (1, 0), (1, 1)}


def test_class_planes_from_compact_against_oracle(dl):
    from nanomotif_b200.device import DeviceAssembly, DevicePileup, compact_rows

    rng = np.random.default_rng(105)
    lengths = EDGE_LENGTHS
    asm = DeviceAssembly.from_sequences({f"c{i}": "ACGT" * (L // 4) + "A" * (L % 4) for i, L in enumerate(lengths)})
    cid, pos, strand, mt, frac = unique_rows(*edge_rows(rng, lengths, 3, grid=True))
    ok = pos >= 0  # compact rows refuse negative positions: those go the float64 way
    cid, pos, strand, mt, frac = cid[ok], pos[ok], strand[ok], mt[ok], frac[ok]
    assert (cid >= len(lengths)).any() and (cid < 0).any()
    rows = compact_rows(cid, pos, strand, frac, mt, len(lengths))
    assert rows is not None
    for low, high in ((0.3, 0.7), (0.5, 0.5), (0.0, 1.0)):
        got = decode(DevicePileup.from_compact(asm, low=low, high=high, n_modtypes=3, **rows))
        want = oracle_classes(cid, pos, strand, mt, frac, lengths, 3, low, high)
        assert got == want, (low, high, sorted(got ^ want)[:10])
        assert got == decode(DevicePileup.from_columns(asm, cid.astype(np.int32), pos, strand, frac, low, high, mt, 3))


def test_dup_count_against_numpy_unique(dl):
    from nanomotif_b200.device import DeviceAssembly, DevicePileup

    rng = np.random.default_rng(106)
    lengths = [5000, 70000, 33]
    asm = DeviceAssembly.from_sequences({f"c{i}": "A" * L for i, L in enumerate(lengths)})
    n = 20000
    cid = rng.integers(-1, 4, n)
    pos = rng.integers(-1, 400, n) * (cid + 1)  # repeats on purpose
    strand, mt = rng.integers(0, 3, n), rng.choice([0, 1, 2, 255], n)
    frac = rng.choice([0.0, 0.2, 0.3, 0.5, 0.7, 0.9, 1.0, np.nan], n)
    low, high = 0.3, 0.7

    def expected(sl):
        """Classified rows minus distinct (contig, position, strand, mod type, class): the rows the planes collapse."""
        c, p, s, m, f = cid[sl], pos[sl], strand[sl], mt[sl], frac[sl]
        ok = (c >= 0) & (c < len(lengths)) & (m < 3) & (s <= 1) & (p >= 0)
        ok &= p < np.asarray(lengths)[np.clip(c, 0, len(lengths) - 1)]
        cls = np.where(f >= high, 0, np.where(f <= low, 1, -1))
        ok &= cls >= 0
        return int(ok.sum()) - len(np.unique(np.stack([c, p, s, m, cls])[:, ok], axis=1).T)

    p = DevicePileup(asm, 3, low, high).clear()
    a, b = slice(0, 12000), slice(8000, n)  # two tables that overlap: repeats across add_columns calls count too
    for sl in (a, b):
        p.add_columns(cid[sl].astype(np.int32), pos[sl], strand[sl], frac[sl], mt[sl])
    both = np.concatenate([np.arange(n)[a], np.arange(n)[b]])
    assert p.duplicate_rows == expected(both) > 1000
    assert decode(p) == oracle_classes(cid, pos, strand, mt, frac, lengths, 3, low, high)
    with pytest.warns(RuntimeWarning):
        one = DevicePileup.from_columns(asm, cid.astype(np.int32), pos, strand, frac, low, high, mt, 3)
    assert one.duplicate_rows == expected(np.arange(n))


# ---------------------------------------------------------------------------------------------------------------------
# the three filters
# ---------------------------------------------------------------------------------------------------------------------
FILTER_NAMES = ["c0", "c1", "c2"]


def filter_table(rng, n, n_pos=60):
    """Rows sorted by (contig, position) of three contigs and three mod types on few positions, so that windows, ties,
    equal positions of several mod types and contig changes are frequent; about one row in ten has an unknown contig
    (-1) or mod type (255).  Fractions at and around the thresholds, NaN."""
    cid = np.where(rng.random(n) < 0.05, -1, rng.integers(0, 3, n))
    pos = rng.integers(0, n_pos, n)
    o = np.lexsort((pos, cid))
    cid, pos = cid[o], pos[o]
    strand = rng.integers(0, 2, n)
    mt = np.where(rng.random(n) < 0.05, 255, rng.integers(0, 3, n))
    special = np.array([0.7, 0.9, 0.9, 1.0, 0.0, 0.5, np.nan, np.nextafter(0.7, 0), np.nextafter(0.7, 1), 0.95])
    frac = np.where(rng.random(n) < 0.7, special[rng.integers(0, len(special), n)], rng.random(n))
    cov = rng.choice([0, 4, 5, 6, 30, -1], n)
    return cid, pos, strand, mt, frac, cov


def device_rows(dl, cid, pos, strand, mt, frac, cov):
    import torch

    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(np.asarray(a).astype(dt))).cuda()
    return dl.DeviceRows(FILTER_NAMES, ("a", "m", "21839"), torch.device("cuda"), contig_id=t(cid, np.int32),
                         position=t(pos, np.int64), strand=t(strand, np.uint8), mod_type=t(mt, np.uint8),
                         Nvalid_cov=t(cov, np.int64), fraction_mod=t(frac, np.float64))


def host_table(cid, pos, strand, mt, frac, cov):
    from nanomotif_b200.pileup import PileupTable

    names = np.array(FILTER_NAMES + ["unknown"], dtype=object)
    mods = np.array(["a", "m", "21839", "x"], dtype=object)
    return PileupTable(names[np.asarray(cid)], np.asarray(pos, np.int64), np.array(["+", "-"], dtype=object)[strand],
                       np.asarray(frac, np.float64), mods[np.minimum(mt, 3)], np.asarray(cov, np.int64))


def kept_positions(rows):
    return rows.position.cpu().numpy(), rows.fraction_mod.cpu().numpy()


@pytest.mark.parametrize("n", [1, 31, 33, 257, 5000])
def test_filters_against_oracle(dl, n):
    """DeviceRows.filter_* (contig and mod type ids; rows of unknown ones belong to no contig_mod group and are dropped by
    the frequency filter) and dataload.filter_pileup* (host tables of names) against the oracle."""
    rng = np.random.default_rng(107 + n)
    cid, pos, strand, mt, frac, cov = filter_table(rng, n)
    t = host_table(cid, pos, strand, mt, frac, cov)
    rows = device_rows(dl, cid, pos, strand, mt, frac, cov)
    valid = (cid >= 0) & (mt < 3)
    for min_cov in (5, 0, -1):  # Nvalid_cov > min_coverage, strict
        want = O.filter_pileup(cov, min_cov)
        np.testing.assert_array_equal(rows.filter_coverage(min_cov).position.cpu().numpy(), pos[want])
        np.testing.assert_array_equal(dl.filter_pileup(t, min_coverage=min_cov).position, pos[want])
    for thr, min_freq, min_mods in ((0.7, 0.0001, 0), (0.7, 0.25, 1), (0.9, 0.5, 2), (0.7, 0.0, -1), (0.95, 0.1, 3)):
        want = O.filter_pileup_minimummod_frequency(t.contig, t.mod_type, frac, thr, min_freq, min_mods)
        np.testing.assert_array_equal(dl.filter_pileup_minimummod_frequency(t, thr, min_freq, min_mods).position, pos[want])
        want = np.zeros(n, dtype=bool)
        want[valid] = O.filter_pileup_minimummod_frequency(t.contig[valid], t.mod_type[valid], frac[valid], thr, min_freq,
                                                           min_mods)
        got = rows.filter_min_mod_frequency(thr, min_freq, min_mods)
        np.testing.assert_array_equal(got.position.cpu().numpy(), pos[want])
        np.testing.assert_array_equal(got.contig_id.cpu().numpy(), cid[want])
    for dist in (0, 1, 8, 1000):
        for thr in (0.7, 0.9):
            want = O.filter_pileup_adjacency_filter(t.contig, t.strand, pos, frac, thr, dist)
            p, f = kept_positions(rows.filter_adjacency(thr, dist))
            np.testing.assert_array_equal(p, pos[want])
            assert f.tobytes() == frac[want].tobytes()
            np.testing.assert_array_equal(dl.filter_pileup_adjacency_filter(t, thr, dist).position, pos[want])


def test_filter_edges_by_hand(dl):
    """Known answers at the comparisons' edges, independent of the oracle."""
    nan = np.nan
    # coverage == threshold is dropped
    rows = device_rows(dl, [0, 0, 0], [1, 2, 3], [0, 0, 0], [0, 0, 0], [0.9] * 3, [4, 5, 6])
    assert rows.filter_coverage(5).position.cpu().tolist() == [3]
    # a group with n_mod == min_mods or n_mod / n_pos == min_freq is dropped; fraction == threshold is not a mod;
    # NaN rows count as positions, not as mods
    f = [0.9, 0.9, 0.7, 0.1, nan, 0.9, 0.9, 0.9, 0.1]
    rows = device_rows(dl, [0] * 5 + [1] * 4, range(9), [0] * 9, [0] * 9, f, [9] * 9)
    assert rows.filter_min_mod_frequency(0.7, 0.4, 1).position.cpu().tolist() == [5, 6, 7, 8]  # 2/5 == 0.4
    assert rows.filter_min_mod_frequency(0.7, 0.3, 2).position.cpu().tolist() == [5, 6, 7, 8]  # 2 mods == 2
    assert rows.filter_min_mod_frequency(0.7, 0.3, 1).position.cpu().tolist() == list(range(9))
    # adjacency: a tie at the window maximum keeps both; fraction == threshold takes part; 4mC and 5mC on one C share a
    # window; NaN neighbours are skipped, NaN rows dropped; a window never reaches into the next contig
    rows = device_rows(dl, [0, 0, 0, 0, 0, 1, 1], [10, 10, 12, 13, 20, 0, 1], [0] * 7, [1, 2, 1, 0, 0, 0, 0],
                       [0.9, 0.9, 0.7, nan, 0.7, 0.8, 0.85], [9] * 7)
    assert rows.filter_adjacency(0.7, 2).fraction_mod.cpu().tolist() == [0.9, 0.9, 0.7, 0.85]
    assert rows.filter_adjacency(0.7, 0).position.cpu().tolist() == [10, 10, 12, 20, 0, 1]
    assert rows.filter_adjacency(0.7, 1000).position.cpu().tolist() == [10, 10, 1]


def test_group_counts_in_a_strided_grid(dl):
    """More rows than one grid of the counting kernel holds (148 * 32 blocks of 256 threads), groups interleaved inside
    every warp and rows of unknown contigs / mod types mixed in: the warp aggregation sees lanes that skip a row."""
    rng = np.random.default_rng(108)
    n = 148 * 32 * 256 + 4099
    cid = rng.integers(-1, 3, n)
    mt = np.where(rng.random(n) < 0.05, 255, rng.integers(0, 3, n))
    frac = rng.choice([0.1, 0.7, 0.8, np.nan, 1.0], n)
    pos = np.arange(n)
    rows = device_rows(dl, cid, pos, np.zeros(n, np.int64), mt, frac, np.full(n, 9))
    valid = (cid >= 0) & (mt < 3)
    n_mod = np.bincount(cid[valid] * 3 + mt[valid], weights=frac[valid] > 0.7)
    middle = int(np.median(n_mod))  # about half of the nine groups have more mods than this
    for thr, min_freq, min_mods in ((0.7, 0.2, middle), (0.7, 0.2, middle - 1), (0.75, 0.4, 0)):
        want = np.zeros(n, dtype=bool)
        want[valid] = O.filter_pileup_minimummod_frequency(cid[valid], mt[valid], frac[valid], thr, min_freq, min_mods)
        got = rows.filter_min_mod_frequency(thr, min_freq, min_mods).position.cpu().numpy()
        np.testing.assert_array_equal(got, pos[want])


# ---------------------------------------------------------------------------------------------------------------------
# end to end
# ---------------------------------------------------------------------------------------------------------------------
def test_text_to_class_planes_end_to_end(dl, tmp_path):
    from test_gpu_ingest import bed_text, write_bgzf

    from nanomotif_b200.device import DeviceAssembly

    rng = np.random.default_rng(109)
    lines, contigs = bed_text(rng, n_contigs=4, length=20000, depth=(3, 30))
    for i in rng.choice(len(lines), len(lines) // 25, replace=False):  # null percentages among the rows
        f = lines[i].split("\t")
        f[10] = "NA" if i % 2 else "null"
        lines[i] = "\t".join(f)
    text = "\n".join(lines) + "\n"
    names = list(contigs)
    lengths = [len(contigs[c]) for c in names]
    mods = ("a", "m", "21839")
    asm = DeviceAssembly.from_sequences(contigs)

    # the oracle chain: load_pileup_text -> filter_pileup -> minimum mod frequency -> adjacency -> classification
    w = O.load_pileup_text(text)
    contig = np.array(w["contig"], dtype=object)
    pos = np.array(w["position"], dtype=np.int64)
    strand = np.array(w["strand"], dtype=object)
    mt = np.array(w["mod_type"], dtype=object)
    frac = np.array([np.nan if v is None else v for v in w["fraction_mod"]], dtype=np.float64)
    k = O.filter_pileup(np.array(w["Nvalid_cov"]), 5)
    k[k] = O.filter_pileup_minimummod_frequency(contig[k], mt[k], frac[k], 0.7, 0.0001, 50)
    k[k] = O.filter_pileup_adjacency_filter(contig[k], strand[k], pos[k], frac[k], 0.7, 8)
    cid = np.array([names.index(c) for c in contig[k]])
    st = np.where(strand[k] == "+", 0, np.where(strand[k] == "-", 1, 2))
    mti = np.array([mods.index(m) for m in mt[k]])
    above_nan = 0
    for i in np.flatnonzero(k & (frac >= 0.7)):  # rows the old np.max oracle would have dropped
        win = (contig == contig[i]) & (strand == strand[i]) & (np.abs(pos - pos[i]) <= 8)
        above_nan += bool(np.isnan(frac[win]).any())
    assert above_nan > 0
    for low, high in ((0.3, 0.7), (0.5, 0.5)):
        want = oracle_classes(cid, pos[k], st, mti, frac[k], lengths, 3, low, high)
        assert len(want) > 1000
        plain = text.encode()
        (tmp_path / "p.bed.gz").write_bytes(write_bgzf(plain))
        for source in (plain, "bgzf"):
            rows = (dl.parse_bedmethyl(source, names, mods) if source != "bgzf"
                    else dl.load_pileup_device(str(tmp_path / "p.bed.gz"), names, mods))
            rows = rows.filter_coverage(5).filter_min_mod_frequency(0.7, 0.0001, 50).filter_adjacency(0.7, 8)
            assert len(rows) == int(k.sum())
            got = decode(rows.class_planes(asm, low, high))
            assert got == want, (low, high, source)
