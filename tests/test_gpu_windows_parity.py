"""K4 (motif-growth step, `csrc/windows.cu`) window by window against the oracle: every extracted window decoded and
compared with `oracle.restate.methylation_windows` at word, chunk, tile and contig edges and around N runs / IUPAC
letters; `nmb_window_hist` with 300 motifs per launch and its `[n_motifs][n]` keep layout; chained filters; the row-range
path (`nmb_window_hist_ranges`) through `WindowPool` round by round against per-slot alive sets kept in numpy; and
`nmb_pssm_kl` against `scipy.stats.entropy` at its special values and on random columns.

Non-ACGT contig letters are written as `N` in the oracle strings: the device treats every one of them as N, where the
reference raises KeyError for IUPAC codes other than N (DESIGN §7)."""
import ctypes as C
import functools
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O

PADDINGS = (0, 1, 16, 20, 30)  # widths 1, 3, 33, 41, 61
TILE, CHUNK, GAP = 65536, 512, 64
LETTERS = "NRYKMSWBDHVnacgtr"  # single letters planted in contig "letters"; lower case is upper-cased (seq.py:55)
N_RUNS = ((3500, 10), (4200, 70))  # (start, length) in contig "letters"
# nmb_pssm_kl is not bit-for-bit scipy.stats.entropy: the device takes CUDA's double log (max error 1 ulp) and may fuse
# the product and the sum into an FMA, scipy takes the host libm's log.  KL_MAX_ULP is the largest distance measured on
# the seeded random columns of test_kl_ulp_distance_to_scipy.  A distance in ulp of the RESULT is not bounded in general
# (the terms p ln(p/q) have both signs and cancel: 515 ulp on a column of test_expand_300_motifs_in_one_launch), so the
# other comparisons measure the difference in units of eps * sum_b |p_b ln(p_b / q_b)|.  KL_TERM_EPS is the largest such
# figure measured over the seeded inputs of this file (10.9, test_expand_300_motifs_in_one_launch; 2.1 on the random
# columns).  Both were measured on an NVIDIA B200 at a 1000 W power limit.
KL_MAX_ULP = 28
KL_TERM_EPS = 11


def _oracle_text(seq: str) -> str:
    return re.sub("[^ACGT]", "N", seq.upper())


@functools.lru_cache(maxsize=1)
def _host():
    """Seeded assembly and pileup-like rows per padding, each edge case asserted present.

    plan_layout keeps >= 64 padding positions after every contig, so no contig can end at the end of the last tile; the
    last contig ends exactly 64 bp before it, the closest it can.  Windows that reach past either end of the position
    space are pinned by test_extract_windows_at_the_ends_of_the_position_space."""
    from nanomotif_b200 import synth
    from nanomotif_b200.device import plan_layout

    rng = np.random.default_rng(20261021)

    def rand(n):
        return synth.random_sequence(rng, n, 0.5).tobytes().decode()

    contigs = {"first": rand(3000)}
    s = bytearray(rand(6000).encode())
    letter_at = [300 + 150 * i for i in range(len(LETTERS))]
    for q, ch in zip(letter_at, LETTERS):
        s[q] = ord(ch)
    for q, n in N_RUNS:
        s[q:q + n] = b"N" * n
    contigs["letters"] = s.decode()
    contigs["long"] = rand(140000)  # holds the tile boundaries 65536 and 131072
    contigs["tiny63"] = rand(63)  # width 61 fits at two positions only
    contigs["one"] = rand(1)
    starts, _ = plan_layout([len(x) for x in contigs.values()])
    last_start = int(starts[-1]) + -(-(len(contigs["one"]) + GAP) // CHUNK) * CHUNK
    end = -(-(last_start + GAP + 200) // TILE) * TILE
    contigs["last"] = rand(end - last_start - GAP)
    names = list(contigs)
    lengths = np.array([len(contigs[n]) for n in names], dtype=np.int64)
    starts, n_tiles = plan_layout(lengths)
    assert starts[0] == 0 and starts[-1] == last_start and starts[-1] + lengths[-1] + GAP == n_tiles * TILE
    long_i, let_i = names.index("long"), names.index("letters")
    tile_bounds = [b for b in range(TILE, n_tiles * TILE, TILE) if starts[long_i] + 40 < b < starts[long_i] + lengths[long_i] - 40]
    assert tile_bounds == [TILE, 2 * TILE]

    rows = {}
    for p in PADDINGS:
        r = []  # (contig, position, strand)

        def both(ci, pos):
            for st in (0, 1):
                r.append((ci, int(pos), st))

        for k in range(32):  # every bit offset of the first column inside a word (long starts on a word)
            both(long_i, 2048 + k + p)
        chunk_b = int(starts[long_i]) + 7 * CHUNK  # a chunk boundary inside one tile
        for d in range(-p - 1, p + 2):
            both(long_i, chunk_b - starts[long_i] + d)
            for b in tile_bounds:
                both(long_i, b - starts[long_i] + d)
        for ci, L in enumerate(lengths):
            for pos in (p - 1, p, p + 1, L - p - 2, L - p - 1, L - p):
                both(ci, pos)
        for q in letter_at + [q for q, _ in N_RUNS] + [q + n - 1 for q, n in N_RUNS] + [q + n // 2 for q, n in N_RUNS]:
            for pos in (q - p, q, q + p):  # the letter at the first, the centre and the last column
                both(let_i, pos)
        ci = rng.choice(len(names), size=4000, p=lengths / lengths.sum())
        rand_rows = np.stack([ci, rng.integers(0, lengths[ci]), rng.integers(0, 2, size=4000)], axis=1)
        a = np.concatenate([np.array(r, dtype=np.int64).reshape(-1, 3), rand_rows])
        frac = np.ones(len(a))
        frac[-4000:][rng.random(4000) < 0.05] = 0.69  # random rows below `high`: never a window
        perm = rng.permutation(len(a))  # row order inside (contig, strand) is the output order
        rows[p] = dict(contig=a[perm, 0], position=a[perm, 1], strand=a[perm, 2].astype(np.uint8), frac=frac[perm])

        # the cases are present among the rows that get a window
        rw = rows[p]
        ok = (rw["frac"] >= 0.7) & (rw["position"] > p) & (rw["position"] < lengths[rw["contig"]] - p)
        g = starts[rw["contig"][ok]] + rw["position"][ok]
        first = g - p
        width = 2 * p + 1
        assert set((first % 32).tolist()) == set(range(32))
        if width + 31 > 64:
            assert np.any(first % 32 + width > 64)  # the third word of take_bits
        if p:
            assert np.any((first // CHUNK != (first + width - 1) // CHUNK) & ((first + width - 1) % TILE >= width))
        for b in tile_bounds:
            for st in (0, 1):
                assert set((g[rw["strand"][ok] == st] - b).tolist()) >= set(range(-p, p + 1))
        for ci, L in enumerate(lengths):
            at = rw["position"][ok][rw["contig"][ok] == ci]
            if L >= 2 * p + 2:
                assert {p + 1, L - p - 1} <= set(at.tolist()), names[ci]
            else:
                assert len(at) == 0
        assert np.any(g + p == n_tiles * TILE - GAP - 1)  # the last column of the last window of the assembly
        at = rw["position"][ok & (rw["contig"] == let_i)]
        for q in letter_at:
            assert {q - p, q, q + p} <= set(at.tolist())
    return dict(contigs=contigs, names=names, lengths=lengths, starts=starts, n_tiles=n_tiles, rows=rows,
                letter_at=letter_at)


def _oracle_windows(h, p, rw=None):
    rw = h["rows"][p] if rw is None else rw
    out = []
    for ci, name in enumerate(h["names"]):
        sel = (rw["contig"] == ci) & (rw["frac"] >= 0.7)
        plus = rw["position"][sel & (rw["strand"] == 0)].tolist()
        minus = rw["position"][sel & (rw["strand"] == 1)].tolist()
        out += O.methylation_windows(_oracle_text(h["contigs"][name]), plus, minus, p)
    return out


def _decode(windows, width: int) -> list[str]:
    """[N, 3] int64 device windows -> strings (bit j = column j; (x, y) = A 00, T 01, G 10, C 11; N bit -> 'N')."""
    w = windows.cpu().numpy().view(np.uint64).reshape(-1, 3)
    if width < 64:
        assert not np.any(w >> np.uint64(width)), "a window has bits set above its width"
    bits = (w[:, :, None] >> np.arange(width, dtype=np.uint64)) & np.uint64(1)
    letters = np.frombuffer(b"ATGC", dtype=np.uint8)[(2 * bits[:, 0] + bits[:, 1]).astype(np.intp)]
    letters[bits[:, 2] == 1] = ord("N")
    return [row.tobytes().decode() for row in letters]


def _assert_windows_equal(got: list, want: list):
    assert len(got) == len(want)
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert not bad, f"{len(bad)} windows differ, first at row {bad[0]}: device {got[bad[0]]} oracle {want[bad[0]]}"


@pytest.fixture(scope="module")
def env():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200 as nmb
    from nanomotif_b200 import growth
    from nanomotif_b200.device import DeviceAssembly

    h = _host()
    asm = DeviceAssembly.from_sequences(h["contigs"])
    assert np.array_equal(asm.starts, h["starts"]) and asm.n_tiles == h["n_tiles"]
    return dict(nmb=nmb, g=growth, torch=torch, asm=asm, h=h)


def _windows(env, p):
    rw = env["h"]["rows"][p]
    return env["g"].methylation_windows(env["asm"], rw["contig"], rw["position"], rw["strand"], rw["frac"], 0.7, p)


# ---- 1. extraction ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("padding", PADDINGS)
def test_windows_equal_the_oracle(env, padding):
    arr = _windows(env, padding)
    want = _oracle_windows(env["h"], padding)
    assert arr.width == 2 * padding + 1 and arr.n_total == arr.n_alive == len(want) and arr.alive is None
    _assert_windows_equal(_decode(arr.windows, arr.width), want)


@pytest.mark.parametrize("padding", (0, 20, 30))
def test_extract_windows_at_the_ends_of_the_position_space(env, padding):
    """nmb_extract_windows called directly at global positions around 0 and around the end of the last tile: columns
    outside [0, n_tiles * 65536) read as N, like the inter-contig padding."""
    import torch
    from nanomotif_b200._lib import check, lib, ptr
    from nanomotif_b200.device import _stream

    h, asm = env["h"], env["asm"]
    end = h["n_tiles"] * TILE
    text = bytearray(b"N" * end)
    for name, s in zip(h["names"], h["starts"]):
        seq = _oracle_text(h["contigs"][name])
        text[s:s + len(seq)] = seq.encode()
    text = "N" * 64 + text.decode() + "N" * 64
    gpos = np.r_[np.arange(-padding - 2, padding + 3), np.arange(end - 3 * GAP - padding, end + padding + 2)]
    gpos = np.repeat(gpos, 2).astype(np.int64)
    strand = np.tile(np.array([0, 1], dtype=np.uint8), len(gpos) // 2)
    want = []
    for g, st in zip(gpos.tolist(), strand.tolist()):
        w = text[64 + g - padding:64 + g + padding + 1]
        want.append(O.reverse_complement_seq(w) if st else w)
    d = asm.device
    gpos_d, strand_d = torch.from_numpy(gpos).to(d), torch.from_numpy(strand).to(d)
    win = torch.empty((len(gpos), 3), dtype=torch.int64, device=d)
    check(lib.nmb_extract_windows(C.byref(asm.view()), ptr(gpos_d), ptr(strand_d), len(gpos), padding, ptr(win),
                                  _stream()), "nmb_extract_windows")
    _assert_windows_equal(_decode(win, 2 * padding + 1), want)


def test_no_window_returns_none(env):
    g, h, asm = env["g"], env["h"], env["asm"]
    p = 20
    L = h["lengths"]
    ci = np.array([0, 0, 1, 1, 3, 3, 4], dtype=np.int64)
    pos = np.array([p, L[0] - p, p, L[1] - p, p, L[3] - p, 0], dtype=np.int64)  # on the strict bound, or in a contig too short
    st = np.array([0, 1, 1, 0, 1, 0, 0], dtype=np.uint8)
    assert O.methylation_windows(h["contigs"]["first"], [p], [L[0] - p], p) == []
    assert g.methylation_windows(asm, ci, pos, st, np.ones(len(ci)), 0.7, p) is None
    assert g.methylation_windows(asm, [0], [100], [0], [0.69], 0.7, p) is None  # below `high`
    assert g.methylation_windows(asm, [], [], [], [], 0.7, p) is None


def test_windows_wider_than_61_are_refused(env):
    g, asm = env["g"], env["asm"]
    for padding in (31, -1):
        with pytest.raises(ValueError):
            g.methylation_windows(asm, [2], [100], [0], [1.0], 0.7, padding)
        with pytest.raises(ValueError):
            g.DeviceDNAarray.from_positions(asm, [2], [100], [0], padding)
    assert g.methylation_windows(asm, [2], [100], [0], [1.0], 0.7, 30).width == 61


# ---- 2. filter + histogram, many motifs per launch -------------------------------------------------------------------
def _random_motif(rng, windows: list, width: int) -> str:
    """A full-width motif built from one of the windows: 1-4 columns fixed to its letter, a class holding it, another
    letter (the source row then fails), or for an N letter '.', 'N', '[ACGT]' or a letter."""
    src = windows[int(rng.integers(len(windows)))]
    toks = ["."] * width
    for col in rng.choice(width, size=int(rng.integers(1, 5)), replace=False):
        b = src[col]
        u = rng.random()
        if b == "N":
            toks[col] = str(rng.choice([".", "N", "[ACGT]", "A"]))
        elif u < 0.5:
            toks[col] = b
        elif u < 0.8:
            others = [c for c in "ACGT" if c != b]
            toks[col] = "[" + "".join(sorted({b, *rng.choice(others, size=int(rng.integers(1, 3)), replace=False)})) + "]"
        else:
            toks[col] = str(rng.choice([c for c in "ACGT" if c != b]))
    return "".join(toks)


@functools.lru_cache(maxsize=1)
def _hist_case():
    """300 width-41 motifs over the padding-20 windows, and the oracle's decisions (rows x motifs)."""
    h = _host()
    p, width = 20, 41
    wins = _oracle_windows(h, p)
    rng = np.random.default_rng(41)
    motifs = ["." * width, "N" * width, "[ACGT]" * width, "A" * width, "." * p + "A" + "." * p, "." * p + "N" + "." * p]
    while len(motifs) < 300:
        motifs.append(_random_motif(rng, wins, width))
    ref = O.one_hot_windows(wins)
    sel = np.stack([O.filter_sequence_matches(ref, O.motif_one_hot(m), True)[0] for m in motifs])
    n_rows = sel.sum(axis=1)
    assert n_rows[0] == len(wins) and n_rows[3] == 0  # all-wildcard and match-nothing
    assert np.sum((n_rows > 0) & (n_rows < len(wins))) > 200
    assert (ref.sum(axis=2) == 4).any(axis=1).sum() > 50  # windows holding N
    return dict(p=p, width=width, wins=wins, motifs=motifs, ref=ref, sel=sel, n=n_rows)


def _column_sums(sel, ref, n_counts_all: int):
    """(motifs, W, 4) column sums of the selected one-hot rows; n_counts_all = 0: N rows (all ones) count for none."""
    oh = ref if n_counts_all else ref * (ref.sum(axis=2, keepdims=True) == 1)
    return (sel.astype(np.int64) @ oh.reshape(len(oh), -1)).reshape(len(sel), *oh.shape[1:])


def _bg(rng, width):
    return rng.dirichlet(np.full(4, 2.0), size=width).T.copy()


def test_expand_300_motifs_in_one_launch(env):
    c = _hist_case()
    arr = _windows(env, c["p"])
    motifs = [env["nmb"].Motif(m, c["p"]) for m in c["motifs"]]
    bg = _bg(np.random.default_rng(5), c["width"])
    n, pssm, kl = arr.expand(motifs, bg)
    np.testing.assert_array_equal(n, c["n"])
    with np.errstate(invalid="ignore"):
        want = _column_sums(c["sel"], c["ref"], 1).transpose(0, 2, 1) / c["n"][:, None, None]
    np.testing.assert_array_equal(pssm, want)  # NaN (0 / 0) for the motifs that keep no row
    live = c["n"] > 0
    _assert_kl(kl[live], np.stack([O.entropy(w, bg) for w in want[live]]), want[live], bg)


@pytest.mark.parametrize("n_counts_all", (0, 1))
@pytest.mark.parametrize("with_alive", (False, True))
def test_window_hist_keep_layout(env, n_counts_all, with_alive):
    """nmb_window_hist with 300 motifs: keep[m][i], hist[m] and n_active[m] against the oracle row by row."""
    import torch
    from nanomotif_b200._lib import check, lib, ptr
    from nanomotif_b200.device import _stream, _to_device
    from nanomotif_b200.motif import window_masks

    c = _hist_case()
    arr = _windows(env, c["p"])
    d = arr.windows.device
    n, m, width = arr.n_total, len(c["motifs"]), c["width"]
    alive_h = np.random.default_rng(3).random(n) < 0.7 if with_alive else np.ones(n, dtype=bool)
    alive = torch.from_numpy(alive_h.astype(np.uint8)).to(d) if with_alive else None
    masks = _to_device(window_masks([env["nmb"].Motif(s, c["p"]) for s in c["motifs"]], width).view(np.uint8).reshape(-1), d)
    hist = torch.full((m, width, 4), -1, dtype=torch.int32, device=d)
    n_active = torch.full((m,), -1, dtype=torch.int64, device=d)
    keep = torch.full((m, n), 0xAB, dtype=torch.uint8, device=d)
    check(lib.nmb_window_hist(ptr(arr.windows), ptr(alive), n, width, ptr(masks), m, n_counts_all, ptr(hist),
                              ptr(n_active), ptr(keep), _stream()), "nmb_window_hist")
    sel = c["sel"] & alive_h[None, :]
    np.testing.assert_array_equal(keep.cpu().numpy(), sel.astype(np.uint8))
    np.testing.assert_array_equal(n_active.cpu().numpy(), sel.sum(axis=1))
    np.testing.assert_array_equal(hist.cpu().numpy(), _column_sums(sel, c["ref"], n_counts_all))


def test_chained_filters(env):
    """keep_matches True -> False -> True on one alive mask: shape, column_counts(1) and exact_pssm() after each step."""
    c = _hist_case()
    arr = _windows(env, c["p"])
    p, ref = c["p"], c["ref"]
    steps = [("." * (p - 3) + "[AG]" + "." * (p + 3), True),
             ("." * (p + 2) + "C" + "." * (p - 2), False),
             ("." * 5 + "[ACT]" + "." * (2 * p - 5), True)]
    rows = np.arange(len(ref))
    for s, keep_matches in steps:
        sel, _ = O.filter_sequence_matches(ref[rows], O.motif_one_hot(s), keep_matches)
        rows = rows[sel]
        assert 0 < len(rows) < len(sel)
        arr = arr.filter_sequence_matches(env["nmb"].Motif(s, p).one_hot(), keep_matches=keep_matches)
        assert arr.shape == (len(rows), 2 * p + 1, 4)
        one = np.zeros(len(ref), dtype=bool)
        one[rows] = True
        np.testing.assert_array_equal(arr.column_counts(1), _column_sums(one[None], ref, 1)[0])
        np.testing.assert_array_equal(arr.exact_pssm(), _column_sums(one[None], ref, 0)[0].T / len(rows))


# ---- 3. row ranges ---------------------------------------------------------------------------------------------------
def _run_rounds(env, pool, slot_oh, slot_wins, rng, n_rounds=4):
    """expand_batch (1-3 requests per slot, the empty slot included, in shuffled order) and remove_batch (at most one
    per slot) against per-slot alive sets kept in numpy; pool.alive outside every slot must stay 1."""
    nmb, width = env["nmb"], pool.width
    p = width // 2
    alive = [np.ones(len(oh), dtype=bool) for oh in slot_oh]
    any_wins = [w for ws in slot_wins for w in ws]
    n_removed = 0
    for _ in range(n_rounds):
        reqs = []
        for s, ws in enumerate(slot_wins):
            for _ in range(int(rng.integers(1, 4))):
                reqs.append((s, nmb.Motif(_random_motif(rng, ws or any_wins, width), p)))
        reqs = [reqs[i] for i in rng.permutation(len(reqs))]
        got = pool.expand_batch(reqs)
        for (s, mo), res in zip(reqs, got):
            sel = alive[s] & O.filter_sequence_matches(slot_oh[s], O.motif_one_hot(mo.string), True)[0]
            if not sel.any():
                assert res is None, (s, mo)
                continue
            assert res is not None and res[0] == sel.sum(), (s, mo)
            np.testing.assert_array_equal(res[1], O.pssm(slot_oh[s][sel]))
        slots = [s for s in range(len(slot_oh)) if rng.random() < 0.7]
        reqs = [(s, nmb.Motif(_random_motif(rng, slot_wins[s] or any_wins, width), p)) for s in slots]
        got = pool.remove_batch(reqs)
        for (s, mo), res in zip(reqs, got):
            hit = O.filter_sequence_matches(slot_oh[s], O.motif_one_hot(mo.string), True)[0]
            n_removed += int((alive[s] & hit).sum())
            alive[s] &= ~hit
            assert res == (int(alive[s].sum()) or None), (s, mo)
        np.testing.assert_array_equal(pool.n_alive, [a.sum() for a in alive])
        want = np.ones(pool.n_total, dtype=np.uint8)
        for s, a in enumerate(alive):
            want[pool.begin[s]:pool.end[s]] = a
        np.testing.assert_array_equal(pool.alive.cpu().numpy(), want)
    assert n_removed > 0
    return alive


def _ranges_call(env, pool, slots, motifs, max_rows, keep_rows):
    import torch
    from nanomotif_b200._lib import check, lib, ptr
    from nanomotif_b200.device import _stream, _to_device
    from nanomotif_b200.motif import window_masks

    d = pool.windows.device
    m = len(slots)
    masks = _to_device(window_masks(motifs, pool.width).view(np.uint8).reshape(-1), d)
    hist = torch.full((m, pool.width, 4), -1, dtype=torch.int32, device=d)
    n_active = torch.full((m,), -1, dtype=torch.int64, device=d)
    rb, re_ = _to_device(pool.begin[slots], d), _to_device(pool.end[slots], d)
    check(lib.nmb_window_hist_ranges(ptr(pool.windows), ptr(pool.alive), pool.n_total, pool.width, ptr(masks), m,
                                     ptr(rb), ptr(re_), max_rows, 1, ptr(hist), ptr(n_active), ptr(keep_rows),
                                     _stream()), "nmb_window_hist_ranges")
    return hist.cpu().numpy(), n_active.cpu().numpy()


def test_window_pool_rounds_from_ranges(env):
    """Slots of 0, 1, 255, 256, 257 and 3000 rows with unowned rows between them."""
    import torch

    g, nmb = env["g"], env["nmb"]
    c = _hist_case()
    arr = _windows(env, c["p"])
    sizes, gap = [0, 1, 255, 256, 257, 3000], 3
    begin = gap + np.cumsum([0] + [s + gap for s in sizes[:-1]])
    end = begin + np.array(sizes)
    assert end[-1] + gap <= arr.n_total
    pool = g.WindowPool.from_ranges(arr.windows, arr.width, begin, end)
    slot_oh = [c["ref"][b:e] for b, e in zip(begin, end)]
    slot_wins = [c["wins"][b:e] for b, e in zip(begin, end)]
    rng = np.random.default_rng(256)
    alive = _run_rounds(env, pool, slot_oh, slot_wins, rng)

    # keep_rows: requested ranges get the decision of their motif, every other row keeps its old value
    d = pool.windows.device
    slots = np.array([5, 0, 2, 4], dtype=np.int64)
    motifs = [nmb.Motif(_random_motif(rng, slot_wins[s] or c["wins"], pool.width), c["p"]) for s in slots]
    keep = torch.full((pool.n_total,), 0xAB, dtype=torch.uint8, device=d)
    alive_before = pool.alive.clone()
    hist, n_active = _ranges_call(env, pool, slots, motifs, int((end[slots] - begin[slots]).max()), keep)
    want = np.full(pool.n_total, 0xAB, dtype=np.uint8)
    for k, (s, mo) in enumerate(zip(slots, motifs)):
        sel = alive[s] & O.filter_sequence_matches(slot_oh[s], O.motif_one_hot(mo.string), True)[0]
        want[begin[s]:end[s]] = sel
        assert n_active[k] == sel.sum()
        np.testing.assert_array_equal(hist[k], slot_oh[s][sel].sum(axis=0))
    np.testing.assert_array_equal(keep.cpu().numpy(), want)
    # max_rows == 0 (only the empty slot asks): zero counts, keep_rows and alive untouched
    keep0 = keep.clone()
    hist, n_active = _ranges_call(env, pool, np.array([0, 0]), motifs[:2], 0, keep)
    assert not hist.any() and not n_active.any()
    assert torch.equal(keep, keep0) and torch.equal(pool.alive, alive_before)
    n_alive = pool.n_alive.copy()
    assert pool.expand_batch([(0, motifs[0]), (0, motifs[1])]) == [None, None]
    assert pool.remove_batch([(0, motifs[0])]) == [None]
    assert torch.equal(pool.alive, alive_before) and np.array_equal(pool.n_alive, n_alive)


def test_window_pool_rounds_from_prepare_searches(env):
    """The same rounds on the pool growth.prepare_searches builds for a three-bin MultiBinScorer; its windows are
    first held against the oracle's windows of each bin."""
    from nanomotif_b200 import synth

    nmb, g = env["nmb"], env["g"]
    rng = np.random.default_rng(3)
    bins, cols = {}, {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod")}
    for b, lens in (("b0", (9000, 4000)), ("b1", (1500,)), ("b2", (6000, 300, 5000))):
        bins[b] = {}
        for i, L in enumerate(lens):
            name = f"{b}_{i}"
            seq = synth.random_sequence(rng, L, 0.5, 3e-4 if L > 1000 else 0.0)
            bins[b][name] = seq.tobytes().decode()
            pl = synth.synth_pileup(seq, rng, depth=20, mod_types=("a",), planted=(("GATC", 1, "a"),))
            n = len(pl["position"])
            cols["contig"].append(np.full(n, name, dtype=object))
            cols["position"].append(pl["position"])
            cols["strand"].append(np.where(pl["strand"] == 0, "+", "-").astype(object))
            cols["mod_type"].append(np.full(n, "a", dtype=object))
            cols["fraction_mod"].append(pl["fraction_mod"])
    perm = rng.permutation(sum(len(x) for x in cols["position"]))
    pile = {k: np.concatenate(v)[perm] for k, v in cols.items()}
    multi = nmb.MultiBinScorer(pile, bins, ["a"], 0.3, 0.7)
    p = 20
    with pytest.raises(ValueError):
        g.prepare_searches(multi, "a", 31, 0.7, seeds=[1, 2, 3])
    pool, _, totals = g.prepare_searches(multi, "a", p, 0.7, seeds=[1, 2, 3])
    slot_wins = []
    for b, contigs in bins.items():
        ws = []
        for name, seq in contigs.items():
            sel = (pile["contig"] == name) & (pile["fraction_mod"] >= 0.7)
            ws += O.methylation_windows(_oracle_text(seq), pile["position"][sel & (pile["strand"] == "+")].tolist(),
                                        pile["position"][sel & (pile["strand"] == "-")].tolist(), p)
        slot_wins.append(ws)
    assert totals == [len(w) for w in slot_wins] and min(totals) > 0
    for s, ws in enumerate(slot_wins):
        _assert_windows_equal(_decode(pool.windows[pool.begin[s]:pool.end[s]], pool.width), ws)
    _run_rounds(env, pool, [O.one_hot_windows(w) for w in slot_wins], slot_wins, np.random.default_rng(9))


# ---- 4. PSSM and KL --------------------------------------------------------------------------------------------------
def _ulp_distance(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """|a - b| in units in the last place of float64 (the distance between their positions on the ordered line)."""
    def ordered(x):
        i = np.ascontiguousarray(x, dtype=np.float64).view(np.int64)
        return np.where(i < 0, -(i & np.int64(0x7FFFFFFFFFFFFFFF)), i)

    return np.abs(ordered(a) - ordered(b))


def _kl_error_in_term_eps(got, want, pssm, bg):
    """|got - want| / (eps * sum_b |p_b ln(p_b / q_b)|) per finite column; pssm (..., 4, W), bg (4, W)."""
    from scipy.special import rel_entr

    with np.errstate(invalid="ignore", divide="ignore"):
        terms = rel_entr(pssm / pssm.sum(axis=-2, keepdims=True), bg / bg.sum(axis=0, keepdims=True))
    scale = np.abs(terms).sum(axis=-2)
    fin = np.isfinite(want)
    return np.abs(got[fin] - want[fin]) / (np.finfo(np.float64).eps * np.maximum(scale[fin], np.finfo(np.float64).tiny))


def _assert_kl(got, want, pssm, bg):
    """Non-finite values equal exactly (NaN == NaN, inf == inf), finite values within KL_TERM_EPS."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
    np.testing.assert_array_equal(np.isinf(got), np.isinf(want))
    inf = np.isinf(want)
    np.testing.assert_array_equal(got[inf], want[inf])
    err = _kl_error_in_term_eps(got, want, pssm, bg)
    assert not err.size or err.max() <= KL_TERM_EPS, f"KL differs from scipy by {err.max():.2f} eps of its terms"


def _pssm_kl_call(hist, n_active, bg):
    import torch
    from nanomotif_b200._lib import check, lib, ptr
    from nanomotif_b200.device import _stream

    d = torch.device("cuda", torch.cuda.current_device())
    m, width = hist.shape[:2]
    h = torch.from_numpy(np.ascontiguousarray(hist, dtype=np.int32)).to(d)
    n = torch.from_numpy(np.ascontiguousarray(n_active, dtype=np.int64)).to(d)
    q = torch.from_numpy(np.ascontiguousarray(bg, dtype=np.float64)).to(d)
    pssm = torch.empty((m, 4, width), dtype=torch.float64, device=d)
    kl = torch.empty((m, width), dtype=torch.float64, device=d)
    check(lib.nmb_pssm_kl(ptr(h), ptr(n), m, width, ptr(q), ptr(pssm), ptr(kl), _stream()), "nmb_pssm_kl")
    return pssm.cpu().numpy(), kl.cpu().numpy()


def test_pssm_kl_special_values(env):
    """p = 0 with q = 0 (0 ln 0 = 0), p > 0 with q = 0 (inf), an all-zero background column and an all-zero
    count column (NaN), n_active = 0, and counts above n_active (an N row counts for all four bases)."""
    cols = [  # (counts A T G C, background A T G C)
        ([10, 0, 0, 0], [1.0, 0, 0, 0]),
        ([5, 5, 0, 0], [0.5, 0, 0.5, 0]),
        ([3, 3, 2, 2], [0.0, 0, 0, 0]),
        ([1, 2, 3, 4], [0.1, 0.2, 0.3, 0.4]),
        ([0, 0, 0, 0], [0.25, 0.25, 0.25, 0.25]),
        ([2, 3, 0, 5], [0.3, 0.3, 0.2, 0.2]),
        ([0, 9, 1, 0], [0.0, 0.5, 0.5, 0]),
    ]
    width = len(cols)
    bg = np.array([q for _, q in cols], dtype=np.float64).T.copy()
    counts = np.array([h for h, _ in cols], dtype=np.int32)
    hist = np.stack([counts, np.zeros_like(counts), counts + 3])
    n_active = np.array([10, 0, 7], dtype=np.int64)
    pssm, kl = _pssm_kl_call(hist, n_active, bg)
    with np.errstate(invalid="ignore", divide="ignore"):
        want = hist.transpose(0, 2, 1) / n_active[:, None, None]
        want_kl = np.stack([O.entropy(w, bg) for w in want])
    np.testing.assert_array_equal(pssm, want)
    assert np.isinf(want_kl[0, 1]) and np.isnan(want_kl[0, 2]) and np.isnan(want_kl[0, 4]) and want_kl[0, 0] == 0
    assert np.isnan(want_kl[1]).all()
    _assert_kl(kl, want_kl, want, bg)


def test_kl_ulp_distance_to_scipy(env):
    """2000 random finite columns (some counts 0): the device KL against scipy.stats.entropy, within KL_MAX_ULP and
    KL_TERM_EPS."""
    rng = np.random.default_rng(2000)
    m, width = 50, 40
    n_active = rng.integers(1, 5000, size=m)
    hist = rng.integers(0, n_active[:, None, None] + 1, size=(m, width, 4))
    hist[rng.random(hist.shape) < 0.05] = 0
    hist[:, :, 0] += hist.sum(axis=2) == 0  # no all-zero count column
    bg = rng.dirichlet(np.full(4, 1.5), size=width).T.copy()
    pssm, kl = _pssm_kl_call(hist, n_active, bg)
    want = hist.transpose(0, 2, 1) / n_active[:, None, None]
    np.testing.assert_array_equal(pssm, want)
    want_kl = np.stack([O.entropy(w, bg) for w in want])
    assert np.isfinite(want_kl).all()
    worst = int(_ulp_distance(kl, want_kl).max())
    err = _kl_error_in_term_eps(kl, want_kl, want, bg)
    print(f"nmb_pssm_kl vs scipy.stats.entropy over {m * width} columns: max {worst} ulp, {err.max():.3f} eps of the "
          f"terms, {np.mean(kl == want_kl):.3f} of the columns bit-identical")
    assert worst <= KL_MAX_ULP
    assert err.max() <= KL_TERM_EPS


def test_kl_children_match_the_oracle(env):
    """For the 300 expansions of test_expand_300_motifs_in_one_launch that keep rows: growth.kl_children with the
    device KL picks the same column and the same children as the oracle's scipy-based restatement."""
    c = _hist_case()
    g, nmb, p = env["g"], env["nmb"], c["p"]
    arr = _windows(env, p)
    motifs = [nmb.Motif(m, p) for m in c["motifs"]]
    bg = _bg(np.random.default_rng(6), c["width"])
    n, pssm, kl = arr.expand(motifs, bg)
    with_children = 0
    for k in np.flatnonzero(n > 0):
        sel = c["sel"][k]
        _, want = O.kl_children(motifs[k].string, p, O.pssm(c["ref"][sel]), bg)
        got = g.kl_children(motifs[k], pssm[k], bg, kl=kl[k])
        assert [(x.string, x.mod_position) for x in got] == want, motifs[k]
        with_children += bool(want)
    assert 50 < with_children < int((n > 0).sum())
