"""K2's sibling runs on generated work lists, held to the general path bit for bit and to the oracle: the split position
at every distance from the modified base (0, +-1, +-31, +-32, +-33, +-61 and random) in one- and two-word-halo launches,
length-1 runs (the all-wildcard parent), runs of 2 to 32 members cut by blocks of 2 to 32 motifs, duplicates inside
runs, runs broken by members that strip shorter, adjacent runs at another position, and multi-job launches whose motif
arrays link across job boundaries.  Pileup rows sit at every base, so a member with any set at the modified base counts.

The generator is seeded; `_coverage` mirrors on the host (motif.sibling_links / sibling_runs) the runs each launch forms
and the tests assert that every (split distance x halo words x run length) bucket holds a run, so a generator that
drifts to lists without runs fails instead of checking the general path against itself."""
import contextlib
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O  # the checker, never the thing under test

SETS = list("ACGT") + ["[" + "".join(c) + "]" for k in (2, 3) for c in itertools.combinations("ACGT", k)]  # 14 sets
EDGE_DELTAS = (0, 1, -1, 31, -31, 32, -32, 33, -33, 61, -61)
NEW_DELTAS = {0, 32, -32, 33, -33, 61, -61}  # split distances no hand-made list of test_gpu_siblings.py reaches
RUN_SIZES = (2, 3, 4, 5, 8, 32)
LENGTHS = (1, 2, 31, 32, 33, 62)  # drawn with weight: one- and two-word halos on both sides of the switch
MPIS = (None, 2, 3, 5, 7, 16, 32)
FRACTIONS = (0.0, 0.3, 0.31, 0.5, 0.69, 0.7, 1.0)  # both thresholds exactly, and their neighbours


def _bucket(delta):
    return delta if delta in EDGE_DELTAS else "other"


def _size_bucket(n):
    return "2" if n == 2 else "3-4" if n <= 4 else "5-8" if n <= 8 else "9-32"


def _token(rng, interior, dot=0.4):
    u = rng.random()
    if interior and u < dot:
        return "."
    return SETS[int(rng.integers(4, 14))] if u > 0.8 else "ACGT"[int(rng.integers(4))]


def _parent(rng, L, canonical, mp):
    dot = 0.95 if L > 20 else 0.35  # sparse long motifs: search-like, and the oracle's time grows with constrained tokens
    toks = [_token(rng, 0 < i < L - 1 and i != mp, dot) for i in range(L)]  # a set at the modified base
    if canonical:
        toks[mp] = canonical
    return toks


def _members(rng, toks, j, mp, r, canonical):
    """r motifs that are `toks` with sets at j drawn from the 14 sets (and '.' inside), duplicates mixed in; at an end
    j a member may get '.' so that it strips shorter and breaks the run."""
    L = len(toks)
    pool = SETS + (["."] if 0 < j < L - 1 else [])
    sets = []
    for k in range(r):
        sets.append(sets[-1] if k and rng.random() < 0.15 else pool[int(rng.integers(len(pool)))])
    if j in (0, L - 1) and j != mp and L > 1 and rng.random() < 0.3:
        sets[int(rng.integers(1, r))] = "."
    out = []
    for s in sets:
        t = list(toks)
        t[j] = s
        out.append(("".join(t), mp))
    return out


def _case(rng, max_len, canonical=None, delta=None, r=None, L=None, far=False):
    """One run, and an adjacent run of the same parent at another position now and then: (motifs, delta, members of
    the first run).  delta=None draws it; far=True puts the modified base at >= 32 with a positive delta."""
    while True:
        d = int(rng.integers(1, 30)) if far else int(rng.integers(-(max_len - 1), max_len)) if delta is None else delta
        if canonical and d == 0:
            if delta == 0:
                return None  # every member keeps the canonical base at the modified position
            continue
        if L is not None:
            n = L
        else:
            fits = [x for x in LENGTHS if abs(d) < x <= max_len]
            n = int(rng.choice(fits)) if fits and rng.random() < 0.6 else int(rng.integers(abs(d) + 1, max_len + 1))
        lo, hi = max(32 if far else 0, -d), min(n - 1, n - 1 - d)
        if lo > hi:
            continue
        mp = hi if rng.random() < 0.3 else int(rng.integers(lo, hi + 1))
        j = mp + d
        toks = _parent(rng, n, canonical, mp)
        motifs = _members(rng, toks, j, mp, r if r is not None else int(rng.choice(RUN_SIZES)), canonical)
        first = len(motifs)
        others = [x for x in range(n) if x != j and not (canonical and x == mp)]
        if others and rng.random() < 0.35:
            motifs += _members(rng, toks, int(rng.choice(others)), mp, int(rng.choice(RUN_SIZES[:4])), canonical)
        return motifs, d, first


def _single(rng, max_len, canonical=None):
    L = int(rng.integers(1, max_len + 1))
    mp = int(rng.integers(L))
    toks = _parent(rng, L, canonical, mp)
    if L == 1 and toks[0] == ".":
        toks[0] = "A"
    return "".join(toks), mp


def fuzz_list(seed, max_len, canonical=None, scale=1):
    """Seeded work list: (motif string, mod_pos) in K2's alphabet, and the indices of the members of runs in the
    buckets the hand-made lists never reach (delta 0, +-32, +-33, +-61, length 1, far modified base with delta > 0).
    Every split-distance bucket that fits `max_len` gets one run of every size in RUN_SIZES (times `scale`), plus
    length-1 runs and runs whose modified base is at >= 32; runs are interleaved with unrelated motifs.  The list
    starts with a 32-member run (one whole block at 32 motifs per item) of length `max_len` and, for two-word halos,
    the next run has length 33: lengths 32 and 33 side by side."""
    rng = np.random.default_rng([seed, 2024])
    deltas = [d for d in EDGE_DELTAS if abs(d) < max_len and not (canonical and d == 0)] + [None]
    plan = [dict(delta=d, r=r) for d in deltas for r in RUN_SIZES for _ in range(scale)]
    if not canonical:
        plan += [dict(delta=0, r=r, L=1) for r in (2, 4, 32)]
    if max_len > 32:
        plan += [dict(far=True, L=62, r=r) for r in RUN_SIZES]
    order = rng.permutation(len(plan))
    plan = [dict(delta=-1 if canonical else 0, r=32, L=max_len)] + [plan[i] for i in order]
    if max_len > 32:
        plan.insert(1, dict(delta=32, r=5, L=33))
    out, new = [], []
    for k, spec in enumerate(plan):
        got = _case(rng, max_len, canonical, **spec)
        if got is None:
            continue
        motifs, d, first = got
        if d in NEW_DELTAS or spec.get("L") == 1 or spec.get("far"):
            new += range(len(out), len(out) + first)
        out += motifs
        if k and rng.random() < 0.4:
            out += [_single(rng, max_len, canonical) for _ in range(int(rng.integers(1, 3)))]
    return out, new


def _coverage(packed, jobs, mpi):
    """Runs K2 forms in one launch (host mirror): {(delta bucket, halo words, size bucket): runs}.  jobs: [(motif
    begin, motif count)]; every job's range is cut into blocks of `mpi` motifs."""
    from nanomotif_b200.motif import sibling_links, sibling_runs

    links = sibling_links(packed)
    H = 1 if int(packed["len"].max()) <= 32 else 2
    out = {}
    if mpi < 2:
        return out  # one motif per item: the general path
    for begin, count in jobs:
        for b in range(begin, begin + count, mpi):
            for first, n, j in sibling_runs(links, b, min(mpi, begin + count - b)):
                key = (_bucket(j - int(packed["mod_pos"][first])), H, _size_bucket(n))
                out[key] = out.get(key, 0) + 1
    return out


def _required(H):
    deltas = [d for d in EDGE_DELTAS if abs(d) < 32 * H] + ["other"]
    return {(d, H, s) for d in deltas for s in ("2", "3-4", "5-8", "9-32")}


@contextlib.contextmanager
def _k2(families, balanced=True):
    from nanomotif_b200 import device as D

    old = D.FAMILIES, D.BALANCED
    try:
        D.FAMILIES, D.BALANCED = families, balanced
        yield
    finally:
        D.FAMILIES, D.BALANCED = old


@contextlib.contextmanager
def _motifs_per_item(mpi):
    """Blocks of `mpi` motifs for launches that choose their own block size (MultiBinScorer.score_batch_device): on
    test-sized inputs the automatic choice is one motif per item, where no sibling run forms.  None = automatic."""
    from nanomotif_b200 import device as D

    old = D.choose_motifs_per_item
    try:
        if mpi is not None:
            D.choose_motifs_per_item = lambda jobs, sms: mpi
        yield
    finally:
        D.choose_motifs_per_item = old


def _contig(rng, L, kind):
    seq = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=L, p=[0.35, 0.15, 0.15, 0.35]).copy()
    if kind == 1 and L > 3:  # N at the very ends
        seq[0] = seq[-1] = ord("N")
    elif kind == 2 and L > 50:  # IUPAC letters inside: those warps score the members one by one
        for s in rng.integers(0, L - 5, 3):
            seq[s:s + int(rng.integers(1, 5))] = ord(rng.choice(list("NRYK")))
    if kind == 0 and L > 50:  # lower-case stretches: the base itself (the reference upper-cases the assembly on load)
        s = int(rng.integers(0, L - 20))
        seq[s:s + 20] += 32
    return seq.tobytes().decode()


def _rows(rng, name, L, cols, mod_types):
    """Rows on both strands at ~70 % of all positions -- every base, not only the canonical one."""
    for mt in mod_types:
        for strand in "+-":
            pos = np.flatnonzero(rng.random(L) < 0.7).astype(np.int64)
            cols["contig"].append(np.full(len(pos), name, dtype=object))
            cols["position"].append(pos)
            cols["strand"].append(np.full(len(pos), strand, dtype=object))
            if "mod_type" in cols:
                cols["mod_type"].append(np.full(len(pos), mt, dtype=object))
            cols["fraction_mod"].append(rng.choice(FRACTIONS, size=len(pos)))


def _lengths(rng):
    """Contigs of 1-80 bp (many per warp), 400-700 bp, 1-4 kbp, 20-70 kbp and one that crosses tiles."""
    lengths = np.concatenate([rng.integers(1, 80, 25), rng.integers(400, 700, 12), rng.integers(1000, 4000, 10),
                              rng.integers(20000, 70000, 1), [135_000]])
    rng.shuffle(lengths)
    return [int(x) for x in lengths]


@pytest.fixture(scope="module")
def nmb():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200 as nmb

    return nmb


@pytest.fixture(scope="module")
def one_bin(nmb):
    rng = np.random.default_rng(5)
    contigs, cols = {}, {k: [] for k in ("contig", "position", "strand", "fraction_mod")}
    for i, L in enumerate(_lengths(rng)):
        contigs[f"f{i}"] = _contig(rng, L, i % 3)
        _rows(rng, f"f{i}", L, cols, ("a",))
    pile = {k: np.concatenate(v) for k, v in cols.items()}
    upper = {name: seq.upper() for name, seq in contigs.items()}  # what the oracle sees (seq.py:55)
    by_contig = {}
    for name in contigs:
        sel = pile["contig"] == name
        by_contig[name] = (pile["position"][sel], pile["strand"][sel], pile["fraction_mod"][sel])
    lists = {H: fuzz_list(H, 32 if H == 1 else 62) for H in (1, 2)}  # max length 32: one-word halos; 62: two
    return dict(contigs=contigs, upper=upper, pile=pile, by_contig=by_contig, lists=lists,
                scorer=nmb.BinScorer(pile, contigs, 0.3, 0.7))


def _motifs(nmb, specs):
    return [nmb.Motif(s, p) for s, p in specs]


def test_every_bucket_holds_a_run(nmb, one_bin):
    """The runs the launches of the tests below form, on the host mirror."""
    import torch

    from nanomotif_b200 import device as D
    from nanomotif_b200.motif import pack_motifs

    for H, (specs, _) in one_bin["lists"].items():
        packed = pack_motifs(_motifs(nmb, specs))
        assert (1 if int(packed["len"].max()) <= 32 else 2) == H
        total = {}
        for mpi in MPIS:
            if mpi is None:
                jobs, _ = one_bin["scorer"]._jobs(len(specs), False)
                mpi = D.choose_motifs_per_item(jobs, D.sm_count(torch.device("cuda", 0)))
            for k, v in _coverage(packed, [(0, len(specs))], mpi).items():
                total[k] = total.get(k, 0) + v
        missing = _required(H) - set(total)
        assert not missing, f"H={H}: no run in {sorted(missing, key=str)}"
        print(f"H={H}: {len(specs)} motifs; runs per (delta, H, size): {dict(sorted(total.items(), key=str))}")


def test_split_equals_general_path(nmb, one_bin):
    """Whole bin and per contig, every block size, dynamic and static scheduling: bit for bit."""
    scorer = one_bin["scorer"]
    for H, (specs, _) in one_bin["lists"].items():
        motifs = _motifs(nmb, specs)
        with _k2(False):
            general = scorer.counts_by_strand(motifs, motifs_per_item=4).cpu().numpy()
            general_pc = scorer.counts_by_strand(motifs, per_contig=True, motifs_per_item=4).cpu().numpy()
        assert int(general.sum()) > 100000
        for balanced in (True, False):
            with _k2(True, balanced):
                for mpi in MPIS:
                    got = scorer.counts_by_strand(motifs, motifs_per_item=mpi).cpu().numpy()
                    np.testing.assert_array_equal(got, general, err_msg=f"H={H} balanced={balanced} mpi={mpi}")
                    got = scorer.counts_by_strand(motifs, per_contig=True, motifs_per_item=mpi).cpu().numpy()
                    np.testing.assert_array_equal(got, general_pc, err_msg=f"per contig H={H} balanced={balanced} mpi={mpi}")


def test_new_buckets_against_oracle(nmb, one_bin):
    """Every member of a run in the new buckets per contig against the oracle (once per distinct motif: duplicates in
    a run must get the same rows), a seeded sample of the rest per bin."""
    scorer, contigs, by_contig, pile = one_bin["scorer"], one_bin["upper"], one_bin["by_contig"], one_bin["pile"]
    names = pile["contig"].astype(str)  # the oracle selects each contig's rows by name: faster on a str array
    keys = ("index_meth_fwd", "index_nonmeth_fwd", "index_meth_rev", "index_nonmeth_rev")
    rng = np.random.default_rng(11)
    for H, (specs, new) in one_bin["lists"].items():
        with _k2(True):
            per = scorer.counts_by_strand(_motifs(nmb, specs), per_contig=True, motifs_per_item=32).cpu().numpy()
        assert len(new) > 100
        want = {}
        for mi in new:
            if specs[mi] not in want:
                s, p = specs[mi]
                want[specs[mi]] = [[len(O.motif_model_contig(*by_contig[name], seq, s, p, 0.3, 0.7, fast=True)[2][k])
                                    for k in keys] for name, seq in contigs.items()]
            np.testing.assert_array_equal(per[mi], want[specs[mi]], err_msg=f"H={H} {specs[mi]}")
        rest = sorted(set(range(len(specs))) - set(new))
        for mi in rng.choice(rest, size=12, replace=False).tolist():
            s, p = specs[mi]
            w = O.motif_model_bin(names, pile["position"], pile["strand"], pile["fraction_mod"], contigs, s, p, fast=True)
            assert (int(per[mi, :, [0, 2]].sum()), int(per[mi, :, [1, 3]].sum())) == w, (H, s, p)


def test_multi_job_launch(nmb):
    """One request per (bin, mod type) of six bins in ONE launch: consecutive bins share a tile, one bin is a single
    short contig, one has no rows; the motif arrays of consecutive jobs link across the job boundary."""
    from nanomotif_b200.motif import pack_motifs, sibling_links

    rng = np.random.default_rng(17)
    mod_types = ("a", "m", "21839")
    layout = {"b0": (600, 3000, 45), "b1": (60,), "b2": (140_000,), "b3": (2000, 2500), "b4": (5, 70, 30_000, 12),
              "b5": (45_000, 62_000)}
    bins, cols = {}, {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod")}
    for b, lens in layout.items():
        bins[b] = {}
        for i, L in enumerate(lens):
            name = f"{b}_c{i}"
            bins[b][name] = _contig(rng, L, i % 3)
            if b != "b3":  # a bin without rows
                _rows(rng, name, L, cols, mod_types)
    pile = {k: np.concatenate(v) for k, v in cols.items()}
    scorer = nmb.MultiBinScorer(pile, bins, mod_types, 0.3, 0.7)
    ctxs = [scorer.context(b, mt) for b in bins for mt in mod_types]
    spans = [(c.tile_begin, c.tile_begin + c.tile_count) for c in ctxs[::len(mod_types)]]
    assert any(s[1] - 1 == t[0] for s, t in zip(spans, spans[1:]))  # consecutive bins share a tile
    lists = [fuzz_list(100 + k, 62)[0] for k in range(len(ctxs))]
    for k in range(len(lists) - 1):  # every job ends with a run whose members open the next job's list
        lists[k] = lists[k] + lists[k + 1][:2]
    requests = [(c, _motifs(nmb, specs)) for c, specs in zip(ctxs, lists)]
    flat = [m for _, ms in requests for m in ms]
    links = sibling_links(pack_motifs(flat))
    starts = np.cumsum([0] + [len(s) for s in lists[:-1]])
    assert (links[starts[1:]] != 0).any()  # some job's first motif is linked to the previous job's last one
    with _k2(False), _motifs_per_item(4):
        general = [c.tolist() for c in scorer.score_batch(requests)]
    packed = pack_motifs(flat)
    for mpi in (None, 5, 32):
        if mpi is not None:
            jobs = [(int(a), len(s)) for a, s in zip(starts, lists)]
            assert sum(_coverage(packed, jobs, mpi).values()) > 500
        for balanced in (True, False):
            with _k2(True, balanced), _motifs_per_item(mpi):
                got = [c.tolist() for c in scorer.score_batch(requests)]
            assert got == general, f"mpi={mpi} balanced={balanced}"
    assert all(sum(map(sum, g)) == 0 for (c, _), g in zip(requests, general) if c.bin_name == "b3")
    assert sum(sum(map(sum, g)) for g in general) > 100000
    for k, (ctx, ms) in enumerate(requests):
        sel = np.isin(pile["contig"], list(bins[ctx.bin_name])) & (pile["mod_type"] == ctx.mod_type)
        cols_b = [pile[c][sel] for c in ("contig", "position", "strand", "fraction_mod")]
        for mi in np.random.default_rng(k).choice(len(ms), size=4, replace=False).tolist():
            upper = {name: seq.upper() for name, seq in bins[ctx.bin_name].items()}
            want = O.motif_model_bin(*cols_b, upper, lists[k][mi][0], lists[k][mi][1], fast=True)
            assert tuple(general[k][mi]) == want, (ctx.bin_name, ctx.mod_type, lists[k][mi])
