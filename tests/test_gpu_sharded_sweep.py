"""The sharded per-bin sweep (sharding.ShardedBinSweep) on CUDA devices, world size 2: every bin's finished histograms on
its designated rank, every candidate frame, and every count equal those of the unsharded BinSweep over all bins.  With
>= 2 GPUs the ranks use NCCL on their own devices; on a one-GPU box both ranks share cuda:0 and the collectives run over
gloo (CUDA tensors).  Each rank compares against its own unsharded sweep and reports what differs, so that a failed
check on one rank cannot leave the other waiting in a collective."""
import os
import socket
import traceback

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MOD_TYPES = ("a", "m", "21839")
CANON = {"a": "A", "m": "C", "21839": "C"}
MIN_MEAN, MIN_MOD = 0.7, 5
PLANTED = (("GATC", 1, "a"), ("CC[AT]GG", 1, "m"), ("GAATTC", 2, "a"), ("GCAC......GTT", 2, "a"), ("CCGG", 0, "21839"),
           ("TCGA", 3, "a"), ("GGCC", 2, "m"), ("G[AG].GAAG[CT]", 5, "a"), ("GGA......TCC", 2, "a"), ("GAGG", 1, "a"))
LAYOUTS = {
    # bin_big alone exceeds half of the assembly: its contigs, short ones included, are spread over the two ranks
    "bins": (("bin_big", (90000, 70000, 60000, 40000, 7, 3)), ("bin_s1", (30000, 8000)), ("bin_s2", (25000,)),
             ("bin_s3", (9000, 7000, 3000, 5))),
    # one contig alone exceeds half of the assembly: it is cut into two ContigPieces with 64 bp of text halo
    "mono": (("mono", (200000, 9000)), ("bin_s1", (12000, 8000))),
    # whole bins; bins packed next to each other on a rank share a tile, bin_6 holds contigs of 3-7 bp
    "tiles": (("bin_0", (150000, 7)), ("bin_1", (250000, 3)), ("bin_2", (20000, 5)), ("bin_3", (60000, 5)),
              ("bin_4", (120000, 2600)), ("bin_5", (120000, 7)), ("bin_6", (2600, 7, 3, 5))),
    # one bin of one contig, not cut: the second rank holds no contig at all
    "solo": (("solo", (30000,)),),
}
NO_ROWS = {"bin_s2", "bin_2"}  # bins without pileup rows
VARIANTS = {  # candidates() keyword arguments per mod type
    "a": ({}, {"prune": True}, {"bipartite_letters": "IUPAC"}, {"bipartite_letters": "IUPAC", "prune": True},
          {"ks": [5, 7]}, {"bipartite": False}, {"scratch_bytes": 1, "capacity": 1}),
    "m": ({}, {"prune": True}),
    "21839": ({}, {"bipartite_letters": "IUPAC", "prune": True}),
}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _make(layout):
    from nanomotif_b200 import synth

    rng = np.random.default_rng(31)
    bins = {}
    cols = {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod")}
    for j, (b, lens) in enumerate(LAYOUTS[layout]):
        bins[b] = {}
        planted = tuple(PLANTED[(2 * j + i) % len(PLANTED)] for i in range(3))
        for i, L in enumerate(lens):
            name = f"{b}_c{i}"
            seq = synth.random_sequence(rng, L, 0.4 + 0.03 * j, 2e-5)
            if L > 1000:
                seq[rng.integers(0, L, 10)] = ord("R")  # isolated non-ACGT letters
            bins[b][name] = seq.tobytes().decode()
            if b in NO_ROWS:
                continue
            p = synth.synth_pileup(seq, rng, planted=planted, depth=12, mod_types=MOD_TYPES)
            n = len(p["position"])
            cols["contig"].append(np.full(n, name, dtype=object))
            cols["position"].append(p["position"])
            cols["strand"].append(np.where(p["strand"] == 0, "+", "-").astype(object))
            cols["mod_type"].append(np.array(MOD_TYPES, dtype=object)[p["mod_type"]])
            cols["fraction_mod"].append(p["fraction_mod"])
    return bins, {k: np.concatenate(v) for k, v in cols.items()}


def _sample(rng, canon, n):
    """(motif, mod_pos) pairs: IUPAC 4..8-mers and ACGT bipartite motifs with the canonical base at mod_pos."""
    out = []
    while len(out) < n:
        if rng.random() < 0.7:
            s = "".join(rng.choice(list("ACGTRYSWKMBDHVN"), size=int(rng.integers(4, 9))))
            if s[0] == "N" or s[-1] == "N":
                continue
        else:
            s = "".join(rng.choice(list("ACGT"), size=int(rng.integers(3, 5)))) + "N" * int(rng.integers(4, 9)) + \
                "".join(rng.choice(list("ACGT"), size=int(rng.integers(3, 5))))
        pos = [i for i, ch in enumerate(s) if ch == canon]
        if pos:
            out.append((s, int(rng.choice(pos))))
    return out


class _Report:
    def __init__(self):
        self.fails, self.rows = [], 0

    def check(self, ok, what):
        if not ok:
            self.fails.append(what)

    def frames(self, got, want, what):
        import pandas as pd

        try:
            pd.testing.assert_frame_equal(got, want)
        except AssertionError as exc:
            self.fails.append(f"{what}: {exc}")
        self.rows += len(want)

    def raises(self, exc, fn, what):
        try:
            fn()
        except exc:
            return
        except Exception as other:  # noqa: BLE001
            self.fails.append(f"{what}: {other!r} instead of {exc.__name__}")
        else:
            self.fails.append(f"{what}: no {exc.__name__}")


def _compare(rep, rank, ssw, ref, what, variants, counts_rng=None):
    """ssw (sharded) against ref (BinSweep over all bins on one GPU): designated histograms, frames, counts."""
    import torch

    from nanomotif_b200.sweep import BIP_SIZE, HIST_SIZE

    sw = ssw.local
    for b in ssw.bins:
        if sw is None or b not in sw.slot:
            continue
        s, r = sw.slot[b], ref.slot[b]
        if ssw.designated[b] == rank:
            rep.check(torch.equal(sw.hist[s], ref.hist[r]), f"{what} {b}: finished IUPAC histogram")
            if ref.bip_raw is not None:
                rep.check(torch.equal(sw.bip[s], ref.bip[r]), f"{what} {b}: finished bipartite histogram")
        else:  # another holder of a split bin: its copy is zero, so it yields no rows
            rep.check(int(sw.raw.view(-1, HIST_SIZE)[s].abs().sum()) == 0, f"{what} {b}: non-designated IUPAC copy")
            if sw.bip_raw is not None:
                rep.check(int(sw.bip_raw.view(-1, BIP_SIZE)[s].abs().sum()) == 0, f"{what} {b}: non-designated bip copy")
    for kw in variants:
        want = ref.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, **kw)
        rep.frames(ssw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, **kw), want, f"{what} candidates({kw})")
    if counts_rng is None:
        return
    from nanomotif_b200.sweep import BIP_LETTERS

    canon = CANON[ssw.mod_type]
    for b in ssw.bins:  # the same calls in the same order on every rank: the seed does not depend on the rank
        for s, p in _sample(counts_rng, canon, 50 // len(ssw.bins) + 4):
            rep.check(ssw.counts(b, s, p) == ref.counts(b, s, p), f"{what} counts({b}, {s}, {p})")
        for _ in range(3):
            a, bb = (int(x) for x in counts_rng.choice([3, 4], 2))
            g = int(counts_rng.integers(4, 9))
            halves = list(counts_rng.choice(list(BIP_LETTERS), a + bb))
            o = int(counts_rng.integers(a + bb))
            halves[o] = canon
            left, right = "".join(halves[:a]), "".join(halves[a:])
            mp = o if o < a else o + g
            rep.check(ssw.bipartite_iupac_counts(b, left, g, right, mp) == ref.bipartite_iupac_counts(b, left, g, right, mp),
                      f"{what} bipartite_iupac_counts({b}, {left}, {g}, {right}, {mp})")


def _checks(rank, world, layout, dev):
    import nanomotif_b200 as nmb
    from nanomotif_b200.sharding import ShardedBinSweep, ShardedMultiBinScorer
    from nanomotif_b200.sweep import BinSweep

    rep = _Report()
    bins, pile = _make(layout)
    scorer = ShardedMultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7, rank, world, dev, split_contigs=layout != "solo")
    single = nmb.MultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7, dev)
    rng = np.random.default_rng(77)
    for mt in MOD_TYPES:
        _compare(rep, rank, ShardedBinSweep(scorer, mt), BinSweep(single, mt), f"{layout}/{mt}", VARIANTS[mt], rng)
    if layout == "tiles":  # bins= of one rank only, in an order of their own: the other rank holds none of them
        only = [b for b in bins if scorer.bin_ranks[b] == [0]][::-1]
        rep.check(1 < len(only) < len(bins), f"bins of rank 0: {only}")
        ssw = ShardedBinSweep(scorer, "a", bins=only)
        rep.check((ssw.local is None) == (rank == 1), "rank 1 holds none of the requested bins")
        _compare(rep, rank, ssw, BinSweep(single, "a", bins=only), "tiles/rank-0 bins", ({}, {"prune": True}), rng)
    if layout == "solo":
        rep.check((scorer.local is None) == (rank == 1), "rank 1 holds no contig")
    if layout == "bins":  # argument errors as BinSweep raises them, on every rank
        ssw = ShardedBinSweep(scorer, "a", bipartite=False)
        ref = BinSweep(single, "a", bipartite=False)
        rep.raises(ValueError, lambda: ssw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD), "bipartite request")
        rep.raises(ValueError, lambda: ssw.candidates(min_mod=0), "min_mod < 1")
        rep.raises(KeyError, lambda: ssw.counts("no_such_bin", "GATC", 1), "unknown bin in counts")
        rep.raises(KeyError, lambda: ssw.bipartite_iupac_counts("no_such_bin", "GAA", 6, "RTCG", 2), "unknown bin")
        rep.raises(KeyError, lambda: ShardedBinSweep(scorer, "a", bins=["bin_s1", "no_such_bin"]), "unknown bin in bins=")
        rep.raises(ValueError, lambda: ssw.counts("bin_big", "GRTC", 1), "bad motif in a split bin")
        rep.raises(ValueError, lambda: ref.counts("bin_big", "GRTC", 1), "bad motif, one GPU")
        rep.frames(ssw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite=False, prune=True),
                   ref.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite=False, prune=True), "bipartite=False sweep")
    local_bp = scorer.local.assembly.total_bp if scorer.local is not None else 0
    return rep.fails, rep.rows, sorted(scorer.split_bins), local_bp


def _worker(rank, world, port, backend, q, layout):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        q.put((rank,) + _checks(rank, world, layout, dev))
    except Exception:  # noqa: BLE001 -- reported to the test process
        q.put((rank, [traceback.format_exc()], 0, [], 0))
    finally:
        dist.destroy_process_group()


def _run_ranks(layout, world=2):
    import torch
    import torch.multiprocessing as mp

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    backend = "nccl" if torch.cuda.device_count() >= world else "gloo"
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, q, layout)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        results = sorted(q.get(timeout=900) for _ in range(world))
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    for rank, fails, rows, _, _ in results:
        assert not fails, f"rank {rank}:\n" + "\n".join(fails[:20])
        assert rows > 0
    assert results[0][2] == results[1][2]  # every rank built the same frames
    return results


def test_split_bin_equals_one_gpu():
    results = _run_ranks("bins")
    for _, _, _, split, local_bp in results:
        assert split == ["bin_big"] and local_bp > 0


def test_contig_cut_into_pieces_equals_one_gpu():
    """The halo argument: a row lies under windows at most 15 bp from it, the pieces carry 64 bp of text on both
    sides, so the two pieces' raw counters add up to those of the whole contig."""
    results = _run_ranks("mono")
    for _, _, _, split, _ in results:
        assert split == ["mono"]


def test_whole_bins_sharing_tiles_and_a_subset_of_one_rank():
    results = _run_ranks("tiles")
    for _, _, _, split, local_bp in results:
        assert split == [] and local_bp > 0


def test_rank_without_contigs_takes_part():
    results = _run_ranks("solo")
    assert [r[4] > 0 for r in results] == [True, False]
