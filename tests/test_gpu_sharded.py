"""The product multi-GPU path (sharding.ShardedMultiBinScorer) on CUDA devices, world size 2: bins sharded by
plan_shards, every rank scans only its contigs, ONE all-reduce per batch.  With >= 2 GPUs the ranks use NCCL on their own
devices; on a one-GPU box both ranks share cuda:0 and the collective runs over gloo (CUDA tensors) -- the sharding logic
and the kernels are the same.  Checked against the unsharded scorer and the oracle."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MOD_TYPES = ("a", "m")
MOTIFS = {"a": [("GATC", 1), ("A", 0), ("GCAC......GTT", 2),
              # a frontier round (synth.frontier_worklist(1, "A")[5]) and a run split 61 right of the modified base: K2
              # scores each as one parent chain pair plus a four-base split, next to the pieces' artificial ends too
              ("C...G....A.G.G....TC", 9), ("G...G....A.G.G....TC", 9), ("T...G....A.G.G....TC", 9),
              ("A...G....A.G.G....TC", 9),
              ("A" + "." * 60 + "C", 0), ("A" + "." * 60 + "G", 0), ("A" + "." * 60 + "[CT]", 0)],
          "m": [("CC[AT]GG", 1), ("C", 0)]}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


LAYOUTS = {
    # bin_big alone exceeds half of the assembly -> its contigs are split over the two ranks (all-reduce merges them)
    "bins": (("bin_big", (90000, 70000, 60000, 40000)), ("bin_s1", (30000, 8000)), ("bin_s2", (25000,)), ("bin_s3", (9000, 7000, 3000))),
    # one contig alone exceeds half of the assembly (a monoculture: chromosome + plasmids) -> it is cut into two
    # position ranges, each rank packs its range + 64 bp of text on both sides and joins the rows of its range
    "mono": (("mono", (200000, 9000)), ("bin_s1", (12000, 8000))),
}


def _make(layout="bins", seed=9):
    from nanomotif_b200 import synth

    rng = np.random.default_rng(seed)
    bins = {}
    cols = {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod")}
    for b, lens in LAYOUTS[layout]:
        bins[b] = {}
        for i, L in enumerate(lens):
            name = f"{b}_c{i}"
            seq = synth.random_sequence(rng, L, 0.5, 1e-5)
            bins[b][name] = seq.tobytes().decode()
            p = synth.synth_pileup(seq, rng, depth=15, mod_types=MOD_TYPES)
            n = len(p["position"])
            cols["contig"].append(np.full(n, name, dtype=object))
            cols["position"].append(p["position"])
            cols["strand"].append(np.where(p["strand"] == 0, "+", "-").astype(object))
            cols["mod_type"].append(np.array(MOD_TYPES, dtype=object)[p["mod_type"]])
            cols["fraction_mod"].append(p["fraction_mod"])
    return bins, {k: np.concatenate(v) for k, v in cols.items()}


def _requests(nmb, scorer, bins):
    return [(scorer.context(b, mt), [nmb.Motif(m, p) for m, p in MOTIFS[mt]]) for b in bins for mt in MOD_TYPES]


def _worker(rank, world, port, backend, q, layout="bins"):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        import nanomotif_b200 as nmb
        from nanomotif_b200 import device as D
        from nanomotif_b200.sharding import ShardedMultiBinScorer

        # blocks of 32 motifs, as in a search round over many bins: at this size the automatic choice is one motif per
        # item, where no sibling run forms (the unsharded scorer below keeps it: the general path is the reference)
        D.choose_motifs_per_item = lambda jobs, sm_count: 32

        bins, pile = _make(layout)
        # every rank knows all lengths; sequences only of the contigs it may own -- here simply all of them
        scorer = ShardedMultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7, rank, world, dev)
        first = scorer.submit(_requests(nmb, scorer, bins))  # two batches in flight before the first result is read
        second = scorer.submit(_requests(nmb, scorer, bins))
        got = [c.tolist() for c in first.result()]
        assert [c.tolist() for c in second.result()] == got
        local_bp = scorer.local.assembly.total_bp if scorer.local is not None else 0
        q.put((rank, got, sorted(scorer.split_bins), local_bp))
    finally:
        dist.destroy_process_group()


def _run_ranks(layout, world=2):
    import torch
    import torch.multiprocessing as mp

    backend = "nccl" if torch.cuda.device_count() >= world else "gloo"
    port = _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, q, layout)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return results


def test_sharded_scorer_equals_unsharded_and_oracle():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200 as nmb
    from oracle import restate as O

    results = _run_ranks("bins")
    bins, pile = _make()
    single = nmb.MultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7)
    want = [c.tolist() for c in single.score_batch(_requests(nmb, single, bins))]
    total_bp = sum(len(s) for cs in bins.values() for s in cs.values())
    assert sum(r[3] for r in results) == total_bp  # every contig packed on exactly one rank
    for rank, got, split, local_bp in results:
        assert got == want, f"rank {rank}"
        assert split == ["bin_big"]
        assert 0.35 * total_bp < local_bp < 0.65 * total_bp
    # and the unsharded scorer against the oracle
    at = 0
    for b in bins:
        for mt in MOD_TYPES:
            sel = pile["mod_type"] == mt
            for j, (m, p) in enumerate(MOTIFS[mt]):
                w = O.motif_model_bin(pile["contig"][sel], pile["position"][sel], pile["strand"][sel],
                                      pile["fraction_mod"][sel], bins[b], m, p, fast=True)
                assert tuple(want[at][j]) == tuple(w), (b, mt, m)
            at += 1


def test_one_huge_contig_is_cut_into_position_ranges():
    """SURVEY 8e, cfg 2 on several GPUs: a contig that alone exceeds a rank's share is scored piecewise -- every rank
    packs its position range (+ 64 bp of text on both sides) and joins the pileup rows of its range; the all-reduce
    adds the pieces up.  Same counts as the unsharded scorer (whose parity with the oracle the test above pins)."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200 as nmb

    results = _run_ranks("mono")
    bins, pile = _make("mono")
    single = nmb.MultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7)
    want = [c.tolist() for c in single.score_batch(_requests(nmb, single, bins))]
    total_bp = sum(len(s) for cs in bins.values() for s in cs.values())
    assert sum(r[3] for r in results) == total_bp + 2 * 64  # the two pieces overlap by their halos
    for rank, got, split, local_bp in results:
        assert got == want, f"rank {rank}"
        assert split == ["mono"]
        assert 0.4 * total_bp < local_bp < 0.6 * total_bp


def test_contigs_of_other_ranks_by_length_only():
    """Every rank must derive the same plan, so it needs all LENGTHS -- not all sequences."""
    from nanomotif_b200 import sharding

    bins, _ = _make()
    lengths = [len(s) for cs in bins.values() for s in cs.values()]
    groups = [i for i, cs in enumerate(bins.values()) for _ in cs]
    owner = sharding.plan_shards(lengths, 2, groups)
    assert set(owner.tolist()) == {0, 1}
    assert sharding._contig_length(1234) == 1234 and sharding._contig_length("ACGT") == 4
