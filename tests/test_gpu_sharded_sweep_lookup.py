"""The sharded sweep lookup (sharding.ShardedBinSweep.count_matrix) on CUDA devices, world size 2: on every rank the
count matrix equals that of the unsharded BinSweep over all bins, for layouts with a split bin, a contig cut into two
pieces and a rank without contigs; an uncovered motif raises on both ranks and leaves neither waiting.  Run like
tests/test_gpu_sharded_sweep.py: NCCL with >= 2 GPUs, else both ranks on cuda:0 over gloo.  Each rank reports what
differs instead of asserting, so a failed check on one rank cannot leave the other in a collective."""
import os
import socket
import traceback

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MOD_TYPES = ("a", "m", "21839")
CANON = {"a": "A", "m": "C", "21839": "C"}
PLANTED = (("GATC", 1, "a"), ("CC[AT]GG", 1, "m"), ("GAATTC", 2, "a"), ("GCAC......GTT", 2, "a"), ("CCGG", 0, "21839"),
           ("TCGA", 3, "a"), ("GGCC", 2, "m"), ("G[AG].GAAG[CT]", 5, "a"), ("GGA......TCC", 2, "a"), ("GAGG", 1, "a"))
LAYOUTS = {
    # bin_big alone exceeds half of the assembly: its contigs, short ones included, are spread over the two ranks
    "bins": (("bin_big", (90000, 70000, 60000, 40000, 7, 3)), ("bin_s1", (30000, 8000)), ("bin_s2", (25000,)),
             ("bin_s3", (9000, 7000, 3000, 5))),
    # one contig alone exceeds half of the assembly: it is cut into two ContigPieces with 64 bp of text halo
    "mono": (("mono", (200000, 9000)), ("bin_s1", (12000, 8000))),
    # one bin of one contig, not cut: the second rank holds no contig at all
    "solo": (("solo", (30000,)),),
}
NO_ROWS = {"bin_s2"}


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
    """(motifs, mod_positions): IUPAC 4..8-mers (flanking and inner N included) and bipartite motifs with halves over
    the 14 letters but N, the canonical base at the modified position."""
    from nanomotif_b200.sweep import BIP_LETTERS, IUPAC_ORDER

    motifs, mps = [], []
    while len(motifs) < n:
        if rng.random() < 0.6:
            s = list(rng.choice(list(IUPAC_ORDER), size=int(rng.integers(4, 9))))
            o = int(rng.integers(len(s)))
            s[o] = canon
            motifs.append("".join(s))
            mps.append(o)
        else:
            a, b = (int(x) for x in rng.choice([3, 4], 2))
            g = int(rng.integers(4, 9))
            halves = list(rng.choice(list(BIP_LETTERS), a + b))
            o = int(rng.integers(a + b))
            halves[o] = canon
            motifs.append("".join(halves[:a]) + "N" * g + "".join(halves[a:]))
            mps.append(o if o < a else o + g)
    return motifs, mps


def _checks(rank, world, layout, dev):
    import nanomotif_b200 as nmb
    from nanomotif_b200.sharding import ShardedBinSweep, ShardedMultiBinScorer
    from nanomotif_b200.sweep import BinSweep

    fails, checked = [], 0

    def same(got, want, what):
        nonlocal checked
        for g, w, cls in zip(got, want, ("n_mod", "n_nomod")):
            if g.dtype != np.int64 or g.shape != w.shape or not np.array_equal(g, w):
                fails.append(f"{what} {cls}: {g.shape} {w.shape}, {int((g != w).sum()) if g.shape == w.shape else '-'} "
                             "entries differ")
        checked += got[0].size

    def raises(exc, fn, what):
        try:
            fn()
        except exc:
            return
        except Exception as other:  # noqa: BLE001
            fails.append(f"{what}: {other!r} instead of {exc.__name__}")
        else:
            fails.append(f"{what}: no {exc.__name__}")

    bins, pile = _make(layout)
    scorer = ShardedMultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7, rank, world, dev, split_contigs=layout != "solo")
    single = nmb.MultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7, dev)
    rng = np.random.default_rng(78)  # the same calls in the same order on every rank
    for mt in MOD_TYPES:
        ssw, ref = ShardedBinSweep(scorer, mt), BinSweep(single, mt)
        motifs, mps = _sample(rng, CANON[mt], 400)
        got = ssw.count_matrix(motifs, mps)
        same(got, ref.count_matrix(motifs, mps, bins=ssw.bins), f"{layout}/{mt}")
        if got[0].sum() <= 0:
            fails.append(f"{layout}/{mt}: no counts")
        order = ssw.bins[::-1]
        same(ssw.count_matrix(motifs[:50], mps[:50], bins=order), ref.count_matrix(motifs[:50], mps[:50], bins=order),
             f"{layout}/{mt} bins reversed")
    ssw = ShardedBinSweep(scorer, "a", bipartite=False)
    ref = BinSweep(single, "a", bipartite=False)
    raises(ValueError, lambda: ssw.count_matrix(["GATC", "GANNNNNNNRTCG"], [1, 1]), "uncovered motif")
    raises(ValueError, lambda: ssw.count_matrix(["GAANNNNNNRTCG"], [2]), "bipartite motif, bipartite=False")
    raises(KeyError, lambda: ssw.count_matrix(["GATC"], [1], bins=["no_such_bin"]), "unknown bin")
    # after the errors every rank still meets the other in the next collective
    same(ssw.count_matrix(["GATC", "NNNANNNN"], [1, 3]), ref.count_matrix(["GATC", "NNNANNNN"], [1, 3], bins=ssw.bins),
         f"{layout} after the errors")
    empty = ssw.count_matrix([], [])
    if empty[0].shape != (len(ssw.bins), 0):
        fails.append(f"empty motif list: {empty[0].shape}")
    return fails, checked, sorted(scorer.split_bins), scorer.local is None


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
        q.put((rank, [traceback.format_exc()], 0, [], False))
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
    for rank, fails, checked, _, _ in results:
        assert not fails, f"rank {rank}:\n" + "\n".join(fails[:20])
        assert checked > 0
    return results


def test_split_bin():
    for _, _, _, split, _ in _run_ranks("bins"):
        assert split == ["bin_big"]


def test_contig_cut_into_pieces():
    for _, _, _, split, _ in _run_ranks("mono"):
        assert split == ["mono"]


def test_rank_without_contigs():
    assert [r[4] for r in _run_ranks("solo")] == [False, True]
