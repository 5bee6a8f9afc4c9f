"""The sharded methylation-pattern table (sharding.ShardedPatternTable, sharding.methylation_pattern) on CUDA devices,
world size 2: every frame equals pattern.methylation_pattern on one GPU exactly, and table(on_device=True) equals
pattern_table over the whole assembly bit for bit, for a pandas table, a bedMethyl text file and a bgzip + tabix file.
With >= 2 GPUs the ranks use NCCL on their own devices; on a one-GPU box both ranks share cuda:0 and the collectives
run over gloo (CUDA tensors).  Each rank compares against its own one-GPU result and reports what differs, so that a
failed check on one rank cannot leave the other waiting in a collective."""
import os
import socket
import traceback

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MOD_TYPES = ("a", "m", "21839")
PLANTED = (("GATC", 1, "a"), ("CC[AT]GG", 1, "m"), ("GAATTC", 2, "a"), ("GCAC......GTT", 2, "a"), ("CCGG", 0, "21839"))
LAYOUTS = {
    # many contigs of mixed lengths, contigs of 3-7 bp; c3 and c9 have no pileup rows
    "mixed": ((90000, 7, 30000, 40000, 5, 25000, 12000, 3, 60000, 800, 4, 2600), {"c3", "c9"}),
    # one contig holds most of the assembly; the other rank's contigs have no pileup rows at all
    "mono": ((200000, 9000, 7), {"c1", "c2"}),
    # a single contig: rank 1 holds nothing
    "solo": ((30000,), set()),
}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _motifs():
    """Three mod types, IUPAC and bipartite N-run motifs, one motif that occurs nowhere, and more than 64 motifs."""
    fixed = ["GATC_a_1", "GATC_m_3", "CCWGG_m_1", "GRNGAAGY_a_5", "A_a_0", "CCGG_21839_0", "GCACNNNNNNGTT_a_2",
             "C" + "N" * 33 + "AT_a_34", "ACGTTGCATGCAAGTCCTAGGACT_a_0", "T_m_0", "GCGC_21839_1", "CCNGG_21839_0"]
    rng = np.random.default_rng(5)
    out = list(fixed)
    while len(out) < 80:
        mt = MOD_TYPES[len(out) % 3]
        canon = "A" if mt == "a" else "C"
        if rng.random() < 0.6:
            s = "".join(rng.choice(list("ACGTRYSWKMBDHVN"), size=int(rng.integers(3, 9))))
        else:
            s = "".join(rng.choice(list("ACGT"), size=3)) + "N" * int(rng.integers(4, 9)) + "".join(rng.choice(list("ACGT"), size=3))
        pos = [i for i, ch in enumerate(s) if ch == canon]
        if not pos or s[0] == "N" or s[-1] == "N":
            continue
        spec = f"{s}_{mt}_{int(rng.choice(pos))}"
        if spec not in out:
            out.append(spec)
    return out


def _make(layout):
    """(contigs, pandas pileup table): rows sorted by contig and position, then rows of a contig absent from the
    assembly (grouped at the end, as a sorted bedMethyl file has them)."""
    import pandas as pd

    from nanomotif_b200 import synth

    lengths, no_rows = LAYOUTS[layout]
    rng = np.random.default_rng(41)
    contigs, parts = {}, []
    for i, L in enumerate(lengths + (5000,)):
        name = f"c{i}" if i < len(lengths) else "ghost"
        seq = synth.random_sequence(rng, L, 0.45, 2e-5)
        if L > 1000:
            seq[rng.integers(0, L, 10)] = ord("R")  # isolated non-ACGT letters
        if name != "ghost":
            contigs[name] = seq.tobytes().decode()
        if name in no_rows:
            continue
        p = synth.synth_pileup(seq, rng, planted=PLANTED, depth=10, mod_types=MOD_TYPES, with_counts=True)
        n = len(p["position"])
        parts.append(pd.DataFrame({"contig": np.full(n, name, dtype=object), "position": p["position"],
                                   "strand": np.where(p["strand"] == 0, "+", "-").astype(object),
                                   "mod_type": np.array(MOD_TYPES, dtype=object)[p["mod_type"]],
                                   "fraction_mod": p["fraction_mod"], "Nvalid_cov": p["Nvalid_cov"], "n_mod": p["n_mod"],
                                   "n_diff": p["n_diff"]}))
    return contigs, pd.concat(parts, ignore_index=True)


def _write_files(layout, tmp):
    """The same pileup as bedMethyl text and as bgzip + tabix."""
    from nanomotif_b200 import bgzf

    _, t = _make(layout)
    pos = t["position"].to_numpy()
    cov = t["Nvalid_cov"].to_numpy()
    lines = [f"{c}\t{p}\t{p + 1}\t{m}\t{v}\t{s}\t{p}\t{p + 1}\t255,0,0\t{v}\t{f * 100:.2f}\t{nm}\t0\t0\t0\t0\t{nd}\t0"
             for c, p, m, v, s, f, nm, nd in zip(t["contig"], pos.tolist(), t["mod_type"], cov.tolist(), t["strand"],
                                                 t["fraction_mod"].tolist(), t["n_mod"].tolist(), t["n_diff"].tolist())]
    text = os.path.join(tmp, f"{layout}.bed")
    with open(text, "w") as f:
        f.write("\n".join(lines) + "\n")
    return text, bgzf.bgzf_pileup(text, os.path.join(tmp, f"{layout}.bed.gz"))


class _Report:
    def __init__(self):
        self.fails, self.rows = [], 0

    def check(self, ok, what):
        if not ok:
            self.fails.append(what)

    def frames(self, got, want, what):
        import pandas as pd

        try:
            pd.testing.assert_frame_equal(got, want, check_exact=True)
        except AssertionError as exc:
            self.fails.append(f"{what}: {exc}")
        self.rows += len(want)

    def raises(self, fn, message, what):
        try:
            fn()
        except ValueError as exc:
            self.check(str(exc) == message, f"{what}: {exc}")
        except Exception as other:  # noqa: BLE001
            self.fails.append(f"{what}: {other!r} instead of ValueError")
        else:
            self.fails.append(f"{what}: no ValueError")


def _same(a, b):
    """Bit-equal tensors, NaN where the other has NaN."""
    import torch

    if a is None or b is None:
        return a is None and b is None
    if a.dtype.is_floating_point:
        nan = a.isnan()
        return torch.equal(nan, b.isnan()) and torch.equal(a[~nan], b[~nan])
    return torch.equal(a, b)


def _checks(rank, world, layout, dev, text, gz, tmp):
    import pandas as pd
    import torch

    from nanomotif_b200 import pattern, sharding, tables
    from nanomotif_b200.device import DeviceAssembly
    from nanomotif_b200.motif import Motif
    from nanomotif_b200.pattern import MethylationOutput, PatternIndex, pattern_table

    rep = _Report()
    contigs, table = _make(layout)
    names = list(contigs)
    motifs = _motifs()
    specs = [pattern.parse_motif_spec(m) for m in motifs]
    mod_types = sorted(MOD_TYPES)
    inputs = {"table": table, "text": text, "bgzip+tbi": gz}
    for kind, pileup in inputs.items():
        for out in (MethylationOutput.Median, MethylationOutput.WeightedMean):
            want = pattern.methylation_pattern(pileup, contigs, motifs, output_type=out, device=dev)
            got = sharding.methylation_pattern(pileup, contigs, motifs, rank, world, output_type=out, device=dev)
            rep.frames(got, want, f"{layout}/{kind}/{out.name}")

    # table(on_device=True) against pattern_table over the whole assembly; K9 on both
    asm = DeviceAssembly.from_sequences(contigs, dev)
    rows, _ = pattern.pileup_rows(table, names, mod_types, True, dev)
    tab = sharding.ShardedPatternTable(gz, contigs, mod_types, rank, world, dev)
    rep.check((tab.assembly is None) == (layout == "solo" and rank == 1), f"{layout}: rank {rank} holds contigs")
    contig_bin = {n: f"bin{i % 3}" for i, n in enumerate(names) if i % 5 != 4}
    for median in (True, False):
        st_s, val_s = tab.table(motifs, median, on_device=True)
        rep.check(st_s.is_cuda and st_s.shape == (len(motifs), len(names), 3), f"{layout}: sharded stats shape")
        st_h, val_h = tab.table(motifs, median)
        rep.check(np.array_equal(st_h, st_s.cpu().numpy()), f"{layout}: host stats")
        rep.check((val_h is None) if not median else np.array_equal(val_h, val_s.cpu().numpy(), equal_nan=True),
                  f"{layout}: host value")
        st_1 = torch.zeros_like(st_s)
        val_1 = torch.full_like(val_s, float("nan")) if median else None
        for ti, mt in enumerate(mod_types):
            sel = [i for i, s in enumerate(specs) if s[1] == mt]
            index = PatternIndex(asm, rows, ti)
            st, val = pattern_table(index, [Motif(specs[i][0], specs[i][2]).from_iupac() for i in sel], median,
                                    on_device=True)
            st_1[sel] = st
            if median:
                val_1[sel] = val
        rep.check(_same(st_s, st_1), f"{layout} median={median}: table stats")
        rep.check(_same(val_s, val_1), f"{layout} median={median}: table value")
        for thr in (24.0, 0.0):
            got_c, got_m, got_f = tables.bin_feature_matrix_device(st_s, val_s, names, motifs, contig_bin, thr)
            want_c, want_m, want_f = tables.bin_feature_matrix_device(st_1, val_1, names, motifs, contig_bin, thr)
            rep.check(got_c.tolist() == want_c.tolist() and got_f.tolist() == want_f.tolist() and _same(got_m, want_m),
                      f"{layout} median={median} thr={thr}: K9 matrix")

    # output: written by rank 0 only, the bytes one GPU writes
    single = os.path.join(tmp, f"{layout}_single_{rank}.tsv")
    pattern.methylation_pattern(table, contigs, motifs, output=single, device=dev)
    calls = []
    to_csv = pd.DataFrame.to_csv
    pd.DataFrame.to_csv = lambda self, *a, **k: (calls.append(a), to_csv(self, *a, **k))[1]
    try:
        sharding.methylation_pattern(table, contigs, motifs, rank, world, output=os.path.join(tmp, f"{layout}_sharded.tsv"),
                                     device=dev)
    finally:
        pd.DataFrame.to_csv = to_csv
    rep.check(len(calls) == (1 if rank == 0 else 0), f"{layout}: rank {rank} wrote {len(calls)} times")
    if rank == 0:
        with open(single, "rb") as a, open(os.path.join(tmp, f"{layout}_sharded.tsv"), "rb") as b:
            rep.check(a.read() == b.read(), f"{layout}: output bytes")

    if layout == "mixed":  # errors on every rank, no rank left in a collective
        for kind, pileup in inputs.items():
            rep.raises(lambda: pattern.methylation_pattern(pileup, contigs, motifs, allow_assembly_pileup_mismatch=False,
                                                           device=dev), pattern.MISMATCH_ERROR, f"{kind}: one GPU mismatch")
            rep.raises(lambda: sharding.methylation_pattern(pileup, contigs, motifs, rank, world, device=dev,
                                                            allow_assembly_pileup_mismatch=False),
                       pattern.MISMATCH_ERROR, f"{kind}: sharded mismatch")
        clean = table[table["contig"] != "ghost"]
        rep.frames(sharding.methylation_pattern(clean, contigs, motifs, rank, world, device=dev,
                                                allow_assembly_pileup_mismatch=False),
                   pattern.methylation_pattern(clean, contigs, motifs, device=dev), "no mismatch, strict")
        mine = motifs if rank == 0 else motifs[:-1]
        rep.raises(lambda: sharding.methylation_pattern(table, contigs, mine, rank, world, device=dev),
                   "the ranks were given different motif lists", "motif lists differ")
        rep.raises(lambda: tab.table(motifs[::-1] if rank == 1 else motifs), "the ranks were given different motif lists",
                   "table(): motif lists differ")
    return rep.fails, rep.rows, len(tab.columns)


def _worker(rank, world, port, backend, q, layout, text, gz, tmp):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        q.put((rank,) + _checks(rank, world, layout, dev, text, gz, tmp))
    except Exception:  # noqa: BLE001 -- reported to the test process
        q.put((rank, [traceback.format_exc()], 0, 0))
    finally:
        dist.destroy_process_group()


def _run_ranks(layout, tmp_path, world=2):
    import torch
    import torch.multiprocessing as mp

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    text, gz = _write_files(layout, str(tmp_path))
    backend = "nccl" if torch.cuda.device_count() >= world else "gloo"
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, q, layout, text, gz, str(tmp_path)))
             for r in range(world)]
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
    for rank, fails, rows, _ in results:
        assert not fails, f"rank {rank}:\n" + "\n".join(fails[:20])
        assert rows > 0
    assert results[0][2] == results[1][2]  # every rank built the same frames
    return [r[3] for r in results]


def test_many_contigs_of_mixed_lengths_equal_one_gpu(tmp_path):
    held = _run_ranks("mixed", tmp_path)
    assert min(held) > 0 and sum(held) == len(LAYOUTS["mixed"][0])


def test_one_large_contig_and_a_rank_without_pileup_rows(tmp_path):
    assert _run_ranks("mono", tmp_path) == [1, 2]


def test_rank_without_contigs_takes_part(tmp_path):
    assert _run_ranks("solo", tmp_path) == [1, 0]


def test_bgzip_fetch_without_rows_has_count_columns(tmp_path):
    """A rank whose contigs have no rows in an indexed pileup gets empty n_mod / n_diff columns, not None."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from nanomotif_b200 import dataload

    _, gz = _write_files("mono", str(tmp_path))
    for want in (["absent"], ["c1", "c2"]):
        rows = dataload.load_contigs_pileup_bgzip(gz, want, with_counts=True)
        assert len(rows) == 0
        assert rows.n_mod is not None and rows.n_mod.dtype == torch.int64 and rows.n_mod.numel() == 0
        assert rows.n_diff is not None and rows.n_diff.dtype == torch.int64 and rows.n_diff.numel() == 0
    assert dataload.load_contigs_pileup_bgzip(gz, ["absent"]).n_mod is None
