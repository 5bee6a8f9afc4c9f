"""Contig-sharded scoring across the GPUs of one box (SURVEY.md 8e).

The reference parallelises over bins with a process pool and no communication
(nanomotif/find_motifs_bin.py:330-372).  Here one process drives one GPU (torchrun); whole contigs are
assigned to ranks by greedy bin-packing on base pairs, every rank scores the replicated motif list
against its own contigs, and the per-motif bin-level counts are summed with ONE all-reduce
(int64, sum) per scoring step -- NCCL over NVLink on GPUs, gloo in the CPU tests.  Per-contig outputs
(the contig x motif table) need no collective: rows are owned by the rank that owns the contig.

A single contig that alone exceeds 1.25 x 1/world_size of the assembly (SURVEY 8d cfg 2: one 4.6 Mbp contig) is cut
into position ranges: the rank of range [a, b) packs the text [a - 64, b + 64) and ingests the pileup rows with
a <= position < b, shifted into the coordinates of that text (`split_ranges`, `ContigPiece`, `remap_split_rows`).
A motif spans at most 62 positions, so an occurrence whose modified base lies in [a, b) lies inside the packed text
exactly when it lies inside the contig, and every pileup row is joined on exactly one rank: the counts of the pieces
add up to the counts of the contig, and the same all-reduce merges them.
"""
from __future__ import annotations

import heapq
from typing import Mapping, Sequence

import numpy as np

from .pattern import MethylationOutput


def plan_shards(lengths: Sequence[int], world_size: int, groups: Sequence[int] | None = None) -> np.ndarray:
    """Rank of every contig.  Longest-first greedy packing balances total bp per rank.  With `groups`
    (bin id per contig) a bin's contigs stay together unless the bin alone exceeds 1.25 x 1/world_size of
    the total, in which case its contigs are spread individually (then the all-reduce merges the bin).  The
    margin keeps bins whole when there are about as many equal-sized bins as ranks."""
    lengths = np.asarray(lengths, dtype=np.int64)
    n = len(lengths)
    owner = np.zeros(n, dtype=np.int32)
    if world_size <= 1 or n == 0:
        return owner
    if groups is None:
        units = [(int(lengths[i]), [i]) for i in range(n)]
    else:
        groups = np.asarray(groups)
        limit = 1.25 * lengths.sum() / world_size
        units = []
        for g in np.unique(groups):
            idx = np.flatnonzero(groups == g).tolist()
            total = int(lengths[idx].sum())
            if total > limit:
                units += [(int(lengths[i]), [i]) for i in idx]
            else:
                units.append((total, idx))
    heap = [(0, r) for r in range(world_size)]
    heapq.heapify(heap)
    for size, idx in sorted(units, key=lambda u: (-u[0], u[1][0])):
        load, r = heapq.heappop(heap)
        owner[idx] = r
        heapq.heappush(heap, (load + size, r))
    return owner


def local_contigs(contigs: Mapping[str, object], owner: np.ndarray, rank: int) -> dict:
    """The sub-dict of `contigs` (insertion order kept) owned by `rank`."""
    return {name: seq for i, (name, seq) in enumerate(contigs.items()) if owner[i] == rank}


HALO_BP = 64  # text kept on both sides of a piece's position range: > the longest motif (62 positions) - 1


class ContigPiece:
    """Position range [a, b) of a contig of `length` bp that one rank scores: the rank packs `text` = the contig's
    letters [lo, hi) = [max(0, a - HALO_BP), min(length, b + HALO_BP)) and keeps pileup rows with a <= position < b
    at position - lo.  `seq` is the whole contig (str / DNAsequence-like) or its length (a rank that does not own the
    piece needs nothing more)."""

    def __init__(self, name: str, a: int, b: int, length: int, seq=None):
        self.name, self.a, self.b, self.length, self.seq = name, int(a), int(b), int(length), seq
        self.lo, self.hi = max(0, self.a - HALO_BP), min(self.length, self.b + HALO_BP)

    @property
    def shift(self) -> int:
        return self.lo

    @property
    def text(self) -> str:
        if self.seq is None or isinstance(self.seq, (int, np.integer)):
            raise ValueError(f"contig {self.name}: this rank owns positions [{self.a}, {self.b}) of a contig that was "
                             "given by length only")
        s = self.seq if isinstance(self.seq, str) else self.seq.sequence
        return s[self.lo:self.hi]

    def __len__(self) -> int:  # what the rank packs (plan bookkeeping)
        return self.hi - self.lo

    def __repr__(self) -> str:
        return f"ContigPiece({self.name!r}, {self.a}, {self.b}, length={self.length})"


def split_ranges(length: int, n_pieces: int) -> list:
    """[a, b) ranges that cut a contig into n_pieces of (almost) equal length, boundaries on multiples of 512 bp (one
    lane chunk of the packed layout; any boundary would be correct)."""
    n_pieces = max(1, min(int(n_pieces), max(1, length // 1024)))
    cuts = [0] + [int(round(length * k / n_pieces / 512)) * 512 for k in range(1, n_pieces)] + [int(length)]
    return [(a, b) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]


def remap_split_rows(contig_id, position, pieces):
    """Rows of split contigs -> rows of the rank's pieces.  contig_id / position: torch tensors (any device) as the
    name lookup wrote them, where every row of a split contig carries the id its NAME resolved to; pieces: [(that id,
    the piece's own contig id, a, b, shift)].  Rows with a <= position < b move to the piece (position - shift); rows
    of a split contig that fall in no local piece get contig id -1 (another rank joins them).  Returns new tensors."""
    import torch

    cid, pos = contig_id.clone(), position.clone()
    for lookup in sorted({int(p[0]) for p in pieces}):
        cid[contig_id == lookup] = -1
    for lookup, own, a, b, shift in pieces:
        m = (contig_id == int(lookup)) & (position >= int(a)) & (position < int(b))
        cid = torch.where(m, torch.full_like(cid, int(own)), cid)
        pos = torch.where(m, position - int(shift), pos)
    return cid, pos


def allreduce_counts(counts, group=None):
    """Sum per-motif count tensors over the ranks in place (int64).  `counts` is a torch tensor on the
    rank's device (CUDA -> NCCL) or on the CPU (gloo).  No-op without an initialised process group."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    return counts


def gather_rows(rows, group=None):
    """Concatenate per-contig result rows of all ranks on every rank (all_gather_object; rows are small
    host objects such as the contig x motif table slices)."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return list(rows)
    out = [None] * dist.get_world_size(group)
    dist.all_gather_object(out, list(rows), group=group)
    return [r for part in out for r in part]


def _contig_length(seq) -> int:
    """Length of a contig given as str, DNAsequence-like (.sequence) or -- for contigs another rank will own --
    as a plain int (every rank must know all lengths to derive the same shard plan, not all sequences)."""
    if isinstance(seq, (int, np.integer)):
        return int(seq)
    return len(seq if isinstance(seq, str) else seq.sequence)


class ShardedContext:
    """One (bin, mod_type) of a ShardedMultiBinScorer; `local` is the rank's BinContext or None."""

    def __init__(self, owner, bin_name, mod_type, local):
        self.owner, self.bin_name, self.mod_type, self.local = owner, bin_name, mod_type, local

    def score(self, motifs) -> np.ndarray:
        return self.owner.score_batch([(self, motifs)])[0]


class PendingScores:
    """Counts of one submitted batch: the scan is enqueued, the all-reduce runs asynchronously."""

    def __init__(self, requests, tensor, work):
        self.requests, self.tensor, self.work = requests, tensor, work

    def result(self) -> list:
        from .api import split_counts

        if self.work is not None:
            self.work.wait()  # orders the current stream after the collective
        return split_counts(self.tensor.cpu().numpy(), self.requests)


class ShardedMultiBinScorer:
    """The multi-GPU form of api.MultiBinScorer -- what replaces the reference's process pool over bins
    (nanomotif/find_motifs_bin.py:330-372) on a box with several GPUs.

    `plan_shards` keeps a bin's contigs on one rank unless the bin alone exceeds 1/world_size of the assembly; every
    rank packs only its own contigs and ingests only the pileup rows of those contigs.  The (replicated) search
    driver calls `score_batch` with the SAME requests on every rank: each rank scans the requests whose bin has local
    contigs in ONE launch and the stacked [total motifs, 4] count tensor is summed over the ranks with ONE all-reduce
    (NCCL over NVLink; SURVEY 8e) -- that merges split bins and replicates the whole-bin results in the same step.
    `submit` returns before the collective has run, so the driver can enqueue the next batch while this one's counts
    are in flight.

    Give every rank the pileup rows of ITS bins: the partitioned form {(bin, mod_type): frame} (frames of bins
    without local contigs are skipped before any copy) or a table that already holds only the rank's rows.  Rows of
    other ranks' contigs in a shared table are ignored, but they are still copied to the device."""

    def __init__(self, pileup, bins: dict, mod_types, low_meth_threshold: float, high_meth_threshold: float,
                 rank: int, world_size: int, device=None, group=None, split_contigs: bool = True):
        import torch

        from .api import MultiBinScorer

        self.rank, self.world_size, self.group = int(rank), int(world_size), group
        self.owner, per_rank, self.split_bins, self.bin_ranks = self.plan(bins, world_size, split_contigs)
        mine, self.pieces = {}, []  # {bin: {local contig name: text}}, [(local name, name the rows carry, a, b, shift)]
        for bin_name, local in per_rank[self.rank].items():
            mine[bin_name] = {}
            for name, seq in local.items():
                if isinstance(seq, ContigPiece):
                    mine[bin_name][name] = seq.text
                    self.pieces.append((name, seq.name, seq.a, seq.b, seq.shift))
                elif isinstance(seq, (int, np.integer)):
                    raise ValueError(f"bin {bin_name}: this rank owns a contig that was given by length only")
                else:
                    mine[bin_name][name] = seq
        self.mod_types = list(mod_types)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        tables = pileup
        if isinstance(pileup, dict) and "position" not in pileup:  # partitioned {(bin, mod_type): frame}
            tables = {k: v for k, v in pileup.items() if not (isinstance(k, tuple) and k[0] in bins and k[0] not in mine)}
        self.local = MultiBinScorer(tables, mine, self.mod_types, low_meth_threshold, high_meth_threshold,
                                    self.device, pieces=self.pieces) if mine else None
        self._local_bins = set(mine)

    @classmethod
    def from_local(cls, local, bins: dict, mod_types, rank: int, world_size: int, device=None, group=None,
                   split_contigs: bool = True) -> "ShardedMultiBinScorer":
        """The sharded scorer over a rank's MultiBinScorer built elsewhere -- e.g. MultiBinScorer.from_device over bins
        generated or parsed on the device, when the host cannot hold the tables.  `bins` = {bin: {contig: sequence or
        length}} of ALL ranks, the same on every rank; `local` must hold exactly the bins plan(bins, world_size) gives
        this rank, with as many contigs (or pieces) each, or be None when the plan gives it none."""
        import torch

        self = cls.__new__(cls)
        self.rank, self.world_size, self.group = int(rank), int(world_size), group
        self.owner, per_rank, self.split_bins, self.bin_ranks = self.plan(bins, world_size, split_contigs)
        mine = per_rank[self.rank]
        held = {} if local is None else {b: hi - lo for b, (lo, hi) in local._ranges.items()}
        if held != {b: len(cs) for b, cs in mine.items()}:
            raise ValueError(f"rank {self.rank}: the local scorer's bins and contig counts are not those the shard plan "
                             "gives this rank")
        if local is not None and [str(m) for m in local.mod_types] != [str(m) for m in mod_types]:
            raise ValueError("the local scorer's mod types differ from mod_types")
        self.pieces = [(name, seq.name, seq.a, seq.b, seq.shift) for cs in mine.values() for name, seq in cs.items()
                       if isinstance(seq, ContigPiece)]
        self.mod_types = list(mod_types)
        if device is None:
            device = local.assembly.device if local is not None else torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        self.local, self._local_bins = local, set(mine)
        return self

    @staticmethod
    def plan(bins: dict, world_size: int, split_contigs: bool = True):
        """The shard plan every rank derives for itself (pure host logic, no device): (owner rank of every contig in
        `bins` order, -1 for a contig cut into pieces; [{bin: {contig: sequence or ContigPiece}} per rank]; set of bins
        that ended up on several ranks; {bin: ranks holding part of it}).  Contigs may be given by length (int)
        instead of sequence.  A contig longer than 1.25 / world_size of the assembly is cut into about
        length / (assembly / world_size) position ranges (module docstring); ranges that land on the same rank next to
        each other are merged again.  The first piece of a contig on a rank keeps the contig's name (the name the
        pileup rows carry), further pieces are named name + chr(31) + str(a)."""
        world = max(1, int(world_size))
        names, lengths, seqs, groups = [], [], [], []
        for b, cs in enumerate(bins.values()):
            for name, seq in cs.items():
                names.append(name)
                seqs.append(seq)
                lengths.append(_contig_length(seq))
                groups.append(b)
        total = int(sum(lengths))
        limit = 1.25 * total / world
        unit_len, unit_group, unit_src = [], [], []
        for i, n in enumerate(lengths):
            ranges = [(0, n)]
            if split_contigs and world > 1 and n > limit:
                ranges = split_ranges(n, -(-n * world // max(1, total)))
            for a, b in ranges:
                unit_len.append(b - a)
                unit_group.append(groups[i])
                unit_src.append((i, a, b))
        unit_owner = plan_shards(unit_len, world, unit_group)
        by_contig = [[] for _ in names]
        for (i, a, b), r in zip(unit_src, unit_owner.tolist()):
            if by_contig[i] and by_contig[i][-1][0] == r and by_contig[i][-1][2] == a:
                by_contig[i][-1] = (r, by_contig[i][-1][1], b)  # next to each other on the same rank: one range
            else:
                by_contig[i].append((r, a, b))
        owner = np.full(len(names), -1, dtype=np.int32)
        per_rank = [dict() for _ in range(world)]
        bin_names = list(bins.keys())
        bin_ranks = {b: set() for b in bin_names}
        for i, parts in enumerate(by_contig):
            bin_name = bin_names[groups[i]]
            if len(parts) == 1 and (parts[0][1], parts[0][2]) == (0, lengths[i]):
                owner[i] = parts[0][0]
            for r, a, b in parts:
                bin_ranks[bin_name].add(r)
                local = per_rank[r].setdefault(bin_name, {})
                if owner[i] >= 0:
                    local[names[i]] = seqs[i]
                else:
                    local[names[i] if names[i] not in local else f"{names[i]}\x1f{a}"] = ContigPiece(
                        names[i], a, b, lengths[i], seqs[i])
        bin_ranks = {b: sorted(r) for b, r in bin_ranks.items()}
        split_bins = {b for b, r in bin_ranks.items() if len(r) > 1}
        return owner, per_rank, split_bins, bin_ranks

    def context(self, bin_name, mod_type) -> ShardedContext:
        if bin_name not in self.bin_ranks:
            raise KeyError(bin_name)
        local = self.local.context(bin_name, mod_type) if bin_name in self._local_bins else None
        return ShardedContext(self, bin_name, mod_type, local)

    def submit(self, requests) -> PendingScores:
        import torch
        import torch.distributed as dist

        requests = [(ctx, list(motifs)) for ctx, motifs in requests]
        local_requests = [(ctx.local, ms) for ctx, ms in requests]
        total = sum(len(ms) for _, ms in requests)
        if self.local is not None:
            t = self.local.score_batch_device(local_requests)
        else:  # a rank without contigs still takes part in the collective
            with torch.cuda.device(self.device):
                t = torch.zeros((total, 4), dtype=torch.int64, device=self.device)
        work = None
        if total and self.world_size > 1 and dist.is_available() and dist.is_initialized():
            work = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        return PendingScores(requests, t, work)

    def score_batch(self, requests) -> list:
        return self.submit(requests).result()


def sweep_layout(bins, bin_ranks: Mapping, split_bins, local_bins) -> tuple:
    """Host logic of ShardedBinSweep for one rank: (designated rank of every bin in `bins` -- the lowest rank holding
    part of it, 0 for a bin without contigs --; the split bins in `bins` order, which is the row order of the packed
    all-reduce on every rank; this rank's bins in `bins` order, the slots of its BinSweep; the position in `bins` of
    each of them, int32)."""
    designated = {b: min(bin_ranks[b], default=0) for b in bins}
    split = [b for b in bins if b in split_bins]
    local = [b for b in bins if b in local_bins]
    position = {b: i for i, b in enumerate(bins)}
    return designated, split, local, np.array([position[b] for b in local], dtype=np.int32)


def global_parts(parts, global_slot) -> list:
    """[(group number, hit records)] of a rank's BinSweep -> the same records with slots numbered in the sharded
    sweep's `bins` (global_slot[local slot]).  Returns new arrays."""
    out = []
    for g, h in parts:
        h = h.copy()
        h["slot"] = np.asarray(global_slot, dtype=np.int32)[h["slot"]]
        out.append((g, h))
    return out


class ShardedBinSweep:
    """The multi-GPU form of sweep.BinSweep over a ShardedMultiBinScorer: every bin's histograms and candidates on the
    GPUs of one box, with the same candidate frame as one GPU.  Every rank makes every call with the same arguments
    (like score_batch); the collectives go over scorer.group.

    Each rank fills one BinSweep over the requested bins it holds (one histogram launch per kind).  A bin split over
    several ranks was counted piecewise: the raw IUPAC and bipartite counters of all split bins are summed by one
    all-reduce per kind, and the marginalisation runs once on the sum, so the finished histograms are those of one GPU
    bit for bit (a row lies under windows at most 15 bp from it, less than a piece's 64 bp of halo; DESIGN.md §5).  The
    bin's designated rank, the lowest holding part of it, keeps the sum; the other holders zero their copy, which then
    passes no filter (min_mod >= 1).  candidates() gathers every rank's hit records and builds the frame on every rank;
    counts() and bipartite_iupac_counts() are answered by the designated rank and broadcast.  A bin without contigs
    has no counters on any rank: its counts are (0, 0) and it has no candidate rows."""

    def __init__(self, scorer, mod_type, bins=None, bipartite: bool = True):
        from .search import CANONICAL
        from .sweep import BinSweep

        self.scorer, self.mod_type, self.bipartite = scorer, mod_type, bool(bipartite)
        scorer.mod_types.index(mod_type)  # an unknown mod type raises ValueError on every rank, as in BinSweep
        self.canonical = CANONICAL[str(mod_type)]
        self.bins = list(scorer.bin_ranks) if bins is None else list(bins)
        for b in self.bins:
            if b not in scorer.bin_ranks:
                raise KeyError(b)
        if len(set(self.bins)) != len(self.bins):
            raise ValueError("a bin is listed twice")
        self.designated, split, local_bins, self._global_slot = sweep_layout(self.bins, scorer.bin_ranks,
                                                                              scorer.split_bins, scorer._local_bins)
        self.local = BinSweep(scorer.local, mod_type, local_bins, bipartite) if local_bins else None
        if split:
            self._merge_split(split)

    def _collective(self) -> bool:
        import torch.distributed as dist

        return self.scorer.world_size > 1 and dist.is_available() and dist.is_initialized()

    def _merge_split(self, split):
        """One all-reduce per histogram kind over a packed [n_split][size] int32 tensor, zero rows where this rank holds
        nothing; the designated rank writes the sums back, the other holders zero their slot."""
        import torch
        import torch.distributed as dist

        from .sweep import BIP_SIZE, HIST_SIZE

        sw, d = self.local, self.scorer.device
        held = [(i, sw.slot[b], self.designated[b] == self.scorer.rank) for i, b in enumerate(split)
                if sw is not None and b in sw.slot]
        kinds = [("raw", HIST_SIZE)] + ([("bip_raw", BIP_SIZE)] if self.bipartite else [])
        for attr, size in kinds:
            with torch.cuda.device(d):
                packed = torch.zeros((len(split), size), dtype=torch.int32, device=d)
                slots = getattr(sw, attr).view(-1, size) if sw is not None else None
                for i, s, _ in held:
                    packed[i] = slots[s]
                if self._collective():
                    dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=self.scorer.group)
                for i, s, keep in held:
                    slots[s] = packed[i] if keep else 0
        if sw is not None:
            sw._hist = sw._bip = None

    def candidates(self, min_mean: float = 0.7, min_mod: int = 50, ks=range(4, 9), bipartite: bool = True,
                   scratch_bytes: int = 8 << 30, capacity: int = 1 << 20, bipartite_letters: str = "ACGT",
                   prune: bool = False):
        """BinSweep.candidates over the sharded bins (same arguments, errors and frame): every rank runs its local
        passes, the hit records of all ranks are gathered, and every rank returns the whole frame."""
        from .sweep import _candidate_groups, _frame

        # the argument checks run on every rank before any collective, so a bad argument raises everywhere
        if self.local is not None:
            groups, bip_groups, parts = self.local._hits(min_mean, min_mod, ks, bipartite, scratch_bytes, capacity,
                                                         bipartite_letters, prune)
            parts = global_parts(parts, self._global_slot)
        else:
            _, groups, bip_groups = _candidate_groups(min_mod, ks, bipartite, bipartite_letters, self.bipartite)
            parts = []
        if self._collective():
            parts = gather_rows(parts, self.scorer.group)
        return _frame(parts, groups, bip_groups, self.bins, self.mod_type, self.canonical)

    def _answer(self, bin_name, method: str, *args):
        """The designated rank's BinSweep.<method>(bin_name, *args), broadcast to every rank; an error raised there is
        raised on every rank (the others would otherwise wait in the broadcast)."""
        import torch.distributed as dist

        if bin_name not in self.designated:
            raise KeyError(bin_name)
        src = self.designated[bin_name]
        out = [None]
        if self.scorer.rank == src:
            try:
                if self.local is not None and bin_name in self.local.slot:
                    out[0] = getattr(self.local, method)(bin_name, *args)
                else:  # a bin without contigs
                    out[0] = (0, 0)
            except Exception as exc:  # noqa: BLE001 -- re-raised below, on every rank
                out[0] = exc
        if self._collective():
            dist.broadcast_object_list(out, group=self.scorer.group, group_src=src)
        if isinstance(out[0], Exception):
            raise out[0]
        return out[0]

    def counts(self, bin_name, motif_iupac: str, mod_pos: int) -> tuple[int, int]:
        """BinSweep.counts: (n_mod, n_nomod) of one IUPAC 4..8-mer or ACGT bipartite motif in one bin, on every rank."""
        return self._answer(bin_name, "counts", motif_iupac, mod_pos)

    def bipartite_iupac_counts(self, bin_name, left: str, gap: int, right: str, mod_pos: int) -> tuple[int, int]:
        """BinSweep.bipartite_iupac_counts: the motif left + "N" * gap + right, halves over the 14 letters but N."""
        return self._answer(bin_name, "bipartite_iupac_counts", left, gap, right, mod_pos)

    def count_matrix(self, motifs, mod_positions, bins=None):
        """BinSweep.count_matrix over the sharded bins (same arguments, errors and result, on every rank): each rank
        gathers the rows of the bins it is the designated rank for (a split bin's sum is there) in one launch, every
        other row is zero, and one all-reduce of the int64 [bin][motif][2] matrix adds the ranks' rows."""
        import torch
        import torch.distributed as dist

        from .sweep import _bin_rows, _lookup_records

        # the checks run on every rank before the collective, so a bad argument raises everywhere
        records = _lookup_records(motifs, mod_positions, self.bipartite, "this BinSweep was made with bipartite=False")
        rows = _bin_rows(self.designated, bins)
        d, sw = self.scorer.device, self.local
        mine = [i for i, b in enumerate(rows)
                if self.designated[b] == self.scorer.rank and sw is not None and b in sw.slot]
        with torch.cuda.device(d):
            out = torch.zeros((len(rows), len(records), 2), dtype=torch.int64, device=d)
            if mine:
                out[torch.tensor(mine, device=d)] = sw._count_device(records, [sw.slot[rows[i]] for i in mine])
            if out.numel() and self._collective():
                dist.all_reduce(out, op=dist.ReduceOp.SUM, group=self.scorer.group)
            out = out.cpu().numpy()
        return out[..., 0], out[..., 1]


# ---------------------------------------------------------------------------------------------
# The contig x motif methylation-pattern table (K5) over the GPUs of one box.
# ---------------------------------------------------------------------------------------------
def _collective(world_size: int) -> bool:
    import torch.distributed as dist

    return world_size > 1 and dist.is_available() and dist.is_initialized()


def rank_extremes(values, device, world_size: int, group=None) -> tuple[np.ndarray, np.ndarray]:
    """(maximum, minimum) over the ranks of each of the small int64 `values`, on every rank, with ONE all-reduce (MAX
    over the values and their negations).  Every rank must call it with as many values."""
    import torch

    v = np.asarray(values, dtype=np.int64)
    t = torch.from_numpy(np.concatenate([v, -v])).to(device)
    if _collective(world_size):
        import torch.distributed as dist

        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    t = t.cpu().numpy()
    return t[:len(v)], -t[len(v):]


def motif_list_key(motifs) -> tuple[int, int]:
    """(count, 62-bit hash) of a list of motif strings -- a hash that does not depend on the process (unlike hash())."""
    import hashlib

    digest = hashlib.blake2b("\n".join(str(m) for m in motifs).encode(), digest_size=8).digest()
    return len(motifs), int.from_bytes(digest, "little") >> 2


def check_same_motifs(motifs, device, world_size: int, group=None) -> None:
    """Raise ValueError on every rank unless every rank passed the same motif list (count and hash compared)."""
    hi, lo = rank_extremes(motif_list_key(motifs), device, world_size, group)
    if (hi != lo).any():
        raise ValueError("the ranks were given different motif lists")


def place_columns(stats, value, columns, n_contigs: int):
    """Zero-filled [n_motifs, n_contigs, 3] int64 and [n_motifs, n_contigs] float64 tensors holding this rank's columns
    at their global contig index `columns` (stats / value: [n_motifs, len(columns)(, 3)] of the rank's contigs in local
    order; value may be None).  A cell without observations gets value 0.0, so that the ranks' tensors can be added."""
    import torch

    idx = torch.as_tensor(np.asarray(columns, dtype=np.int64), device=stats.device)
    out_s = torch.zeros((stats.shape[0], n_contigs, 3), dtype=torch.int64, device=stats.device)
    out_s[:, idx] = stats
    out_v = None
    if value is not None:
        out_v = torch.zeros((stats.shape[0], n_contigs), dtype=torch.float64, device=stats.device)
        out_v[:, idx] = torch.where(stats[:, :, 0] > 0, value, torch.zeros_like(value))
    return out_s, out_v


def gather_columns(stats, value, columns, n_contigs: int, world_size: int, group=None):
    """The whole table on every rank from each rank's own contig columns (place_columns): one all-reduce (sum) per
    tensor, then NaN where n_motif_obs == 0.  Exact: every cell has one owner and the other ranks add integer zeros or
    +0.0 to it."""
    out_s, out_v = place_columns(stats, value, columns, n_contigs)
    if _collective(world_size):
        import torch.distributed as dist

        dist.all_reduce(out_s, op=dist.ReduceOp.SUM, group=group)
        if out_v is not None:
            dist.all_reduce(out_v, op=dist.ReduceOp.SUM, group=group)
    if out_v is not None:
        out_v[out_s[:, :, 0] == 0] = float("nan")
    return out_s, out_v


class ShardedPatternTable:
    """The multi-GPU form of the K5 contig x motif table (pattern.methylation_pattern, the table detect_contamination
    and include_contigs read, nanomotif/main.py:167-178).  Every rank passes the same arguments.

    Whole contigs are assigned to ranks by plan_shards (greedy on bp, no bins); each rank packs only its own contigs and
    builds one PatternIndex per mod type over them, so the K5 kernels run unchanged on every rank.  Contigs are never
    cut: counts of pieces would add, medians would not (an exact merge needs every fraction of the contig in one place),
    and a contig larger than one rank's share only occurs in assemblies small enough for one GPU.  A rank without
    contigs still takes part in every collective.

    Rows each rank reads: a table (pandas / pyarrow / polars-like, with n_mod and n_diff) is cut to the rank's contigs
    on the host before the copy; a bgzip pileup with a tabix index (.tbi next to it) is read member by member for the
    rank's contigs only (dataload.load_contigs_pileup_bgzip); plain text, or bgzip without an index, is parsed whole on
    every rank against all contig names and then cut -- that path does not split the parse cost.

    With allow_assembly_pileup_mismatch=False a pileup row of a contig absent from the whole assembly raises the same
    ValueError on every rank, after one all-reduce of the flag (the first collective)."""

    def __init__(self, pileup, assembly, mod_types, rank: int, world_size: int, device=None, group=None,
                 min_valid_read_coverage: int = 3, min_valid_cov_to_diff_fraction: float = 0.8,
                 allow_assembly_pileup_mismatch: bool = True):
        import torch

        from .device import DeviceAssembly
        from .pattern import MISMATCH_ERROR, load_contigs, pileup_rows

        contigs = load_contigs(assembly)
        self._plan(list(contigs), [len(s) for s in contigs.values()], mod_types, rank, world_size, group)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        asm, rows, mismatch = None, None, False
        if len(self.columns):  # the rank holding the longest contig (rank 0) always reads, so it sees any mismatch
            asm = DeviceAssembly.from_sequences({n: contigs[n] for n in self.local_names}, self.device)
            if isinstance(pileup, str) and _tabix_indexed(pileup):
                rows, mismatch = self._tabix_rows(pileup, allow_assembly_pileup_mismatch)
            else:
                renumber = np.full(len(self.names), -1, dtype=np.int32)
                renumber[self.columns] = np.arange(len(self.columns), dtype=np.int32)
                rows, mismatch = pileup_rows(pileup, self.names, self.mod_types, allow_assembly_pileup_mismatch,
                                             self.device, renumber)
        if rank_extremes([int(mismatch)], self.device, self.world_size, group)[0][0]:
            raise ValueError(MISMATCH_ERROR)
        self._index(asm, rows, min_valid_read_coverage, min_valid_cov_to_diff_fraction)

    @classmethod
    def from_local(cls, assembly, rows, contigs, mod_types, rank: int, world_size: int, device=None, group=None,
                   min_valid_read_coverage: int = 3, min_valid_cov_to_diff_fraction: float = 0.8) -> "ShardedPatternTable":
        """The sharded table over a rank's DeviceAssembly and pileup rows built elsewhere -- e.g. generated or parsed on
        the device, when the rows cannot go through host text.  `contigs` = {name: sequence or length} of ALL ranks, the
        same on every rank; `assembly` must hold exactly the contigs plan_shards gives this rank, in `contigs` order, or
        be None when it gives none.  `rows`: device tensors as PatternIndex takes them, contig ids indexing `assembly`."""
        import torch

        self = cls.__new__(cls)
        self._plan(list(contigs), [_contig_length(s) for s in contigs.values()], mod_types, rank, world_size, group)
        held = [] if assembly is None else list(assembly.names)
        if held != self.local_names:
            raise ValueError(f"rank {self.rank}: the local assembly's contigs are not those the shard plan gives this rank")
        if assembly is not None:
            device = assembly.device
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._index(assembly, rows, min_valid_read_coverage, min_valid_cov_to_diff_fraction)
        return self

    def _plan(self, names, lengths, mod_types, rank, world_size, group):
        self.rank, self.world_size, self.group = int(rank), int(world_size), group
        self.names, self.mod_types = list(names), [str(m) for m in mod_types]
        self.owner = plan_shards(lengths, self.world_size)
        self.columns = np.flatnonzero(self.owner == self.rank)  # global index of every local contig, ascending
        self.local_names = [self.names[i] for i in self.columns]

    def _tabix_rows(self, path, allow_assembly_pileup_mismatch):
        from .bgzf import tabix_contigs
        from .dataload import load_contigs_pileup_bgzip

        mismatch = not allow_assembly_pileup_mismatch and bool(set(tabix_contigs(path)) - set(self.names))
        dr = load_contigs_pileup_bgzip(path, self.local_names, self.mod_types, with_counts=True, device=self.device)
        return dict(contig_id=dr.contig_id, position=dr.position, strand=dr.strand, mod_type=dr.mod_type, n_mod=dr.n_mod,
                    Nvalid_cov=dr.Nvalid_cov, n_diff=dr.n_diff), mismatch

    def _index(self, asm, rows, min_valid_read_coverage, min_valid_cov_to_diff_fraction):
        from .pattern import PatternIndex

        self.assembly = asm
        self.indices = [] if asm is None else [
            PatternIndex(asm, rows, ti, min_valid_read_coverage, min_valid_cov_to_diff_fraction)
            for ti in range(len(self.mod_types))]

    def table(self, motifs, median: bool = True, on_device: bool = False):
        """(stats int64 [n_motifs, n_contigs, 3], value float64 [n_motifs, n_contigs] or None) over ALL contigs in the
        assembly's order, on every rank: the arrays pattern.pattern_table returns for an index over the whole assembly,
        bit for bit (NaN where a cell has no observation).  `motifs`: strings <IUPAC>_<mod_type>_<mod_position>, the
        same list on every rank (checked; a difference raises ValueError on every rank).  on_device=True returns device
        tensors (for tables.bin_feature_matrix_device)."""
        import torch

        from .motif import Motif
        from .pattern import parse_motif_spec, pattern_table

        motifs = [str(m) for m in motifs]
        check_same_motifs(motifs, self.device, self.world_size, self.group)
        specs = [parse_motif_spec(m) for m in motifs]
        for _, mt, _ in specs:
            if mt not in self.mod_types:
                raise KeyError(f"mod type {mt!r} is not one of {self.mod_types}")
        nl, d = len(self.columns), self.device
        with torch.cuda.device(d):
            stats = torch.zeros((len(specs), nl, 3), dtype=torch.int64, device=d)
            value = torch.full((len(specs), nl), float("nan"), dtype=torch.float64, device=d) if median else None
            for ti, mt in enumerate(self.mod_types):
                sel = [i for i, s in enumerate(specs) if s[1] == mt]
                if not sel or self.assembly is None:
                    continue
                st, val = pattern_table(self.indices[ti], [Motif(specs[i][0], specs[i][2]).from_iupac() for i in sel],
                                        median, on_device=True)
                sel_d = torch.tensor(sel, dtype=torch.int64, device=d)
                stats[sel_d] = st
                if median:
                    value[sel_d] = val
            stats, value = gather_columns(stats, value, self.columns, len(self.names), self.world_size, self.group)
            if on_device:
                return stats, value
            return stats.cpu().numpy(), (value.cpu().numpy() if median else None)


def _tabix_indexed(path: str) -> bool:
    """A bgzip pileup with its tabix index next to it."""
    import os

    with open(path, "rb") as f:
        magic = f.read(2)
    return magic == b"\x1f\x8b" and os.path.exists(path + ".tbi")


def methylation_pattern(pileup, assembly, motifs, rank: int, world_size: int, group=None, threads: int = 1,
                        min_valid_read_coverage: int = 3, batch_size: int = 1000,
                        min_valid_cov_to_diff_fraction: float = 0.8, output: str | None = None,
                        allow_assembly_pileup_mismatch: bool = True,
                        output_type: MethylationOutput = MethylationOutput.Median, device=None):
    """pattern.methylation_pattern over the GPUs of one box (ShardedPatternTable): the same keyword arguments, and on
    every rank the DataFrame one GPU returns (same rows, order, values and dtypes).  Every rank passes the same
    arguments; only rank 0 writes `output`."""
    import torch

    from .pattern import load_contigs, parse_motif_spec, pattern_frame

    motifs = [str(m) for m in motifs]
    median = output_type == MethylationOutput.Median
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    check_same_motifs(motifs, device, world_size, group)  # the mod types below are derived from the motifs
    specs = [parse_motif_spec(m) for m in motifs]
    tab = ShardedPatternTable(pileup, load_contigs(assembly), sorted({mt for _, mt, _ in specs}), rank, world_size,
                              device, group, min_valid_read_coverage, min_valid_cov_to_diff_fraction,
                              allow_assembly_pileup_mismatch)
    stats, value = tab.table(motifs, median)
    df = pattern_frame(stats, value, specs, tab.names, median)
    if output is not None and int(rank) == 0:
        df.to_csv(output, sep="\t", index=False)
    return df
