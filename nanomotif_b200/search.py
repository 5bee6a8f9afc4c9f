"""Host-side motif search over the device operators (the caller of the hot path).

Restates the control flow of the reference's best-first search and candidate loop

    MotifSearcher.run                  nanomotif/find_motifs_bin.py:1026-1182
    find_best_candidates (loop part)   nanomotif/find_motifs_bin.py:688-834
    get_parent_scores                  nanomotif/find_motifs_bin.py:1382-1433
    MotifTree.get_missed_candidates    nanomotif/motif.py:594-608

as *coroutines*: a search never calls the GPU itself, it yields requests

    ("score",  [motifs])   -> [BetaBernoulliModel]      (K2: motif_model_bin for each motif)
    ("expand", motif)      -> None | (n_active, pssm)   (K4: filter_sequence_matches(...).pssm())
    ("remove", motif)      -> None | remaining windows  (K4: filter_sequence_matches(keep_matches=False))

so that one driver can advance the searches of many (bin, mod_type) pairs in lock-step and submit ONE
batched scan launch per step (`run_lockstep`), which is what keeps a B200 busy (SURVEY.md 7 hard part
3, 8f rank 1).  Every decision (heap order, thresholds, pruning) follows the cited reference lines, so
a search visits exactly the motifs the reference visits.
"""
from __future__ import annotations

import heapq
from typing import Iterable, Mapping

import numpy as np

from .growth import kl_children
from .model import BetaBernoulliModel, predictive_evaluation_score, priority as priority_function
from .motif import Motif

CANONICAL = {"m": "C", "a": "A", "21839": "C"}  # nanomotif/constants.py:31-35


class MotifGraph:
    """Minimal directed graph with node attributes (the part of networkx.DiGraph / MotifTree the search uses)."""

    def __init__(self):
        self.nodes: dict[Motif, dict] = {}
        self._succ: dict[Motif, dict] = {}
        self._pred: dict[Motif, dict] = {}

    def has_node(self, n) -> bool:
        return n in self.nodes

    def add_node(self, n, **attrs):
        if n in self.nodes:
            self.nodes[n].update(attrs)
        else:
            self.nodes[n] = dict(attrs)
            self._succ[n] = {}
            self._pred[n] = {}

    def has_edge(self, u, v) -> bool:
        return u in self._succ and v in self._succ[u]

    def add_edge(self, u, v):
        for n in (u, v):
            if n not in self.nodes:
                self.add_node(n)
        self._succ[u][v] = True
        self._pred[v][u] = True

    def edges(self):
        return [(u, v) for u, vs in self._succ.items() for v in vs]

    def _reach(self, n, adj) -> set:
        seen, stack = set(), list(adj[n])
        while stack:
            x = stack.pop()
            if x not in seen:
                seen.add(x)
                stack.extend(adj[x])
        return seen

    def ancestors(self, n) -> set:
        return self._reach(n, self._pred)

    def descendants(self, n) -> set:
        return self._reach(n, self._succ)

    def get_missed_candidates(self, best_candidates, threshold: float = 3) -> set:
        """High-scoring nodes without a high-scoring ancestor and without a kept descendant (motif.py:594-608)."""
        high = {n for n, d in self.nodes.items() if d["score"] > threshold}
        out = set()
        for n in high:
            if any(a in high for a in self.ancestors(n)) or any(d in best_candidates for d in self.descendants(n)):
                continue
            if n not in best_candidates:
                out.add(n)
        return out


def motif_search(root: Motif, graph: MotifGraph | None, bin_pssm: np.ndarray, min_kl: float = 0.1,
                 freq_threshold: float = 0.15, max_rounds_since_new_best: int = 30, max_motif_length: int = 25):
    """Best-first expansion from `root` (coroutine; returns (graph, best_guess)).  find_motifs_bin.py:1026-1182."""
    graph = graph if graph is not None else MotifGraph()
    best_guess = root
    root_model = (yield ("score", [root]))[0]  # :1035
    best_score = predictive_evaluation_score(root_model, root_model)
    rounds_since_new_best = 0
    visited: set[Motif] = set()
    if not graph.has_node(root):
        graph.add_node(root, model=root_model, motif=root, visited=False, score=best_score, priority=0, depth=0)
    queue: list[tuple] = []
    heapq.heappush(queue, (0, 0, root))
    while queue:
        _, _, current = heapq.heappop(queue)
        if current in visited:
            continue
        attrs = graph.nodes[current]
        current_model, current_depth = attrs["model"], attrs.get("depth", 0)
        n_mod, n_nomod = current_model.get_raw_counts()
        if n_mod + n_nomod < 10:  # :1079 low support
            continue
        if len(current.string.strip(".")) > max_motif_length:  # :1088
            continue
        visited.add(current)
        attrs["visited"] = True
        rounds_since_new_best += 1
        expansion = yield ("expand", current)  # :1108-1113
        if expansion is None:
            continue
        _, meth_pssm = expansion
        neighbors = kl_children(current, meth_pssm, bin_pssm, min_kl=min_kl, freq_threshold=freq_threshold)
        fresh = [m for m in neighbors if m not in graph.nodes]
        fresh_models = dict(zip(fresh, (yield ("score", fresh)))) if fresh else {}
        for nxt in neighbors:
            is_new = nxt not in graph.nodes
            nxt_model = fresh_models[nxt] if is_new else graph.nodes[nxt]["model"]
            score = predictive_evaluation_score(nxt_model, current_model)  # :1140
            n_isolated = nxt.count_isolated_bases(isolation_size=1)
            prio = priority_function(nxt_model, root_model)
            if n_isolated > 0:
                prio *= pow(10, n_isolated)
            if not is_new:
                if graph.nodes[nxt]["score"] < score:
                    graph.nodes[nxt]["score"] = score
            else:
                graph.add_node(nxt, model=nxt_model, motif=nxt, visited=False, score=score, priority=prio,
                               depth=current_depth + 1)
            if not graph.has_edge(current, nxt):
                graph.add_edge(current, nxt)
            if nxt not in visited:
                a = graph.nodes[nxt]
                heapq.heappush(queue, (a["priority"], a["depth"], nxt))
            if score > best_score:
                best_score, best_guess, rounds_since_new_best = score, nxt, 0
        if rounds_since_new_best >= max_rounds_since_new_best:  # :1179
            break
    return graph, best_guess


def parent_scores(motif: Motif):
    """Coroutine form of get_parent_scores (find_motifs_bin.py:1382-1433): one batched score request."""
    split = motif.split()
    parents, positions = [], []
    for i, base in enumerate(split):
        if i == motif.mod_position or base in (".", "N"):
            continue
        toks = list(split)
        toks[i] = "."
        parents.append(Motif("".join(toks), motif.mod_position))
        positions.append(i)
    models = yield ("score", [motif] + parents)
    child = models[0]
    out = {}
    for parent, i, pm in zip(parents, positions, models[1:]):
        out[parent] = dict(motif_position=i, parent_model=pm, child_model=child,
                           score=predictive_evaluation_score(child, pm))
    return out


def find_candidates(mod_type: str, padding: int, bin_pssm: np.ndarray, total_windows: int, min_kl: float = 0.2,
                    max_dead_ends: int = 25, max_rounds_since_new_best: int = 30, score_threshold: float = 0.2,
                    remaining_sequences_threshold: float = 0.001, trace: list | None = None):
    """Candidate loop of find_best_candidates (find_motifs_bin.py:688-834) as a coroutine.
    Returns (graph, best_candidates) or None.  `trace` collects one record per outer round."""
    root = Motif("." * padding + CANONICAL[mod_type] + "." * padding, padding)
    best, dead_ends, graph = [], 0, None
    while True:
        if dead_ends >= max_dead_ends:
            break
        graph, naive = yield from motif_search(root, graph, bin_pssm, min_kl=min_kl,
                                               max_rounds_since_new_best=max_rounds_since_new_best)
        if naive == root:  # :717
            break
        temp, prune, single = naive, set(), False
        while True:  # prune positions whose parent scores are poor (:722-768)
            parents = yield from parent_scores(temp)
            mean_score = np.mean([d["score"] for d in parents.values()])
            for d in parents.values():
                if d["score"] < 0.4:
                    prune.add(d["motif_position"])
            if not prune:
                break
            toks = temp.split()
            for i in prune:
                toks[i] = "."
            pruned = Motif("".join(toks), temp.mod_position)
            if len(pruned.string.replace(".", "")) == 1:
                single = True
                break
            if pruned == temp:
                break
            temp = pruned
        if single or mean_score < score_threshold:  # :770-778
            graph.nodes[naive]["score"] = np.mean([d["score"] for d in parents.values()])
        elif temp != naive:  # :780-795
            child_model = next(iter(parents.values()))["child_model"]
            graph.add_node(temp, model=child_model, motif=temp, visited=True, score=mean_score, priority=0, depth=0)
            naive = temp
        else:
            graph.nodes[naive]["score"] = np.mean([d["score"] for d in parents.values()])
        remaining = yield ("remove", naive)  # :803
        rec = dict(naive=naive.string, score=float(graph.nodes[naive]["score"]), remaining=remaining)
        if trace is not None:
            trace.append(rec)
        if remaining is None:
            break
        if graph.nodes[naive]["score"] < score_threshold:  # :813
            dead_ends += 1
            rec["kept"] = False
            continue
        rec["kept"] = True
        best.append(naive)
        if remaining / total_windows < remaining_sequences_threshold:  # :821
            break
    if graph is None or len(graph.nodes) == 0:
        return None
    missed = graph.get_missed_candidates(best, score_threshold)  # :829-834
    missed = [c for c in missed if not c.sub_motif_of_any(best) or not any(b.sub_motif_of(c) for b in best)]
    for c in sorted(missed):
        best.append(c)
    return graph, best


# ---------------------------------------------------------------------------------------------
# merge re-scoring (SURVEY 8f rank 4)
# ---------------------------------------------------------------------------------------------


def merge_group(rows: list, clusters, merge_threshold: float = 0.5, trace: list | None = None):
    """Coroutine form of the per-(bin, mod_type) body of merge_motifs_in_df (find_motifs_bin.py:1438-1533).

    `rows`: this group's motif rows (dicts with motif, mod_position, score, reference, mod_type, model);
    `clusters`: the values of nanomotif.motif.merge_motifs(motifs) (motif.py:519-560): (merged motif, pre-merge
    motifs, pre-merge variants, new variants).  The reference scores the merged motif and every exploded variant
    with one motif_model_bin call each, cluster after cluster, then every accepted motif and its parents; here
    the group issues TWO score requests (all clusters at once, then all accepted motifs with their parents), and
    run_lockstep folds the requests of all groups into one launch each.  Returns the new rows."""
    clusters = [tuple(c) for c in clusters]
    request, layout = [], []
    for merged, _premerge, pre_variants, new_variants in clusters:
        if len(new_variants) == 0:  # :1456-1460
            layout.append(None)
            continue
        variants = list(pre_variants)
        layout.append((len(request), len(variants)))
        request += [merged] + variants
    models = (yield ("score", request)) if request else []
    merged_motifs, premerge_motifs = [], []
    for (merged, premerge, _pre, _new), where in zip(clusters, layout):
        rec = dict(merged=merged, scored=where is not None)
        if where is not None:
            at, n = where
            merge_model = models[at]
            variants_model = BetaBernoulliModel()  # :1470-1479: one model threaded through all variants
            for m in models[at + 1:at + 1 + n]:
                variants_model.update(m._alpha - m._alpha_prior, m._beta - m._beta_prior)
            rec["merge_score"] = predictive_evaluation_score(variants_model, merge_model)  # :1480
            rec["merge_model"], rec["variants_model"] = merge_model, variants_model
            rec["accepted"] = rec["merge_score"] < merge_threshold
        else:
            rec["accepted"] = True
        if trace is not None:
            trace.append(rec)
        if rec["accepted"]:
            merged_motifs.append(merged)
            premerge_motifs.extend(premerge)
    if not premerge_motifs:  # :1492-1496
        return list(rows)
    gone = {str.__str__(m) for m in premerge_motifs}
    out = [r for r in rows if str(r["motif"]) not in gone]  # :1498
    request, layout = [], []
    for motif in merged_motifs:  # :1501-1517, one request for every motif and all its parents
        split = motif.split()
        parents = []
        for i, base in enumerate(split):
            if i == motif.mod_position or base in (".", "N"):
                continue
            toks = list(split)
            toks[i] = "."
            parents.append(Motif("".join(toks), motif.mod_position))
        layout.append((len(request), len(parents)))
        request += [motif] + parents
    models = yield ("score", request)
    for motif, (at, n) in zip(merged_motifs, layout):
        model = models[at]
        scores = [predictive_evaluation_score(model, pm) for pm in models[at + 1:at + 1 + n]]
        out.append(dict(motif=motif.string, score=float(np.mean(scores)) if scores else -1, mod_position=motif.mod_position,
                        reference=rows[0]["reference"] if rows else None, mod_type=rows[0]["mod_type"] if rows else None,
                        model=model))  # :1518-1527
    return out


def merge_motifs_in_groups(groups: list, batch_score=None) -> list:
    """merge_motifs_in_df over many (bin, mod_type) groups in lock-step.  groups = [(rows, clusters, backend)] or
    [(rows, clusters, backend, merge_threshold)]; returns the new rows of every group, in order."""
    searches = [(merge_group(g[0], g[1], *(g[3:4])), g[2]) for g in groups]
    return run_lockstep(searches, batch_score)


# ---------------------------------------------------------------------------------------------
# drivers
# ---------------------------------------------------------------------------------------------


class GpuBinBackend:
    """Serves the requests of one (bin, mod_type) search from a BinScorer (K2) and a DeviceDNAarray (K4)."""

    def __init__(self, scorer, windows):
        self.scorer = scorer
        self.windows = windows
        self.remaining = windows

    def score(self, motifs: Iterable[Motif]) -> list[BetaBernoulliModel]:
        out = []
        for n_mod, n_nomod in self.scorer.score(list(motifs)):
            m = BetaBernoulliModel()
            m.update(int(n_mod), int(n_nomod))
            out.append(m)
        return out

    def expand(self, motif: Motif):
        import warnings

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            active = self.remaining.copy().filter_sequence_matches(motif.one_hot())
        return None if active is None else (active.shape[0], active.pssm())

    def remove(self, motif: Motif):
        import warnings

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            self.remaining = self.remaining.filter_sequence_matches(motif.one_hot(), keep_matches=False)
        return None if self.remaining is None else self.remaining.shape[0]

    def handle(self, request):
        kind, arg = request
        return {"score": self.score, "expand": self.expand, "remove": self.remove}[kind](arg)


class PoolBackend:
    """Backend of one search whose windows live in a shared growth.WindowPool (slot = its row range) and whose
    scorer is a BinContext of a shared MultiBinScorer: every request kind can be batched across searches."""

    def __init__(self, scorer, pool, slot: int):
        self.scorer, self.pool, self.slot = scorer, pool, slot

    def handle(self, request):
        kind, arg = request
        if kind == "score":
            return gpu_batch_score([(self, arg)])[0]
        if kind == "expand":
            return self.pool.expand_batch([(self.slot, arg)])[0]
        return self.pool.remove_batch([(self.slot, arg)])[0]


def _per_pool(requests, call):
    """Serve window requests pool by pool (one WindowPool per mod type): one launch per pool and round."""
    pools = []
    for b, _ in requests:
        if not any(b.pool is p for p in pools):
            pools.append(b.pool)
    if len(pools) == 1:
        return call(pools[0], [(b.slot, motif) for b, motif in requests])
    out = [None] * len(requests)
    for pool in pools:
        idx = [i for i, (b, _) in enumerate(requests) if b.pool is pool]
        for i, r in zip(idx, call(pool, [(requests[i][0].slot, requests[i][1]) for i in idx])):
            out[i] = r
    return out


def gpu_batch_expand(requests):
    """`batch_expand` for run_lockstep over PoolBackends (one launch per WindowPool)."""
    return _per_pool(requests, lambda pool, reqs: pool.expand_batch(reqs))


def gpu_batch_remove(requests):
    return _per_pool(requests, lambda pool, reqs: pool.remove_batch(reqs))


def gpu_batch_score(requests):
    """`batch_score` for run_lockstep when every backend's scorer is a BinContext of ONE MultiBinScorer:
    all pending motifs of all searches go into a single scan launch."""
    owner = requests[0][0].scorer.owner
    counts = owner.score_batch([(b.scorer, motifs) for b, motifs in requests])
    out = []
    for c in counts:
        models = []
        for n_mod, n_nomod in c:
            m = BetaBernoulliModel()
            m.update(int(n_mod), int(n_nomod))
            models.append(m)
        out.append(models)
    return out


def run(coroutine, backend):
    """Drive one search to completion against `backend`."""
    try:
        request = next(coroutine)
        while True:
            request = coroutine.send(backend.handle(request))
    except StopIteration as stop:
        return stop.value


DISCOVERY_COLUMNS = ("bin", "mod_type", "motif", "mod_position", "n_mod", "n_nomod", "score")


def candidate_rows(bin_name, mod_type, result) -> list:
    """Rows of one (bin, mod type) search: `result` = find_candidates' (graph, best) or None.  One row per best
    candidate, in the order of `best` (found, then missed): the motif and mod_position after new_stripped_motif(),
    n_mod / n_nomod = the node model's alpha - alpha0 and beta - beta0, score = the node's score in the graph."""
    if result is None:
        return []
    graph, best = result
    rows = []
    for motif in best:
        node = graph.nodes[motif]
        n_mod, n_nomod = node["model"].get_raw_counts()
        stripped = motif.new_stripped_motif()
        rows.append(dict(bin=bin_name, mod_type=mod_type, motif=stripped.string, mod_position=int(stripped.mod_position),
                         n_mod=int(n_mod), n_nomod=int(n_nomod), score=float(node["score"])))
    return rows


def discovery_frame(rows):
    """pandas frame of candidate_rows (DISCOVERY_COLUMNS, in the order given; int64 counts, float64 score)."""
    import pandas as pd

    df = pd.DataFrame(list(rows), columns=list(DISCOVERY_COLUMNS))
    return df.astype({"bin": object, "mod_type": object, "motif": object, "mod_position": np.int64, "n_mod": np.int64,
                      "n_nomod": np.int64, "score": np.float64})


def discover(scorer, mod_types=None, bins=None, padding: int = 20, min_kl: float = 0.05, min_motif_score: float = 1.5,
             seed=1):
    """The motif search of every (bin, mod type) pair of a MultiBinScorer on its GPU, all pairs in lock-step: the
    candidate loop of find_best_candidates (find_motifs_bin.py:330-372 + process_subpileup up to find_best_candidates)
    for a whole metagenome.  Returns a pandas frame with DISCOVERY_COLUMNS, one row per best candidate of every pair:
    bins in `bins` order (default: the scorer's), then `mod_types` order (default: the scorer's), then the order of
    find_candidates' `best` (found, then missed).  Defaults are the reference CLI's (search_frame_size 40 -> padding
    20, minimum_kl_divergence 0.05, min_motif_score 1.5, seed 1); the high methylation threshold is the scorer's.

    One growth.prepare_searches per mod type builds every pair's windows and background PSSM; then every score round
    of all pairs is ONE K2 launch, every expand / remove round one K4 launch per mod type.  Like the reference's
    per-worker set_seed(seed) (find_motifs_bin.py:171), the background draws of every pair start from random.seed(seed),
    so a pair's rows depend only on its own bin: not on the other bins, their order or a `bins` subset.  `seed` may
    also be a {bin: seed} mapping.  The caller's `random` state is restored afterwards.  A pair without methylation
    windows starts no search and has no rows.  Errors of prepare_searches (a contig too short for its background
    samples, a scorer without kept rows) pass through."""
    import random

    from . import growth

    mod_types = list(scorer.mod_types) if mod_types is None else list(mod_types)
    names = list(scorer._ranges) if bins is None else list(bins)
    for b in names:
        if b not in scorer._ranges:
            raise KeyError(b)
    if len(set(names)) != len(names):
        raise ValueError("a bin is listed twice")
    if len(set(mod_types)) != len(mod_types):
        raise ValueError("a mod type is listed twice")
    for mt in mod_types:
        scorer.mod_types.index(mt)  # ValueError for a mod type the scorer does not hold
    seeds = [seed[b] for b in names] if isinstance(seed, Mapping) else [seed] * len(names)
    if not names or not mod_types:
        return discovery_frame([])
    high = scorer.pileup.high
    pairs = []  # ((bin index, mod type index), coroutine, backend)
    state = random.getstate()
    try:
        for j, mt in enumerate(mod_types):
            pool, pssms, totals = growth.prepare_searches(scorer, mt, padding, high, bin_names=names, seeds=seeds)
            for i, b in enumerate(names):
                if totals[i] == 0:
                    continue
                co = find_candidates(mt, padding, pssms[i], totals[i], min_kl=min_kl, score_threshold=min_motif_score)
                pairs.append(((i, j), co, PoolBackend(scorer.context(b, mt), pool, i)))
    finally:
        random.setstate(state)
    results = run_lockstep([(co, be) for _, co, be in pairs], gpu_batch_score, gpu_batch_expand, gpu_batch_remove)
    by_pair = {key: res for (key, _, _), res in zip(pairs, results)}
    rows = []
    for key in sorted(by_pair):
        rows += candidate_rows(names[key[0]], mod_types[key[1]], by_pair[key])
    return discovery_frame(rows)


def run_lockstep(searches: list, batch_score=None, batch_expand=None, batch_remove=None) -> list:
    """Advance many searches together.  `searches` = [(coroutine, backend)].  Each round the pending requests
    of one kind are answered by ONE call of the matching hook -- `batch_score([(backend, motifs)])` (one K2
    launch with a job per search), `batch_expand` / `batch_remove` ([(backend, motif)], one K4 launch over a
    shared WindowPool); kinds without a hook go to each search's own backend.  Returns the results in order."""
    n = len(searches)
    results: list = [None] * n
    pending: dict[int, tuple] = {}
    for i, (co, _) in enumerate(searches):
        try:
            pending[i] = next(co)
        except StopIteration as stop:
            results[i] = stop.value
    while pending:
        answers: dict[int, object] = {}
        for kind, hook in (("score", batch_score), ("expand", batch_expand), ("remove", batch_remove)):
            ids = [i for i, r in pending.items() if r[0] == kind]
            if hook is not None and len(ids) > 1:
                answers.update(zip(ids, hook([(searches[i][1], pending[i][1]) for i in ids])))
        for i, r in pending.items():
            if i not in answers:
                answers[i] = searches[i][1].handle(r)
        nxt = {}
        for i, a in answers.items():
            try:
                nxt[i] = searches[i][0].send(a)
            except StopIteration as stop:
                results[i] = stop.value
        pending = nxt
    return results
