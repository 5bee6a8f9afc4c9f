"""TEST INFRASTRUCTURE ONLY -- CPU restatement of nanomotif's motif-scoring hot path.

This module is the parity oracle for the CUDA path in ``nanomotif_b200/``.  It may be imported by
``tests/``, by ``__graft_entry__.smoke()`` and by ``bench.py``'s cpu_baseline / ``--impl reference``
legs, and by nothing else; the product never routes through it.

Every function restates one reference function with numpy / ``regex`` / scipy (the same third-party
calls the reference makes), citing the file:line it follows in MicrobialDarkMatter/nanomotif 1.1.2.
Parity status: PINNED.  ``tests/test_oracle_golden.py`` checks it against (a) the reference's own
known-answer tests (tests/test_fasta.py:95-109, tests/test_motif_find.py:14-39,
tests/test_dataload.py:37-69, tests/test_candidate.py:42-58) and (b) golden vectors produced by
running the real reference functions through ``oracle/ref_shim.py``
(``tests/golden/generate_golden.py`` -> ``tests/golden/*.json``).  The polars-dependent glue
(motif_model_contig's row split, motif_model_bin, get_parent_scores, filter_pileup,
filter_pileup_minimummod_frequency) is pinned too: ``oracle/minipolars.py`` implements the handful of
polars calls those functions make on numpy columns, the UNMODIFIED reference functions were run through
it (``tests/golden/generate_binmodel_golden.py`` -> ``binmodel_vectors.json``) and
``tests/test_binmodel_golden.py`` holds this module against the recorded results (and against the live
functions where the reference tree is mounted).  The adjacency filter is pinned by the reference's own
known answers (tests/test_dataload.py:37-69); its polars ``rolling`` call is not emulated.
``methylation_pattern`` (external Rust package, no source in the tree) is a written spec:
PARITY UNPINNED for that one function.
"""
from __future__ import annotations

import math
import random

import numpy as np
import regex
from scipy.special import psi
from scipy.stats import entropy

BASES = ["A", "T", "G", "C"]  # nanomotif/constants.py:1
COMPLEMENT = {"A": "T", "T": "A", "G": "C", "C": "G", "N": "N", ".": ".", "[": "]", "]": "[",
              "R": "Y", "Y": "R", "S": "S", "W": "W", "K": "M", "M": "K", "B": "V", "D": "H", "H": "D",
              "V": "B"}  # nanomotif/constants.py:14-20
MOD_TYPE_TO_CANONICAL = {"m": "C", "a": "A", "21839": "C"}  # nanomotif/constants.py:31-35
BASE_TO_VECTOR = {"A": [1, 0, 0, 0], "T": [0, 1, 0, 0], "G": [0, 0, 1, 0], "C": [0, 0, 0, 1],
                  "N": [1, 1, 1, 1], ".": [1, 1, 1, 1]}  # nanomotif/seq.py:41-48


# ---------------------------------------------------------------------------------------------
# motif string helpers (nanomotif/motif.py)
# ---------------------------------------------------------------------------------------------
def split_motif(s: str) -> list[str]:
    """motif.py:226-245."""
    return regex.findall(r"\[[^\]]*\]|.", s)


def strip_motif(s: str, mod_pos: int) -> tuple[str, int]:
    """new_stripped_motif, motif.py:213-224."""
    m = regex.search(r"[^.]", s)
    if m is None:
        return s, mod_pos
    return s.lstrip(".").rstrip("."), mod_pos - m.start()


def reverse_complement_motif(s: str, mod_pos: int) -> tuple[str, int]:
    """reverse_compliment, motif.py:260-266."""
    return "".join(COMPLEMENT[c] for c in reversed(s)), len(split_motif(s)) - mod_pos - 1


def motif_one_hot(s: str) -> np.ndarray:
    """one_hot, motif.py:247-258."""
    toks = split_motif(s)
    arr = np.zeros((len(toks), 4), dtype=int)
    for i, tok in enumerate(toks):
        for ch in tok:
            if ch in BASE_TO_VECTOR:
                arr[i, :] += BASE_TO_VECTOR[ch]
    return arr


# ---------------------------------------------------------------------------------------------
# a1 / a2: scan and gather-join
# ---------------------------------------------------------------------------------------------
def subseq_indices(subseq: str, seq: str) -> np.ndarray:
    """utils.py:44-67 -- overlapping regex matches, start positions, int64."""
    pattern = regex.compile(subseq)
    return np.fromiter((m.start() for m in pattern.finditer(seq, overlapped=True)), dtype=np.int64)


def subseq_indices_np(subseq: str, seq_bytes: np.ndarray) -> np.ndarray:
    """Same result as subseq_indices, vectorised for large contigs: a position matches when every
    non-'.' token contains the contig letter (regex-literal semantics: N only matches '.')."""
    toks = split_motif(subseq)
    n = len(seq_bytes) - len(toks) + 1
    if n <= 0:
        return np.zeros(0, dtype=np.int64)
    ok = np.ones(n, dtype=bool)
    for j, tok in enumerate(toks):
        if tok == ".":
            continue
        letters = tok.strip("[]").encode()
        ok &= np.isin(seq_bytes[j : j + n], np.frombuffer(letters, dtype=np.uint8))
    return np.flatnonzero(ok).astype(np.int64)


def methylated_motif_occourances(motif: str, mod_pos: int, sequence, meth: np.ndarray, nonmeth: np.ndarray,
                                 fast: bool = False):
    """find_motifs_bin.py:1234-1263."""
    assert len(motif) > 0, "Motif is empty"
    assert len(sequence) > 0, "Sequence is empty"
    if fast:
        idx = subseq_indices_np(motif, sequence) + mod_pos
    else:
        idx = subseq_indices(motif, sequence) + mod_pos
    meth_occ = meth[np.isin(meth, idx, assume_unique=True)]
    nonmeth_occ = nonmeth[np.isin(nonmeth, idx, assume_unique=True)]
    return meth_occ, nonmeth_occ


# ---------------------------------------------------------------------------------------------
# a3 / a4: per-contig and per-bin counts
# ---------------------------------------------------------------------------------------------
def motif_model_contig(position, strand, fraction_mod, contig, motif: str, mod_pos: int, low=0.3, high=0.7,
                       fast: bool = False):
    """find_motifs_bin.py:1285-1331 with the polars frame replaced by its columns.
    strand: array of '+'/'-'.  Returns (n_mod, n_nomod, positions dict)."""
    position = np.asarray(position, dtype=np.int64)
    strand = np.asarray(strand)
    fraction_mod = np.asarray(fraction_mod, dtype=np.float64)
    s_motif, s_pos = strip_motif(motif, mod_pos)  # :1307
    is_high = fraction_mod >= high  # :1308
    is_low = fraction_mod <= low  # :1309
    plus, minus = strand == "+", strand == "-"
    meth_fwd, non_fwd = position[is_high & plus], position[is_low & plus]  # :1311-1312
    meth_rev, non_rev = position[is_high & minus], position[is_low & minus]  # :1313-1314
    seq = np.frombuffer(contig.encode(), dtype=np.uint8) if fast else contig
    i_mf, i_nf = methylated_motif_occourances(s_motif, s_pos, seq, meth_fwd, non_fwd, fast)  # :1316
    rc_motif, rc_pos = reverse_complement_motif(s_motif, s_pos)
    i_mr, i_nr = methylated_motif_occourances(rc_motif, rc_pos, seq, meth_rev, non_rev, fast)  # :1317
    n_mod = len(i_mf) + len(i_mr)  # :1320
    n_nomod = len(i_nf) + len(i_nr)
    return n_mod, n_nomod, dict(index_meth_fwd=i_mf, index_nonmeth_fwd=i_nf, index_meth_rev=i_mr,
                                index_nonmeth_rev=i_nr)


def motif_model_bin(contig_col, position, strand, fraction_mod, contigs: dict, motif: str, mod_pos: int,
                    low=0.3, high=0.7, fast: bool = False):
    """find_motifs_bin.py:1265-1283: the same model threaded through every contig = plain sums.
    Returns (n_mod, n_nomod) to be added to the Beta(5,5) prior."""
    contig_col = np.asarray(contig_col)
    n_mod = n_nomod = 0
    for name, seq in contigs.items():
        sel = contig_col == name  # :1274
        a, b, _ = motif_model_contig(np.asarray(position)[sel], np.asarray(strand)[sel],
                                     np.asarray(fraction_mod)[sel], seq, motif, mod_pos, low, high, fast)
        n_mod += a
        n_nomod += b
    return n_mod, n_nomod


# ---------------------------------------------------------------------------------------------
# a5 - a7: posterior and scores (nanomotif/model.py, find_motifs_bin.py:1360-1379, :901-924)
# ---------------------------------------------------------------------------------------------
PRIOR_ALPHA = PRIOR_BETA = 5  # model.py:8-9


def posterior(n_mod: int, n_nomod: int) -> tuple[int, int]:
    return PRIOR_ALPHA + n_mod, PRIOR_BETA + n_nomod  # model.py:37-39


def beta_mean(alpha, beta) -> float:
    return alpha / (alpha + beta)  # model.py:48-49


def _ppc_per_obs(alpha, beta, n_pos, n_neg) -> float:
    """posterior_predictive_per_obs, model.py:78-92."""
    n_new = n_pos + n_neg
    if n_new == 0:
        return 0.0
    e_log_p = psi(alpha) - psi(alpha + beta)
    e_log_1mp = psi(beta) - psi(alpha + beta)
    return (n_pos * e_log_p + n_neg * e_log_1mp) / n_new


def predictive_evaluation_score(next_ab, cur_ab) -> float:
    """find_motifs_bin.py:1360-1379; arguments are (alpha, beta) INCLUDING the priors."""
    a_n, b_n = next_ab
    a_c, b_c = cur_ab
    extra_pos, extra_neg = a_c - a_n, b_c - b_n
    ppcp_next = _ppc_per_obs(a_n, b_n, a_n, b_n)
    ppcp_extra = _ppc_per_obs(a_n, b_n, extra_pos, extra_neg)
    return (beta_mean(a_n, b_n) / beta_mean(a_c, b_c)) * (ppcp_next - ppcp_extra)


def priority_function(next_ab, root_ab) -> float:
    """find_motifs_bin.py:915-923."""
    return (1 - next_ab[0] / root_ab[0]) * (next_ab[1] / root_ab[1])


# ---------------------------------------------------------------------------------------------
# a9 - a12: motif-growth step
# ---------------------------------------------------------------------------------------------
def reverse_complement_seq(s: str) -> str:
    return "".join(COMPLEMENT[c] for c in reversed(s))  # seq.py:297-299


def sample_at_indices(seq: str, indices, padding: int) -> list[str]:
    """seq.py:170-189 (strict bounds) + sample_at_index :148-168."""
    keep = [i for i in indices if (i > padding) and (i < (len(seq) - padding))]
    return [seq[i - padding : i + padding + 1] for i in keep]


def methylation_windows(seq: str, index_plus, index_minus, padding: int) -> list[str]:
    """find_motifs_bin.py:652-662: '+' windows, then reverse-complemented '-' windows."""
    out = list(sample_at_indices(seq, index_plus, padding))
    out += [reverse_complement_seq(w) for w in sample_at_indices(seq, index_minus, padding)]
    return out


def one_hot_windows(windows: list[str]) -> np.ndarray:
    """convert_to_DNAarray, seq.py:474-478 -> (N, W, 4) int64."""
    return np.array([[BASE_TO_VECTOR[b] for b in w] for w in windows], dtype=np.int64)


def filter_sequence_matches(arr: np.ndarray, mask: np.ndarray, keep_matches: bool = True):
    """seq.py:499-524; returns the boolean row selector and the filtered array (None when empty)."""
    if keep_matches:
        sel = np.all(arr <= mask, axis=(1, 2))
    else:
        sel = np.any(arr > mask, axis=(1, 2))
    out = arr[sel, :]
    return sel, (None if out.shape[0] == 0 else out)


def pssm(arr: np.ndarray) -> np.ndarray:
    """DNAarray.pssm, seq.py:526-537 -> (4, W) float64."""
    return arr.sum(axis=0).transpose() / arr.shape[0]


def background_pssm(windows: list[str]) -> np.ndarray:
    """EqualLengthDNASet.pssm, seq.py:391-422 (exact-letter counts; N adds nothing)."""
    n = len(windows)
    width = len(windows[0])
    out = np.zeros((4, width))
    for b, nuc in enumerate(BASES):
        for i in range(width):
            out[b, i] = sum(1 for w in windows if w[i] == nuc) / n
    return out


def sample_background(seq: str, length: int, n: int, base: str, rng: random.Random) -> list[str]:
    """sample_n_subsequences_unique, seq.py:202-225 (the reference uses the module-level `random`)."""
    max_start = len(seq) - length + 1
    mid = length // 2
    valid = [s for s in range(max_start) if seq[s + mid] == base]
    starts = rng.sample(valid, n)
    return [seq[s : s + length] for s in starts]


def n_background_samples(contig_length: int, frequency: float = 0.01) -> int:
    return int(max(math.ceil(contig_length * frequency), 50))  # find_motifs_bin.py:633


def kl_children(motif: str, mod_pos: int, meth_pssm: np.ndarray, bin_pssm: np.ndarray, min_kl: float = 0.05,
                freq_threshold: float = 0.15):
    """_motif_child_nodes_kl_dist_max, find_motifs_bin.py:957-1023.
    Returns (kl vector, list of (child motif string, mod_pos))."""
    kl = entropy(meth_pssm, bin_pssm)  # :974
    toks = split_motif(motif)
    evaluated = np.array([i for i, b in enumerate(toks) if b == "."])  # :978
    if evaluated.size == 0:
        return kl, []
    masked = kl.copy()
    masked[~np.isin(np.arange(len(toks)), evaluated)] = 0  # :983
    if np.max(masked) < min_kl:  # :985-987
        return kl, []
    pos = int(np.argmax(masked))  # :989
    higher = meth_pssm[:, pos] > bin_pssm[:, pos] * 0.5  # :992
    above = meth_pssm[:, pos] > freq_threshold  # :995
    bases = [BASES[int(i)] for i in np.argwhere(np.logical_and(higher, above)).reshape(-1)]
    children = []
    for base in bases:  # :1019-1023
        t = list(toks)
        t[pos] = base
        children.append(("".join(t), mod_pos))
    return kl, children


# ---------------------------------------------------------------------------------------------
# a13: load_pileup (nanomotif/dataload.py:72-100), plain Python instead of polars' CSV reader
# ---------------------------------------------------------------------------------------------
def load_pileup_text(text: str) -> dict:
    """dataload.py:72-100 on the text of a modkit bedMethyl file: tab-separated, no header, 18 columns
    (schema :15-34); keeps columns 1, 2, 4, 6, 11, 10 and divides column 11 by 100 (:85).  polars parses
    Float64 text to the correctly rounded double, which is what float() does.  "NA" / "null" are nulls
    (:82) -> None here.  Extra columns 12 (n_mod) and 17 (n_diff) are returned for the pattern table."""
    null = ("NA", "null", "")
    num = lambda s, f: None if s in null else f(s)
    cols = {k: [] for k in ("contig", "position", "mod_type", "strand", "fraction_mod", "Nvalid_cov", "n_mod", "n_diff")}
    for line in text.split("\n"):
        line = line.rstrip("\r")
        if not line:
            continue
        f = line.split("\t")
        if len(f) < 18:
            raise ValueError("bedMethyl line with fewer than 18 columns")
        pct = num(f[10], float)
        cols["contig"].append(f[0])
        cols["position"].append(num(f[1], int))
        cols["mod_type"].append(f[3])
        cols["strand"].append(f[5])
        cols["fraction_mod"].append(None if pct is None else pct / 100)
        cols["Nvalid_cov"].append(num(f[9], int))
        cols["n_mod"].append(num(f[11], int))
        cols["n_diff"].append(num(f[16], int))
    return cols


# ---------------------------------------------------------------------------------------------
# a13: pileup filters (nanomotif/dataload.py:191-247), columns instead of a polars frame
# ---------------------------------------------------------------------------------------------
def filter_pileup(nvalid_cov, min_coverage: int = 5) -> np.ndarray:
    """dataload.py:191-200 -> boolean keep mask."""
    return np.asarray(nvalid_cov) > min_coverage


def filter_pileup_minimummod_frequency(contig, mod_type, fraction_mod, methylation_threshold=0.7,
                                       min_mod_frequency=0.0001, min_mods_pr_contig=50) -> np.ndarray:
    """dataload.py:202-226 -> boolean keep mask."""
    contig, mod_type = np.asarray(contig), np.asarray(mod_type)
    fraction_mod = np.asarray(fraction_mod, dtype=np.float64)
    key = np.char.add(np.char.add(contig.astype(str), "_"), mod_type.astype(str))
    uniq, inv = np.unique(key, return_inverse=True)
    n_pos = np.bincount(inv, minlength=len(uniq))
    n_mod = np.bincount(inv, weights=(fraction_mod > methylation_threshold).astype(np.float64),
                        minlength=len(uniq)).astype(np.int64)
    ok = ((n_mod / n_pos) > min_mod_frequency) & (n_mod > min_mods_pr_contig)
    return ok[inv]


def filter_pileup_adjacency_filter(contig, strand, position, fraction_mod, methylation_threshold=0.7,
                                   adjacency_distance=8) -> np.ndarray:
    """dataload.py:228-247 -> boolean keep mask (row order of the input; the reference returns rows
    sorted by position within (contig, strand) groups).

    polars rolling(index_column=position, period=window, offset=-(window//2+1)) looks at rows with
    position in (p - window//2 - 1, p - window//2 - 1 + window] = [p - d, p + d] for window = 2d+1,
    over ALL mod types of the (contig, strand) group.  A row is kept when its fraction equals the
    window maximum or is below the threshold.

    Null fractions ("NA" / "null" in column 11, NaN here): polars' rolling max skips nulls, so a NaN
    neighbour does not take part in the window maximum (np.max would return NaN and drop every
    above-threshold row whose window holds one).  A NaN row itself is dropped: both of its tests are
    null in polars, which filter() treats as false."""
    contig, strand = np.asarray(contig), np.asarray(strand)
    position = np.asarray(position, dtype=np.int64)
    fraction_mod = np.asarray(fraction_mod, dtype=np.float64)
    window = adjacency_distance * 2 + 1
    lo_off = -(window // 2 + 1)
    keep = np.zeros(len(position), dtype=bool)
    key = np.char.add(np.char.add(contig.astype(str), "\t"), strand.astype(str))
    for g in np.unique(key):
        rows = np.flatnonzero(key == g)
        order = rows[np.argsort(position[rows], kind="stable")]
        p, f = position[order], fraction_mod[order]
        left = np.searchsorted(p, p + lo_off, side="right")  # first index with pos > p + lo_off
        right = np.searchsorted(p, p + lo_off + window, side="right")  # one past last pos <= upper
        for k in range(len(order)):
            w = f[left[k] : right[k]]
            w = w[~np.isnan(w)]
            roll_max = w.max() if len(w) else np.nan
            keep[order[k]] = (f[k] == roll_max) or (f[k] < methylation_threshold)
    return keep


# ---------------------------------------------------------------------------------------------
# a14: contig x motif methylation-pattern table.  NOT a restatement of reference code: the operator is
# the external Rust package epimetheus-py 0.7.5 (call site nanomotif/main.py:167-178) whose source is
# not in the reference tree.  This is the written spec of SURVEY.md 8c / DESIGN.md K5 -- parity of the
# CUDA path is "exact vs this spec, UNPINNED vs the reference".
# ---------------------------------------------------------------------------------------------
IUPAC_TO_REGEX = {"A": "A", "T": "T", "C": "C", "G": "G", "R": "[AG]", "Y": "[CT]", "S": "[CG]", "W": "[AT]",
                  "K": "[GT]", "M": "[AC]", "B": "[CGT]", "D": "[AGT]", "H": "[ACT]", "V": "[ACG]", "N": "."}  # seq.py:571-601


def methylation_pattern(contigs: dict, contig, position, strand, mod_type, n_mod, n_valid_cov, n_diff, motifs,
                        min_valid_read_coverage=3, min_valid_cov_to_diff_fraction=0.8, weighted_mean=False):
    """Returns rows (contig, motif, mod_type, mod_position, methylation_value, mean_read_cov, n_motif_obs)."""
    contig = np.asarray(contig).astype(str)
    position = np.asarray(position, dtype=np.int64)
    strand = np.asarray(strand).astype(str)
    mod_type = np.asarray(mod_type).astype(str)
    n_mod = np.asarray(n_mod, dtype=np.int64)
    cov = np.asarray(n_valid_cov, dtype=np.int64)
    diff = np.asarray(n_diff, dtype=np.int64)
    rows = []
    for spec in motifs:
        iupac, mt, mp = spec.rsplit("_", 2)
        mp = int(mp)
        rx = "".join(IUPAC_TO_REGEX[c] for c in iupac)
        rc_rx, rc_mp = reverse_complement_motif(rx, mp)
        for name, seq in contigs.items():
            fwd = set((subseq_indices(rx, seq) + mp).tolist())
            rev = set((subseq_indices(rc_rx, seq) + rc_mp).tolist())
            sel = (contig == name) & (mod_type == mt) & (cov >= min_valid_read_coverage)
            with np.errstate(divide="ignore", invalid="ignore"):
                sel &= (cov / (cov + diff)) >= min_valid_cov_to_diff_fraction
            idx = [i for i in np.flatnonzero(sel) if (position[i] in fwd if strand[i] == "+" else position[i] in rev)]
            if not idx:
                continue
            m, c = n_mod[idx], cov[idx]
            value = m.sum() / c.sum() if weighted_mean else float(np.median(m / c))
            rows.append((name, iupac, mt, mp, float(value), float(c.mean()), len(idx)))
    return rows


# ---------------------------------------------------------------------------------------------
# 8f rank 3: table products (nanomotif/utils.py:15-34, binnary/data_processing.py:174-269), pandas instead of polars
# ---------------------------------------------------------------------------------------------
def motif_type(motif_str: str) -> str:
    """utils.py:26-34 with seq.reverse_compliment (seq.py:645-647, constants.py:14-20)."""
    import re

    comp = {"A": "T", "T": "A", "G": "C", "C": "G", "N": "N", "R": "Y", "Y": "R", "S": "S", "W": "W", "K": "M", "M": "K",
            "B": "V", "D": "H", "H": "D", "V": "B"}
    if len(re.findall(r"(N){2,}", motif_str)) >= 2:
        return "ambiguous"
    if re.search(r"(N){3,}", motif_str):
        return "bipartite"
    if "".join(comp[b] for b in reversed(motif_str)) == motif_str:
        return "palindrome"
    return "non-palindrome"


def binnary_matrix(contig_methylation, contig_bins: dict, methylation_threshold: float = 24.0):
    """main.py:192-193 filter, then add_bin (:174-187), impute_contig_methylation_within_bin (:189-213) and
    create_matrix (:255-269) on a pandas frame with the columns of main.py:157-161.  Returns (contig names,
    matrix, feature names)."""
    df = contig_methylation
    df = df[df["n_motif_obs"].astype(np.float64) * df["mean_read_cov"] >= methylation_threshold].copy()
    df["motif_mod"] = df["motif"] + "_" + df["mod_type"] + "_" + df["mod_position"].astype(str)
    df["bin"] = [contig_bins.get(c, "unbinned") for c in df["contig"]]
    df = df.drop(columns=["mod_position", "mod_type", "motif"])
    df = df[df["bin"] != "unbinned"]
    g = df.assign(w=df["methylation_value"] * df["n_motif_obs"]).groupby(["bin", "motif_mod"], as_index=False).agg(
        num=("w", "sum"), den=("n_motif_obs", "sum"))
    g["mean_bin_methylation"] = g["num"] / g["den"]
    cross = df.drop_duplicates(subset=["contig", "bin"])[["contig", "bin"]]
    imp = cross.merge(g[["bin", "motif_mod", "mean_bin_methylation"]], on="bin", how="left")
    imp = imp.merge(df[["bin", "contig", "motif_mod", "methylation_value"]], on=["bin", "contig", "motif_mod"], how="left")
    imp = imp.sort_values(["bin", "contig", "motif_mod"], kind="stable")
    imp["methylation_value"] = imp["methylation_value"].where(imp["methylation_value"].notna(), imp["mean_bin_methylation"])
    contigs = list(dict.fromkeys(imp["contig"]))  # pivot keeps the order of first appearance
    feats = sorted(imp["motif_mod"].unique())
    mat = np.zeros((len(contigs), len(feats)))
    ci = {c: i for i, c in enumerate(contigs)}
    fi = {f: i for i, f in enumerate(feats)}
    for c, f, v in zip(imp["contig"], imp["motif_mod"], imp["methylation_value"]):
        mat[ci[c], fi[f]] = v
    return np.array(contigs, dtype=object), mat, np.array(feats, dtype=object)


# ---------------------------------------------------------------------------------------------
# K8: the exhaustive sweep as a table computation (no reference callable: the counts are those of motif_model_bin,
# find_motifs_bin.py:1265-1331, for every IUPAC motif of one length at once).  Used to check the identity the CUDA
# kernels rely on -- counts are additive over the concrete context of each classified row -- against brute force.
# ---------------------------------------------------------------------------------------------
IUPAC_ORDER = "ATGCRYSWKMBDHVN"  # nanomotif/constants.py:2
_IUPAC_MEMBERS = {"A": "A", "T": "T", "G": "G", "C": "C", "R": "AG", "Y": "CT", "S": "GC", "W": "AT", "K": "GT", "M": "AC",
                  "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT"}


def sweep_table(contigs: dict, contig, position, strand, fraction_mod, k: int, mod_pos: int, canonical: str = "A",
                low=0.3, high=0.7):
    """(n_mod, n_nomod) int64 arrays of 15^(k-1) entries: entry = the motif's letters except the modified position as
    base-15 digits in IUPAC_ORDER, first letter most significant.  Step 1: every classified pileup row adds one to
    hist[class][window], window = the k letters around it with the row at offset mod_pos ('-' rows: the reverse
    complement of the forward window, offset mirrored -- find_motifs_bin.py:1317), five letter states A T G C other.
    Step 2: per axis, sum the states that each IUPAC letter stands for (N, the regex wildcard, includes other)."""
    state = {"A": 0, "T": 1, "G": 2, "C": 3}
    comp = {0: 1, 1: 0, 2: 3, 3: 2, 4: 4}
    contig = np.asarray(contig).astype(str)
    position = np.asarray(position, dtype=np.int64)
    strand = np.asarray(strand).astype(str)
    fraction_mod = np.asarray(fraction_mod, dtype=np.float64)
    hist = np.zeros((2,) + (5,) * k, dtype=np.int64)
    for name, seq in contigs.items():
        d = [state.get(ch, 4) for ch in seq.upper()]
        sel = np.flatnonzero(contig == name)
        for p, st, f in zip(position[sel], strand[sel], fraction_mod[sel]):
            cls = 0 if f >= high else 1 if f <= low else -1
            if cls < 0 or not 0 <= p < len(d):
                continue
            if st == "+":
                s = p - mod_pos                      # window start on the forward strand
                letters = d[s:s + k] if s >= 0 and s + k <= len(d) else None
            else:
                s = p - (k - 1 - mod_pos)            # the motif is the reverse complement of the forward window
                letters = [comp[x] for x in reversed(d[s:s + k])] if s >= 0 and s + k <= len(d) else None
            if letters is not None:
                hist[(cls,) + tuple(letters)] += 1
    # fix the modified position's own letter, then expand every remaining axis 5 -> 15
    expand = np.zeros((15, 5), dtype=np.int64)
    for i, letter in enumerate(IUPAC_ORDER):
        for b in _IUPAC_MEMBERS[letter]:
            expand[i, state[b]] = 1
    expand[14, 4] = 1
    out = []
    for cls in (0, 1):
        t = np.take(hist[cls], state[canonical], axis=mod_pos)
        for axis in range(k - 1):
            t = np.moveaxis(np.tensordot(expand, t, axes=([1], [axis])), 0, axis)
        out.append(t.reshape(-1))
    return out[0], out[1]
