"""Seeded synthetic assemblies and modkit-style pileups (SURVEY.md section 8d generators).

Used by bench.py and the tests; there is no network for real datasets and the reference's bundled
pileups are absent from the mount.  Everything is numpy ``Generator(PCG64(seed))``.
"""
from __future__ import annotations

import numpy as np

# This module is loaded BY PATH by `bench.py --impl reference` (which must not import the package: the package
# dlopens libnmb200.so), so it has no package-relative imports at module level.
_BITS = {"A": 1, "T": 2, "G": 4, "C": 8}


def tokenize(motif_string: str) -> list[str]:
    """Per-position tokens of a regex-subset motif, bracket classes kept together."""
    return [t for t in __import__("re").findall(r"\[[^\]]*\]|.", motif_string)]


def token_mask(token: str) -> int:
    """Allowed-set of a token: bit0=A bit1=T bit2=G bit3=C; '.' = 0xF."""
    if token == ".":
        return 0xF
    m = 0
    for ch in token.strip("[]"):
        m |= _BITS[ch]
    return m


MOD_TYPES = ("a", "m", "21839")
CANONICAL = {"a": "A", "m": "C", "21839": "C"}  # nanomotif/constants.py:31-35
_COMP = {"A": "T", "T": "A", "G": "C", "C": "G"}
_CODE_OF = np.full(256, 4, dtype=np.uint8)
for _i, _b in enumerate("ATGC"):
    _CODE_OF[ord(_b)] = _i

# planted motifs in the style of nanomotif/datasets/e_coli_bin-motifs.tsv:2-4 (+ a 4mC motif)
DEFAULT_PLANTED = (("GATC", 1, "a"), ("CC[AT]GG", 1, "m"), ("GCAC......GTT", 2, "a"), ("AAC......GTGC", 1, "a"),
                   ("CCGG", 0, "21839"))


def random_sequence(rng: np.random.Generator, length: int, gc: float = 0.5, n_run_rate: float = 0.0) -> np.ndarray:
    """ASCII (uint8) i.i.d. sequence with GC fraction `gc`; optional runs of N (rate per bp, length 10-100)."""
    p = np.array([(1 - gc) / 2, (1 - gc) / 2, gc / 2, gc / 2])
    seq = np.frombuffer(b"ATGC", dtype=np.uint8)[rng.choice(4, size=length, p=p)].copy()
    if n_run_rate > 0 and length > 200:
        for s in rng.choice(length - 100, size=rng.poisson(n_run_rate * length), replace=False):
            seq[s : s + int(rng.integers(10, 101))] = ord("N")
    return seq


def find_occurrences(seq: np.ndarray, motif: str) -> np.ndarray:
    """Start positions of a regex-subset motif in an ASCII array (generator-side helper)."""
    toks = tokenize(motif)
    n = len(seq) - len(toks) + 1
    if n <= 0:
        return np.zeros(0, dtype=np.int64)
    codes = _CODE_OF[seq]
    ok = np.ones(n, dtype=bool)
    for j, t in enumerate(toks):
        m = token_mask(t)
        if m == 0xF:
            continue
        allowed = np.array([(m >> c) & 1 for c in range(4)] + [0], dtype=bool)
        ok &= allowed[codes[j : j + n]]
    return np.flatnonzero(ok).astype(np.int64)


def reverse_complement_motif(motif: str, mod_pos: int) -> tuple[str, int]:
    toks = tokenize(motif)
    out = []
    for t in reversed(toks):
        if t.startswith("["):
            out.append("[" + "".join(_COMP[c] for c in reversed(t[1:-1])) + "]")
        else:
            out.append(_COMP.get(t, t))
    return "".join(out), len(toks) - mod_pos - 1


def synth_pileup(seq: np.ndarray, rng: np.random.Generator, planted=DEFAULT_PLANTED, depth: int = 100,
                 mod_types=MOD_TYPES, p_meth: float = 0.95, p_unmeth: float = 0.02, false_high: float = 0.003,
                 with_counts: bool = False) -> dict:
    """Pileup columns for one contig: one row per canonical base on '+' and per complementary base on
    '-' for every mod type; rows are unique per (position, strand, mod_type) and sorted by position."""
    cols = {k: [] for k in ("position", "strand", "mod_type", "fraction_mod", "Nvalid_cov", "n_mod", "n_diff")}
    for mt in mod_types:
        base = CANONICAL[mt]
        truth_plus = np.zeros(len(seq), dtype=bool)
        truth_minus = np.zeros(len(seq), dtype=bool)
        for motif, mp, mtype in planted:
            if mtype != mt:
                continue
            truth_plus[find_occurrences(seq, motif) + mp] = True
            rc, rmp = reverse_complement_motif(motif, mp)
            truth_minus[find_occurrences(seq, rc) + rmp] = True
        for strand, letter, truth in ((0, base, truth_plus), (1, _COMP[base], truth_minus)):
            pos = np.flatnonzero(seq == ord(letter)).astype(np.int64)
            n = len(pos)
            cov = np.maximum(1, rng.poisson(depth, size=n)).astype(np.int64)
            is_meth = truth[pos] | (rng.random(n) < false_high)
            n_mod = rng.binomial(cov, np.where(is_meth, p_meth, p_unmeth)).astype(np.int64)
            percent = np.round(100.0 * n_mod / cov, 2)  # modkit prints two decimals
            cols["position"].append(pos)
            cols["strand"].append(np.full(n, strand, dtype=np.uint8))
            cols["mod_type"].append(np.full(n, mod_types.index(mt), dtype=np.uint8))
            cols["fraction_mod"].append(percent / 100.0)  # dataload.py:85
            cols["Nvalid_cov"].append(cov)
            cols["n_mod"].append(n_mod)
            cols["n_diff"].append(rng.poisson(depth * 0.02, size=n).astype(np.int64))
    out = {k: np.concatenate(v) for k, v in cols.items()}
    order = np.lexsort((out["mod_type"], out["strand"], out["position"]))
    out = {k: v[order] for k, v in out.items()}
    if not with_counts:
        out.pop("n_mod")
        out.pop("n_diff")
    return out


def random_motifs(rng: np.random.Generator, n: int, canonical: str = "A") -> list[tuple[str, int]]:
    """Fixed work list of SURVEY 8d cfg 2: length 4-13, 0-2 degenerate positions, 0-1 gap of 4-8; the
    modified base is a position holding `canonical`."""
    out = []
    while len(out) < n:
        length = int(rng.integers(4, 14))
        toks = [str(b) for b in rng.choice(list("ATGC"), size=length)]
        for _ in range(int(rng.integers(0, 3))):
            j = int(rng.integers(1, length - 1))
            k = int(rng.integers(2, 4))
            toks[j] = "[" + "".join(sorted(rng.choice(list("ACGT"), size=k, replace=False))) + "]"
        if rng.random() < 0.5 and length >= 6:
            gap = int(rng.integers(4, 9))
            at = int(rng.integers(2, length - 2))
            toks = toks[:at] + ["."] * gap + toks[at:]
        cands = [i for i, t in enumerate(toks) if t == canonical]
        if not cands:
            j = int(rng.integers(0, len(toks)))
            if toks[j] == "." or j in (0, len(toks) - 1) and False:
                continue
            toks[j] = canonical
            cands = [j]
        mp = int(rng.choice(cands))
        if toks[0] == "." or toks[-1] == ".":
            continue
        out.append(("".join(toks), mp))
    return out


def device_workload(device, total_bp: int = 1_500_000_000, n_contigs: int = 17000, seed: int = 3, n_modtypes: int = 1):
    """cfg3-shaped synthetic assembly built ON the device (text for 1.5 Gbp would not fit a host pipeline):
    lognormal contig lengths (min 2.5 kbp), i.i.d. bases, and class planes drawn directly as random subsets
    of the A ('+') / T ('-') positions (~25 % methylated, ~50 % unmethylated).  Returns
    (DeviceAssembly, DevicePileup)."""
    import torch

    from . import _lib
    from .device import DeviceAssembly, DevicePileup

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    rng = np.random.default_rng(seed)
    lens = rng.lognormal(mean=0.0, sigma=1.0, size=n_contigs)
    lens = np.maximum(2500, (lens / lens.sum() * total_bp).astype(np.int64))
    off = np.zeros(n_contigs, dtype=np.int64)
    off[1:] = np.cumsum(lens)[:-1]
    codes = torch.randint(0, 4, (int(lens.sum()),), dtype=torch.uint8, device=device, generator=g)
    # A=65 T=84 G=71 C=67 for codes 0..3 (order of nanomotif/constants.py:1)
    ascii_d = 65 + (codes == 1).to(torch.uint8) * 19 + (codes == 2).to(torch.uint8) * 6 + (codes == 3).to(torch.uint8) * 2
    del codes
    asm = DeviceAssembly([f"c{i}" for i in range(n_contigs)], lens, ascii_d, off, device)
    del ascii_d
    pile = DevicePileup(asm, n_modtypes, 0.3, 0.7)
    rec = asm.seq_records.view(asm.n_tiles, _lib.SEQ_REC_WORDS)
    x = rec[:, _lib.HALO_WORDS:_lib.HALO_WORDS + _lib.TILE_WORDS]
    y = rec[:, _lib.SEQ_PLANE_WORDS + _lib.HALO_WORDS:_lib.SEQ_PLANE_WORDS + _lib.HALO_WORDS + _lib.TILE_WORDS]
    # x, y and the class planes are lane-interleaved (slot order); bring the flat non-ACGT plane to slot order
    nn = asm.nonacgt[_lib.HALO_WORDS:_lib.HALO_WORDS + asm.n_words].view(asm.n_tiles, _lib.TILE_WORDS)
    nn = nn[:, torch.from_numpy(_lib.SLOT_WORD).to(device)]
    is_a, is_t = ~x & ~y & ~nn, ~x & y & ~nn
    cls = pile.class_records.view(n_modtypes, asm.n_tiles, 4, _lib.TILE_WORDS)

    def rnd():
        return torch.randint(-2**31, 2**31 - 1, x.shape, dtype=torch.int32, device=device, generator=g)

    for mt in range(n_modtypes):
        r1, r2 = rnd(), rnd()
        cls[mt, :, 0] = is_a & r1 & r2
        cls[mt, :, 1] = is_a & ~r1
        r1, r2 = rnd(), rnd()
        cls[mt, :, 2] = is_t & r1 & r2
        cls[mt, :, 3] = is_t & ~r1
    return asm, pile


def pattern_workload_lengths(total_bp: int = 1_500_000_000, n_contigs: int = 50_000, seed: int = 4) -> np.ndarray:
    """Contig lengths of device_pattern_workload (host only: what every rank needs to derive a shard plan)."""
    rng = np.random.default_rng(seed)
    lens = rng.lognormal(mean=0.0, sigma=1.0, size=n_contigs)
    return np.maximum(2500, (lens / lens.sum() * total_bp).astype(np.int64))


def device_pattern_workload(device, total_bp: int = 1_500_000_000, n_contigs: int = 50_000, seed: int = 4, depth: int = 30,
                            keep=None):
    """cfg4-shaped input of the contig x motif table built ON the device: `n_contigs` lognormal contigs and one
    read-level pileup row (n_mod, Nvalid_cov, n_diff) for every A on '+' and every T on '-' (mod type 'a').
    Returns (DeviceAssembly, rows) with rows = device tensors contig_id int32, position int64, strand uint8,
    n_mod / Nvalid_cov / n_diff int64 in (strand, contig, position) order.  `keep` (ascending contig indices): only
    those contigs, with the letters and rows they have in the whole workload; contig ids then index `keep` (one rank's
    share of a sharded run, the same data at every world size)."""
    import torch

    from .device import DeviceAssembly

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    lens = pattern_workload_lengths(total_bp, n_contigs, seed)
    off = np.zeros(n_contigs, dtype=np.int64)
    off[1:] = np.cumsum(lens)[:-1]
    codes = torch.randint(0, 4, (int(lens.sum()),), dtype=torch.uint8, device=device, generator=g)
    ascii_d = 65 + (codes == 1).to(torch.uint8) * 19 + (codes == 2).to(torch.uint8) * 6 + (codes == 3).to(torch.uint8) * 2
    names = [f"c{i}" for i in range(n_contigs)]
    if keep is None:
        asm = DeviceAssembly(names, lens, ascii_d, off, device)
    else:
        keep = np.asarray(keep, dtype=np.int64)
        sel = torch.zeros(n_contigs, dtype=torch.bool, device=device)
        sel[torch.from_numpy(keep).to(device)] = True
        sub_off = np.zeros(len(keep), dtype=np.int64)
        sub_off[1:] = np.cumsum(lens[keep])[:-1]
        asm = DeviceAssembly([names[i] for i in keep], lens[keep], ascii_d[torch.repeat_interleave(
            sel, torch.from_numpy(lens).to(device))], sub_off, device)
        renumber = torch.full((n_contigs,), -1, dtype=torch.int32, device=device)
        renumber[torch.from_numpy(keep).to(device)] = torch.arange(len(keep), dtype=torch.int32, device=device)
    del ascii_d
    bounds = torch.from_numpy(off[1:].copy()).to(device)
    off_d = torch.from_numpy(off).to(device)
    cols = {k: [] for k in ("contig_id", "position", "strand", "n_mod", "Nvalid_cov", "n_diff")}
    for strand, code in ((0, 0), (1, 1)):
        idx = torch.nonzero(codes == code).view(-1)
        cid = torch.bucketize(idx, bounds, right=True)
        n = int(idx.numel())
        cov = torch.randint(1, 2 * depth, (n,), dtype=torch.int64, device=device, generator=g)
        part = dict(contig_id=cid.to(torch.int32), position=idx - off_d[cid],
                    strand=torch.full((n,), strand, dtype=torch.uint8, device=device),
                    n_mod=(torch.rand(n, device=device, generator=g) * (cov + 1).to(torch.float32)).to(torch.int64).clamp_(max=cov),
                    Nvalid_cov=cov,
                    n_diff=torch.randint(0, depth // 3, (n,), dtype=torch.int64, device=device, generator=g))
        if keep is not None:
            mine = sel[cid]
            part = {k: v[mine] for k, v in part.items()}
            part["contig_id"] = renumber[part["contig_id"].long()]
        for k, v in part.items():
            cols[k].append(v)
        del idx, cid, part
    del codes
    return asm, {k: torch.cat(v) for k, v in cols.items()}


# ---------------------------------------------------------------------------------------------
# cfg 3 (BASELINE.json configs[2], SURVEY 8d): metagenome of 300 bins x 5 Mbp, 20-200 contigs per bin,
# per-bin GC in U(0.3, 0.7), 1-5 planted motifs per bin, depth 30, three mod types.
# The PLAN (contig lengths, GC, planted motifs of every bin) is pure numpy and cheap, so every rank and
# the CPU arm derive the same one; a bin's sequence + pileup come either from numpy on the host
# (cfg3_bin_host: the bins the end-to-end leg and the CPU arm share) or from torch on the device
# (cfg3_bin_device: 1.5 Gbp would take ~15 minutes of numpy).
# ---------------------------------------------------------------------------------------------
PLANT_POOL = {
    "a": (("GATC", 1), ("GCAC......GTT", 2), ("AAC......GTGC", 1), ("G[AG].GAAG[CT]", 5), ("CTGCAG", 4),
          ("GAATTC", 2), ("GGA......TCC", 2), ("TCGA", 3), ("GAGG", 1)),
    "m": (("CC[AT]GG", 1), ("GGCC", 2), ("GC.GC", 1), ("CCGG", 1), ("GATC", 3)),
    "21839": (("CCGG", 0), ("GCGC", 1), ("CC[AT]GG", 0)),
}


def cfg3_plan(n_bins: int = 300, bin_bp: int = 5_000_000, seed: int = 3) -> dict:
    """Contig lengths, bin of every contig, per-bin GC and planted motifs.  Contig names are contig_<i>,
    bins bin_<j> (SURVEY 8d); contigs of a bin are consecutive."""
    rng = np.random.default_rng(seed)
    lengths, bin_of, gc, planted, ranges = [], [], [], [], []
    for b in range(n_bins):
        n = int(round(20 * 10 ** rng.uniform(0.0, 1.0)))  # 20-200 contigs, log-uniform (~78 on average)
        w = rng.lognormal(mean=0.0, sigma=1.0, size=n)
        lens = np.maximum(2500, (w / w.sum() * bin_bp).astype(np.int64))
        ranges.append((len(lengths), len(lengths) + n))
        lengths.extend(lens.tolist())
        bin_of.extend([b] * n)
        gc.append(float(rng.uniform(0.3, 0.7)))
        pool = [(m, p, mt) for mt in MOD_TYPES for m, p in PLANT_POOL[mt]]
        k = int(rng.integers(1, 6))
        planted.append(tuple(pool[i] for i in sorted(rng.choice(len(pool), size=k, replace=False))))
    return {"lengths": np.asarray(lengths, dtype=np.int64), "bin_of": np.asarray(bin_of, dtype=np.int32),
            "gc": gc, "planted": planted, "ranges": ranges, "n_bins": n_bins, "seed": seed, "depth": 30}


def cfg3_bin_host(plan: dict, b: int) -> dict:
    """Bin b generated with numpy: {"ascii": uint8 (contigs concatenated), "lengths", and pileup columns
    contig (index within the bin, int32), position, strand, mod_type (index into MOD_TYPES), fraction_mod,
    Nvalid_cov} -- rows sorted by (contig, position) like a modkit pileup."""
    rng = np.random.default_rng([plan["seed"], 1000 + b])
    lo, hi = plan["ranges"][b]
    lens = plan["lengths"][lo:hi]
    seqs, cols = [], {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod", "Nvalid_cov")}
    for c, n in enumerate(lens.tolist()):
        seq = random_sequence(rng, n, plan["gc"][b], 1e-6)
        p = synth_pileup(seq, rng, planted=plan["planted"][b], depth=plan["depth"])
        seqs.append(seq)
        cols["contig"].append(np.full(len(p["position"]), c, dtype=np.int32))
        for k in ("position", "strand", "mod_type", "fraction_mod", "Nvalid_cov"):
            cols[k].append(p[k])
    out = {k: np.concatenate(v) for k, v in cols.items()}
    out["ascii"] = np.concatenate(seqs)
    out["lengths"] = lens
    return out


def _planted_truth_device(codes, starts_ok_len, motif: str, mod_pos: int):
    """Boolean tensor over the bin's concatenated positions: True at the modified base of every occurrence of
    `motif` that lies inside one contig.  codes: uint8 (0 A, 1 T, 2 G, 3 C, 4 other); starts_ok_len(len) ->
    bool tensor of the starts whose whole occurrence stays inside its contig."""
    import torch

    toks = tokenize(motif)
    n = codes.numel() - len(toks) + 1
    ok = starts_ok_len(len(toks))[:n].clone()
    for j, t in enumerate(toks):
        m = token_mask(t)
        if m == 0xF:
            continue
        allowed = torch.tensor([(m >> c) & 1 for c in range(4)] + [0], dtype=torch.bool, device=codes.device)
        ok &= allowed[codes[j:j + n].long()]
    truth = torch.zeros(codes.numel(), dtype=torch.bool, device=codes.device)
    truth[torch.nonzero(ok).view(-1) + mod_pos] = True
    return truth


def cfg3_bin_device(plan: dict, b: int, device, p_meth: float = 0.95, p_unmeth: float = 0.02,
                    false_high: float = 0.003, ascii_only: bool = False) -> dict:
    """Bin b generated with torch on `device` (same distributions as cfg3_bin_host, different draws):
    {"ascii": uint8 device tensor, "lengths", "contig" int32, "position" int64, "strand" uint8, "mod_type" uint8,
    "fraction_mod" float64} (device tensors; rows grouped by mod type and strand, positions ascending).
    ascii_only: just the sequence (the first draw of the bin's generator, so a later full call repeats it)."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(plan["seed"] * 100003 + b)
    lo, hi = plan["ranges"][b]
    lens = plan["lengths"][lo:hi]
    total = int(lens.sum())
    gc = plan["gc"][b]
    u = torch.rand(total, device=device, generator=g)
    at = (1.0 - gc) / 2
    codes = (u >= at).to(torch.uint8) + (u >= 2 * at).to(torch.uint8) + (u >= 2 * at + gc / 2).to(torch.uint8)
    del u
    rng = np.random.default_rng([plan["seed"], 2000 + b])
    for s in rng.integers(0, max(1, total - 100), size=rng.poisson(1e-6 * total)):
        codes[int(s):int(s) + int(rng.integers(10, 101))] = 4
    lut = torch.tensor([65, 84, 71, 67, 78], dtype=torch.uint8, device=device)  # A T G C N
    ascii_d = lut[codes.long()]
    if ascii_only:  # the sequence is the generator's first draw: a second call with the same seed repeats it
        return {"ascii": ascii_d, "lengths": lens}
    ends = torch.from_numpy(np.cumsum(lens)).to(device)
    pos_all = torch.arange(total, device=device)
    cid_all = torch.bucketize(pos_all, ends, right=True)
    start_of = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)[:-1]])).to(device)
    local_all = pos_all - start_of[cid_all]
    remain = ends[cid_all] - pos_all  # positions left in the contig, this one included

    def starts_ok_len(n):
        return remain >= n

    comp = {0: 1, 1: 0, 2: 3, 3: 2}
    cols = {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod")}
    for mt, name in enumerate(MOD_TYPES):
        base = "ATGC".index(CANONICAL[name])
        truth_p = torch.zeros(total, dtype=torch.bool, device=device)
        truth_m = torch.zeros(total, dtype=torch.bool, device=device)
        for motif, mp, mtype in plan["planted"][b]:
            if mtype != name:
                continue
            truth_p |= _planted_truth_device(codes, starts_ok_len, motif, mp)
            rc, rmp = reverse_complement_motif(motif, mp)
            truth_m |= _planted_truth_device(codes, starts_ok_len, rc, rmp)
        for strand, code, truth in ((0, base, truth_p), (1, comp[base], truth_m)):
            idx = torch.nonzero(codes == code).view(-1)
            n = int(idx.numel())
            cov = torch.poisson(torch.full((n,), float(plan["depth"]), device=device), generator=g).clamp_(min=1.0)
            is_meth = truth[idx] | (torch.rand(n, device=device, generator=g) < false_high)
            prob = torch.where(is_meth, torch.full_like(cov, p_meth), torch.full_like(cov, p_unmeth))
            n_mod = torch.binomial(cov, prob, generator=g)
            key = torch.round(1e4 * n_mod.double() / cov.double())  # modkit prints the percentage with two decimals
            cols["contig"].append(cid_all[idx].to(torch.int32))
            cols["position"].append(local_all[idx])
            cols["strand"].append(torch.full((n,), strand, dtype=torch.uint8, device=device))
            cols["mod_type"].append(torch.full((n,), mt, dtype=torch.uint8, device=device))
            cols["fraction_mod"].append((key / 100.0) / 100.0)  # dataload.py:85
    out = {k: torch.cat(v) for k, v in cols.items()}
    out["ascii"] = ascii_d
    out["lengths"] = lens
    return out


def frontier_worklist(seed: int, canonical: str, rounds: int = 64, width: int = 4, window: int = 20) -> list:
    """Search-shaped work list of one (bin, mod type): `rounds` expansions, each the <= `width` children of one
    parent that differ in the base added at ONE new position (find_motifs_bin.py:1116-1145: the children of an
    expansion share every other position).  A chain grows from the bare canonical base until it has 7-10
    constrained positions, then a new chain starts.  Returns [[(motif string, mod_pos), ...] per round]."""
    rng = np.random.default_rng([seed, 77])
    out = []
    parent, target = None, 0
    while len(out) < rounds:
        if parent is None:
            parent = {0: canonical}  # offset from the modified base -> base
            target = int(rng.integers(7, 11))
        free = [o for o in range(-window // 2, window // 2 + 1) if o not in parent and min(abs(o - k) for k in parent) <= 6]
        o = int(rng.choice(free))
        bases = [str(x) for x in rng.permutation(list("ACGT"))[:int(rng.integers(max(1, width - 1), width + 1))]]
        kids = []
        for bs in bases:
            cons = dict(parent)
            cons[o] = bs
            lo_, hi_ = min(cons), max(cons)
            kids.append(("".join(cons.get(i, ".") for i in range(lo_, hi_ + 1)), -lo_))
        out.append(kids)
        parent = dict(parent)
        parent[o] = bases[0]
        if len(parent) >= target:
            parent = None
    return out
