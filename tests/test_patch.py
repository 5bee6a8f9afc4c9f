"""patch.install / the spawn-safe import hook against the UNMODIFIED reference package (when /root/reference is
mounted) or a stand-in namespace with the same by-name imports (GPU box).  The GPU tests re-run the bodies of the
reference's own tests of the patched names (tests/test_fasta.py:95-109, tests/test_motif_find.py:14-39) through the
patched module attributes, so they exercise exactly what a nanomotif caller would."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from nanomotif_b200 import api, patch
from oracle import ref_shim
from oracle import restate as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _stand_in():
    """A package shaped like the reference where it matters: find_motifs_bin imports subseq_indices BY NAME."""
    utils = types.SimpleNamespace(subseq_indices=O.subseq_indices)
    fmb = types.SimpleNamespace(subseq_indices=utils.subseq_indices,
                                methylated_motif_occourances=lambda m, s, a, b: O.methylated_motif_occourances(str(m), m.mod_position, s, a, b),
                                motif_model_contig=None, motif_model_bin=None, get_parent_scores=None)
    return types.SimpleNamespace(utils=utils, find_motifs_bin=fmb, motif=types.SimpleNamespace(Motif=api.Motif))


def _package():
    return ref_shim.load_reference() if ref_shim.reference_available() else _stand_in()


def test_install_swaps_every_name_and_uninstall_restores():
    pkg = _package()
    before = {(m, n): getattr(getattr(pkg, m), n) for m, names in patch._PATCHED.items() for n in names}
    saved = patch.install(pkg)
    try:
        assert pkg.utils.subseq_indices is api.subseq_indices
        assert pkg.find_motifs_bin.subseq_indices is api.subseq_indices  # imported by name, find_motifs_bin.py:18
        assert pkg.find_motifs_bin.methylated_motif_occourances is api.methylated_motif_occourances
        assert pkg.find_motifs_bin.motif_model_bin is api.motif_model_bin
        assert pkg.find_motifs_bin.motif_model_contig is api.motif_model_contig
        assert pkg.find_motifs_bin.get_parent_scores is api.get_parent_scores
    finally:
        patch.uninstall(pkg, saved)
    assert all(getattr(getattr(pkg, m), n) is f for (m, n), f in before.items())


def _write_stand_in_package(parent) -> None:
    """An importable `nanomotif` with the reference's module layout where the hook acts on it: find_motifs_bin
    imports subseq_indices from nanomotif.utils BY NAME (find_motifs_bin.py:18)."""
    pkg = parent / "nanomotif"
    pkg.mkdir()
    stub = "def {}(*args, **kwargs):\n    raise NotImplementedError\n\n\n"
    (pkg / "__init__.py").write_text("from . import find_motifs_bin, utils  # noqa: F401\n")
    (pkg / "utils.py").write_text(stub.format("subseq_indices"))
    (pkg / "find_motifs_bin.py").write_text("from nanomotif.utils import subseq_indices  # noqa: F401\n\n\n" + "".join(
        stub.format(n) for n in ("methylated_motif_occourances", "motif_model_contig", "motif_model_bin", "get_parent_scores")))


def test_spawned_interpreter_gets_the_backend_through_the_import_hook(tmp_path):
    """What a worker of get_context("spawn") sees: a fresh interpreter whose environment was prepared by
    enable_for_workers() patches nanomotif while importing it -- the reference package where its tree is mounted,
    otherwise a stand-in package written to a temporary directory."""
    env = dict(os.environ)
    if ref_shim.reference_available():
        load = "from oracle import ref_shim; nm = ref_shim.load_reference()"
    else:
        _write_stand_in_package(tmp_path)
        env["PYTHONPATH"] = os.pathsep.join(p for p in (str(tmp_path), env.get("PYTHONPATH")) if p)
        load = "import nanomotif as nm"
    code = ("import os, sys; sys.path.insert(0, %r); from nanomotif_b200 import patch; patch.enable_for_workers(); "
            "print(os.environ['PYTHONPATH']); print(os.environ['NMB200_PATCH'])" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, check=True).stdout.split("\n")
    env["PYTHONPATH"], env["NMB200_PATCH"] = out[0], out[1]
    child = (load + "; f = nm.find_motifs_bin; "
             "print(f.motif_model_bin.__module__, f.subseq_indices.__module__, nm.utils.subseq_indices.__module__, "
             "f.methylated_motif_occourances.__module__, f.get_parent_scores.__module__)")
    got = subprocess.run([sys.executable, "-c", child], capture_output=True, text=True, env=env, cwd=ROOT)
    assert got.returncode == 0, got.stderr
    assert got.stdout.split() == ["nanomotif_b200.api"] * 5
    env["NMB200_PATCH"] = "0"  # hook directory on the path but not enabled: the reference stays untouched
    got = subprocess.run([sys.executable, "-c", child], capture_output=True, text=True, env=env, cwd=ROOT)
    assert got.returncode == 0 and "nanomotif_b200" not in got.stdout


@pytest.mark.gpu
def test_reference_test_bodies_through_the_patched_names():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    pkg = _package()
    saved = patch.install(pkg)
    try:
        # body of tests/test_fasta.py:95-109 (test_subseq_indices), through both patched names
        seq = "AATTAAATTAAGTAAAT"
        for fn in (pkg.utils.subseq_indices, pkg.find_motifs_bin.subseq_indices):
            for pattern, expected in {"AATT": [0, 5], "AA.T": [0, 4, 5, 9, 13]}.items():
                assert fn(pattern, seq).tolist() == expected, f"Mismatch for pattern {pattern}"
        # bodies of tests/test_motif_find.py:14-39 (TestMethylatedMotifOccurrences), with the package's own Motif type
        motif = pkg.motif.Motif("ACG", 0)
        sequence = "TACGGACGCCACG"
        result = pkg.find_motifs_bin.methylated_motif_occourances(motif, sequence, np.array([1, 5]), np.array([10]))
        np.testing.assert_array_equal(result[0], np.array([1, 5]))
        np.testing.assert_array_equal(result[1], np.array([10]))
        result = pkg.find_motifs_bin.methylated_motif_occourances(motif, sequence, np.array([]), np.array([1, 10]))
        np.testing.assert_array_equal(result[0], np.array([]))
        np.testing.assert_array_equal(result[1], np.array([1, 10]))
        # motif_model_bin through the patched name: mutates and returns the model it is given (find_motifs_bin.py:1319)
        from nanomotif_b200 import synth

        rng = np.random.default_rng(3)
        s = synth.random_sequence(rng, 30000, 0.5)
        p = synth.synth_pileup(s, rng, depth=20, mod_types=("a",))
        pile = {"contig": np.full(len(p["position"]), "c", dtype=object), "position": p["position"],
                "strand": np.where(p["strand"] == 0, "+", "-").astype(object), "fraction_mod": p["fraction_mod"]}
        contigs = {"c": s.tobytes().decode()}
        model = api.BetaBernoulliModel()
        out = pkg.find_motifs_bin.motif_model_bin(pile, contigs, pkg.motif.Motif("GATC", 1), model, 0.3, 0.7)
        want = O.motif_model_bin(pile["contig"], pile["position"], pile["strand"], pile["fraction_mod"], contigs, "GATC", 1, fast=True)
        assert out is model and (model._alpha - 5, model._beta - 5) == tuple(want)
    finally:
        patch.uninstall(pkg, saved)
