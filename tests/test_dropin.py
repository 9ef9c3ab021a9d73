"""-m gpu: the drop-in claim, exercised.  A seeded GP loop written against the EvoGP python API (tests/dropin_run.py)
runs in a fresh process through this repo's `evogp` package, its front-end over its operator library.  The same loop,
run by the reference's unmodified package over its own CUDA extension, is recorded in tests/golden/ref_dropin.npz
(tests/golden/make_golden.py dropin).  Every generation must agree: populations bit for bit on the valid prefixes
(integer / index work), fitness within 1e-5 relative (BASELINE.json north_star)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_dropin.npz")
pytestmark = pytest.mark.gpu
GENS = 12


@pytest.fixture(scope="module")
def runs(native, tmp_path_factory):
    d = tmp_path_factory.mktemp("dropin")
    path = str(d / "ours.npz")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_run.py"), "shim", path, "600", str(GENS)],
                       cwd=str(d), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"run failed:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"
    return {"reference": np.load(GOLDEN), "ours": np.load(path)}


def close(a, b, rtol=1e-5):
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False
    ia = np.isinf(a)
    if not (np.array_equal(ia, np.isinf(b)) and np.array_equal(a[ia], b[ia])):
        return False
    m = ~(na | ia)
    return bool((np.abs(a[m].astype(np.float64) - b[m]) <= rtol * np.abs(b[m].astype(np.float64))).all())


def test_the_two_runs_used_different_native_code(runs):
    assert any(str(n).startswith("evogp_cuda.cpython") for n in runs["reference"]["native"])
    assert "evogp_cuda_ops.so" in list(runs["ours"]["native"]) and "libevogp_b200.so" in list(runs["ours"]["native"])


def test_seeded_loop_is_identical_to_the_reference_run(runs):
    ref, ours = runs["reference"], runs["ours"]
    for g in range(GENS):
        for name in ("type", "size", "value"):
            # SHA-256 of the valid prefixes of node_<name>, all trees of the generation
            assert ours[f"{name}{g}"] == ref[f"{name}{g}"], f"generation {g}: node_{name} differs"
        assert close(ours[f"fitness{g}"], ref[f"fitness{g}"]), f"generation {g}: fitness beyond 1e-5 relative"
        # per-tree outputs (Forest.batch_forward -> tree_evaluate) carry the same bits under both libraries, so the torch-mode
        # fitness that drives selection in both runs is identical, NaNs included
        ta, tb = ref[f"torch_fitness{g}"], ours[f"torch_fitness{g}"]
        assert np.array_equal(np.isnan(ta), np.isnan(tb)) and np.array_equal(ta[~np.isnan(ta)], tb[~np.isnan(tb)]), \
            f"generation {g}: torch-mode fitness differs in {(ta != tb).sum()} trees"


def test_forward_paths_and_pareto_front_agree(runs):
    ref, ours = runs["reference"], runs["ours"]
    assert close(ours["best_forward"], ref["best_forward"])
    assert close(ours["forest_forward"], ref["forest_forward"])
    assert close(ours["pareto_fitness"], ref["pareto_fitness"])
