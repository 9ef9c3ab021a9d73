#!/usr/bin/env python
"""Runs a seeded GP loop written against the EvoGP python API (Forest / GeneticProgramming / operators /
SymbolicRegression) and dumps every generation.
    python tests/dropin_run.py reference out.npz   # the reference's UNMODIFIED package (baseline/_ref/evogp) over its own extension
    python tests/dropin_run.py ours out.npz        # the reference's package over this repo's operator library (evogp_cuda_ops.so)
    python tests/dropin_run.py shim out.npz        # this repo's `evogp` import shim: its own front-end and operator library
In `ours` mode the only thing replaced is the module `evogp.evogp_cuda` that evogp/tree/__init__.py:2 imports: a stub
whose import registered torch.ops.evogp_cuda.* from this repo instead — the swap INTEGRATION.md describes.
Populations are dumped as SHA-256 digests of their valid prefixes; fitness and forward outputs as values."""
import hashlib
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")


def main():
    mode, out = sys.argv[1], sys.argv[2]
    pop = int(sys.argv[3]) if len(sys.argv) > 3 else 600
    gens = int(sys.argv[4]) if len(sys.argv) > 4 else 12
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") not in (ROOT, os.path.join(ROOT, "tests"))]
    import numpy as np
    import torch

    if mode == "ours":
        sys.path.append(ROOT)
        from evogp_b200 import _native
        _native.load_ops()                                  # TORCH_LIBRARY(evogp_cuda) from evogp_cuda_ops.so
        sys.modules["evogp.evogp_cuda"] = types.ModuleType("evogp.evogp_cuda")
    front = ROOT if mode == "shim" else REF
    sys.path.insert(0, front)
    import evogp
    import evogp.tree as rt
    assert os.path.realpath(evogp.__file__).startswith(os.path.realpath(front)), evogp.__file__
    from evogp.algorithm import DefaultCrossover, DefaultMutation, DefaultSelection, GeneticProgramming
    from evogp.problem import SymbolicRegression

    loaded = [l.split()[-1] for l in open("/proc/self/maps") if "evogp" in l and l.rstrip().endswith(".so")]
    native = sorted(set(os.path.basename(p) for p in loaded))
    if mode != "reference":
        assert "evogp_cuda_ops.so" in native and not any(n.startswith("evogp_cuda.cpython") for n in native), native
    else:
        assert any(n.startswith("evogp_cuda.cpython") for n in native) and "libevogp_b200.so" not in native, native

    torch.manual_seed(1234)
    N, V = 256, 3
    X = torch.rand(N, V, device="cuda") * 4 - 2
    y = (X[:, :1] ** 2 * 0.5 + X[:, 1:2] * X[:, 2:3] - 1.0).contiguous()
    problem = SymbolicRegression(datapoints=X, labels=y)                      # fitness from the SR-fitness kernel (tree_SR_fitness)
    # Selection is driven by the reference's own "torch" mode (symbolic_regression.py:73-81: Forest.batch_forward ->
    # tree_evaluate per (tree, datapoint), reduced by torch): per-tree OUTPUTS are bit-identical under both operator
    # libraries, so both runs sort identical numbers.  (Kernel fitness differs in the last bits by summation order -
    # inside 1e-5, but enough to flip a near-tie in torch.sort and send the two runs down different histories.)
    selector = SymbolicRegression(datapoints=X, labels=y, execute_mode="torch")
    desc = rt.GenerateDescriptor(max_tree_len=64, input_len=V, output_len=1, using_funcs=["+", "-", "*", "/", "sin", "neg"],
                                 max_layer_cnt=5, const_samples=[-1, 0, 1, 0.5])
    algo = GeneticProgramming(initial_forest=rt.Forest.random_generate(pop_size=pop, descriptor=desc),
                              crossover=DefaultCrossover(),
                              mutation=DefaultMutation(mutation_rate=0.2, descriptor=desc.update(max_layer_cnt=3)),
                              selection=DefaultSelection(survival_rate=0.3, elite_rate=0.01), enable_pareto_front=True)
    dump = {}
    for g in range(gens):
        f = algo.forest
        fit = problem.evaluate(f)
        sel = selector.evaluate(f)
        lens = f.batch_subtree_size[:, 0].long()
        valid = (torch.arange(f.max_tree_len, device="cuda")[None, :] < lens[:, None])
        for name, a in (("value", f.batch_node_value), ("type", f.batch_node_type), ("size", f.batch_subtree_size)):
            prefixes = torch.where(valid, a, torch.zeros_like(a)).cpu().numpy()
            dump[f"{name}{g}"] = np.array(hashlib.sha256(prefixes.tobytes()).hexdigest())
        dump[f"fitness{g}"] = fit.cpu().numpy()
        dump[f"torch_fitness{g}"] = sel.cpu().numpy()
        sel = torch.where(torch.isnan(sel), torch.full_like(sel, float("-inf")), sel)     # pipeline/standard.py:43
        algo.step(sel)
    best = algo.forest[int(torch.argmax(torch.nan_to_num(problem.evaluate(algo.forest), nan=float("-inf"))))]
    dump["best_forward"] = best.forward(X).cpu().numpy()                     # Tree.forward -> tree_evaluate
    rows = X[torch.arange(algo.forest.pop_size, device="cuda") % N].contiguous()
    dump["forest_forward"] = algo.forest.forward(rows).cpu().numpy()          # Forest.forward -> tree_evaluate, one input row per tree
    dump["pareto_fitness"] = algo.pareto_front.fitness.cpu().numpy()
    dump["native"] = np.array(native)
    np.savez(out, **dump)
    print(f"{mode}: {gens} generations of {pop} trees; native libraries: {native}")


if __name__ == "__main__":
    main()
