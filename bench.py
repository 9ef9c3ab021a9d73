#!/usr/bin/env python
"""bench.py — tree-evals/s of the batched fitness evaluation (BASELINE.json metric).

A step = one SR-fitness pass (lower_kernel + replay_kernel) over this rank's population shard
against the whole dataset, plus — for N > 1 — the exchange of the fitness scalars.

Workloads (BASELINE.json `configs`):
  --gpus 1   configs[1]: synthetic SR, 3 inputs, pop 100000, max_tree_len 64, 1024 datapoints
  --gpus N>1 configs[2]: synthetic SR, 10 inputs, pop 1000000 TOTAL (strong scaling: every rank evaluates 1e6 / N
             trees of the replicated population), max_tree_len 64, 1024 datapoints
  (--config 2|3 overrides the choice.)
Extra keys: the config-5 GP loop (100 generations, pop 500000, P*N*G / t_total), config 3 on one GPU (N = 1 line, so
the strong-scaling efficiency can be computed on one workload), achieved GB/s of the HBM-bound genetic kernels.

--impl reference runs the UNMODIFIED reference: its own package installed in baseline/_ref (pip install of
/root/reference; torch ops `evogp_cuda` = its own CUDA kernels) through its public API Forest.SR_fitness — the
reference ships no CPU implementation of this path (torch_wrapper.cu:301-307 registers CUDA only), so its arm is its
CUDA path on ONE B200 (it has no multi-GPU form).  The CPU restatement (oracle/) is timed only as `cpu_baseline`.
See DESIGN.md "Measurement".
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tree-evals/sec (pop x datapoints)"
FUNCS = ["+", "-", "*", "/"]
CONSTS = [-1.0, 0.0, 1.0]
ROTATE = 4            # populations the timed steps rotate over (inputs larger than L2)

WORKLOADS = {
    2: dict(name="configs[1]: synthetic SR, 3 inputs, pop 100000, max_tree_len 64, 1024 datapoints, funcs + - * /",
            pop=100000, L=64, N=1024, V=3, O=1, max_layer_cnt=6, scaling="weak"),
    3: dict(name="configs[2]: synthetic SR, 10 inputs, pop 1000000 total (population-sharded), max_tree_len 64, 1024 datapoints, funcs + - * /",
            pop=1000000, L=64, N=1024, V=10, O=1, max_layer_cnt=6, scaling="strong"),
}
CONFIG5 = dict(pop=500000, L=64, N=1024, V=10, O=1, max_layer_cnt=6, generations=100, mutation_rate=0.2,
               survival_rate=0.3, elite_rate=0.01)


def algorithmic_bytes(P, L, N, V, O):
    # SURVEY.md §8d: node_value + node_type at fixed width, one subtree_size per tree, dataset once, fitness out
    return P * (6 * L + 2) + 4 * N * (V + O) + 4 * P


def make_config(cfg_id, world):
    """The `config` object — identical in both arms (the driver compares them)."""
    w = WORKLOADS[cfg_id]
    per = (w["pop"] + world - 1) // world
    return {"workload": w["name"], "pop_size": w["pop"], "max_tree_len": w["L"], "datapoints": w["N"], "inputs": w["V"],
            "outputs": w["O"], "funcs": FUNCS, "max_layer_cnt": w["max_layer_cnt"], "const_samples": CONSTS,
            "rotating_populations": ROTATE,
            "l2": "inputs rotate over %d populations (%.0f MB of rows + %.0f MB of programs per GPU) > 126 MB L2"
                  % (ROTATE, ROTATE * per * w["L"] * 8 / 1e6, per * (w["L"] + 2) * 8 / 1e6),
            "parallelism": "1 GPU" if world == 1 else
                           "population replicated, evaluation sharded x%d by rows, fitness slices exchanged through peer-mapped symmetric memory" % world}


def target_fn(X):
    # fixed closed-form target (shape of the reference's sr_test.py:17-19, plus a sum over the remaining inputs)
    t = X[:, 0:1] ** 4 / (X[:, 0:1] ** 4 + 1) + X[:, 1:2] ** 4 / (X[:, 1:2] ** 4 + 1)
    if X.shape[1] > 2:
        t = t + 0.1 * X[:, 2:].sum(1, keepdim=True)
    return t


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_facts(cfg_id):
    """DRAM traffic (per tree: it is the program rows the kernel streams) and issue-slot utilisation of the dominant
    kernel, from the committed ncu capture of this workload (profiles/r2_ncu_facts.json <- profiles/r2_eval_config*_ncu.txt)
    — null when there is none."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_facts.json")) as f:
            return json.load(f).get("config%d" % cfg_id)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.active, self.ready = False, threading.Event()   # NVML is initialised before the timed region; samples only inside it

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            self.ready.set()
            while not self.stop_flag:
                if not self.active:
                    time.sleep(0.0002)
                    continue
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
                time.sleep(0.0005)
        except Exception as e:   # NVML missing: report that rather than fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")
            self.ready.set()

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "sampled": "during every timed region of this run (device-timed steps, e2e steps)"}


class StdoutGuard:
    """Keeps stdout to the ONE JSON line: while active, file descriptor 1 points at stderr, so banners that native
    libraries write to stdout (NCCL prints its version there) cannot precede the result; emit() writes to the real one."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        os.write(self.saved, (text + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def dump_outputs(path, **arrays):
    """--dump-outputs: what the last timed step returned, so that the outputs of two builds on the same seeded inputs
    can be compared file for file.  Every file holds finite float32 values: <name>.npy the array with its non-finite
    entries set to 0, <name>_nonfinite.npy which entries those were (0 finite, 1 NaN, 2 +inf, 3 -inf).  A tree that
    divides by zero anywhere has a NaN fitness, as in the reference; with 0 among the constants many trees do."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32)
        kind = np.select([np.isnan(a), a == np.inf, a == -np.inf], [1, 2, 3], 0).astype(np.float32)
        np.save(os.path.join(path, name + ".npy"), np.where(kind == 0, a, np.float32(0)).astype(np.float32))
        np.save(os.path.join(path, name + "_nonfinite.npy"), kind)


def descriptor_args(w, max_layer_cnt=None):
    return dict(max_tree_len=w["L"], input_len=w["V"], output_len=w["O"], using_funcs=FUNCS,
                max_layer_cnt=max_layer_cnt or w["max_layer_cnt"], const_samples=CONSTS)


def keys_for(r, dev):
    import torch
    return torch.tensor([1000 + r, 7], dtype=torch.uint32, device=dev)


def dataset(w, dev):
    import torch
    g = torch.Generator(device="cpu").manual_seed(0)
    X = (torch.rand(w["N"], w["V"], generator=g) * 2 - 1).to(dev).contiguous()
    return X, target_fn(X).contiguous()


# ---------------------------------------------------------------------------------------------------------------
# cpu_baseline: the oracle's C restatement on the host cores (the reference has no CPU path)
# ---------------------------------------------------------------------------------------------------------------
def cpu_baseline_leg(w, reps=5):
    import oracle

    threads = os.cpu_count() or 1        # explicit: OpenMP's default is clamped to 1 under torch.distributed.run
    L, N, V = w["L"], w["N"], w["V"]
    rng = np.random.default_rng(0)
    X = rng.uniform(-1, 1, (N, V)).astype(np.float32)
    import torch
    y = target_fn(torch.from_numpy(X)).numpy().astype(np.float32)
    inner = w["max_layer_cnt"] - 1
    d2l = np.array([0.2] * inner + [1.0] * (10 - inner), np.float32)
    p = np.zeros(29, np.float32); p[1:5] = 0.25
    roul = np.cumsum(p, dtype=np.float32)
    consts = np.array(CONSTS, np.float32)
    P = min(w["pop"], 100000)            # whole population of configs[1]; a 1e5-tree slice of larger ones
    pop = oracle.generate(P, L, V, 1, 0.5, 0.5, np.array([1000, 7], np.uint32), d2l, roul, consts, nthreads=threads)
    oracle.sr_fitness(*pop, X, y, nthreads=threads)      # warm-up (thread pool, page faults)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        oracle.sr_fitness(*pop, X, y, nthreads=threads)
        ts.append(time.perf_counter() - t0)
    med = float(np.median(ts))
    return {"value": P * N / med, "unit": "tree-evals/s", "cores": threads, "kind": "port",
            "sample": "%d of %d trees x %d datapoints per pass, median of %d passes (%.0f ms each); OpenMP over trees, all host threads"
                      % (P, w["pop"], N, reps, med * 1e3),
            "what": "oracle/evogp_oracle.c (C restatement of forward.cu:79-302,375-479); the reference ships no CPU implementation"}


# ---------------------------------------------------------------------------------------------------------------
# the reference arm
# ---------------------------------------------------------------------------------------------------------------
class ReferencePackage:
    """The reference's own python package + torch extension from baseline/_ref (pip install of /root/reference)."""

    def __init__(self):
        path = os.path.join(ROOT, "baseline", "_ref")
        if not os.path.isdir(os.path.join(path, "evogp")):
            raise FileNotFoundError("baseline/_ref/evogp missing (see DESIGN.md: pip install --target baseline/_ref /root/reference)")
        for m in [k for k in sys.modules if k == "evogp" or k.startswith("evogp.")]:
            del sys.modules[m]
        sys.path.insert(0, path)
        import evogp.tree as rt            # loads the reference's evogp_cuda extension
        import evogp.algorithm as ra
        import evogp.problem as rp
        assert os.path.realpath(rt.__file__).startswith(os.path.realpath(path)), "evogp resolved outside baseline/_ref"
        self.rt, self.ra, self.rp = rt, ra, rp
        self.build = "baseline/_ref (pip install of /root/reference, unmodified: its python package + its torch extension evogp_cuda)"

    def forest(self, P, w, keys, max_layer_cnt=None):
        import torch
        d = self.rt.GenerateDescriptor(**descriptor_args(w, max_layer_cnt))
        v, t, s = torch.ops.evogp_cuda.tree_generate(P, d.max_tree_len, d.input_len, d.output_len, d.const_samples.shape[0],
                                                     d.out_prob, d.const_prob, keys, d.depth2leaf_probs, d.roulette_funcs,
                                                     d.const_samples)
        return self.rt.Forest(d.input_len, d.output_len, v, t, s), d

    def wrap(self, w, v, t, s):
        return self.rt.Forest(w["V"], w["O"], v, t, s)

    def sr_fitness(self, forest, X, y):
        return forest.SR_fitness(X, y)     # execute_mode="auto" -> advanced_SR_fitness (forward.cu:514-549,849-851)


class ReferenceKernels:
    """Fallback: the reference's three .cu files compiled unmodified by oracle/build_ref.sh, called through ctypes."""

    def __init__(self):
        import oracle
        if not oracle.ref_gpu_available():
            raise FileNotFoundError("oracle/_ref/libevogp_ref.so missing")
        self.ref = oracle.ref_gpu()
        self.build = "oracle/_ref/libevogp_ref.so (the reference's forward.cu / generate.cu / mutation.cu compiled unmodified with nvcc)"

    class _F:
        def __init__(self, v, t, s):
            self.batch_node_value, self.batch_node_type, self.batch_subtree_size = v, t, s

    def forest(self, P, w, keys, max_layer_cnt=None):
        import torch
        dev = keys.device
        inner = (max_layer_cnt or w["max_layer_cnt"]) - 1
        d2l = torch.tensor([0.2] * inner + [1.0] * (10 - inner), dtype=torch.float32, device=dev)
        p = torch.zeros(29); p[1:5] = 0.25
        roul = torch.cumsum(p, 0).to(dev)
        consts = torch.tensor(CONSTS, dtype=torch.float32, device=dev)
        v, t, s = self.ref.generate(P, w["L"], w["V"], w["O"], 0.5, 0.5, keys, d2l, roul, consts)
        return self._F(v, t, s), None

    def wrap(self, w, v, t, s):
        return self._F(v, t, s)

    def sr_fitness(self, f, X, y):
        return self.ref.sr_fitness(f.batch_node_value, f.batch_node_type, f.batch_subtree_size, X, y)


def run_reference(args, out):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                       # the reference is single-GPU: rank 0 alone runs it
    world = args.gpus
    cfg_id = args.config or (2 if world == 1 else 3)
    w = WORKLOADS[cfg_id]
    import torch
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    why = []
    ref = None
    for cls in (ReferencePackage, ReferenceKernels):
        try:
            ref = cls()
            break
        except Exception as e:
            why.append("%s: %s: %s" % (cls.__name__, type(e).__name__, e))
    if ref is None:
        out.emit(json.dumps({"impl": "reference", "unavailable": "; ".join(why)[:400]}))
        return
    P, L, N, V, O = w["pop"], w["L"], w["N"], w["V"], w["O"]
    X, y = dataset(w, dev)
    pops = [ref.forest(P, w, keys_for(r, dev))[0] for r in range(ROTATE)]
    torch.cuda.synchronize()
    sampler = ClockSampler(0); sampler.start(); sampler.ready.wait(timeout=10)

    def step(i):
        return ref.sr_fitness(pops[i % ROTATE], X, y)

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active = True
    e0.record()
    for i in range(args.steps):
        fit = step(i)
    e1.record()
    torch.cuda.synchronize()
    sampler.active = False
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, fitness=fit.cpu().numpy())
    total_ms = e0.elapsed_time(e1)
    value = P * N * args.steps / (total_ms * 1e-3)
    check = float(torch.nan_to_num(fit, nan=0.0, posinf=0.0, neginf=0.0).clamp(max=1e6).mean())

    # ---- e2e: host buffers -> device -> Forest.SR_fitness -> host, every step ----
    R2 = 2
    host = [tuple(a.cpu().pin_memory() for a in (p.batch_node_value, p.batch_node_type, p.batch_subtree_size)) for p in pops[:R2]]
    hX, hy = X.cpu().pin_memory(), y.cpu().pin_memory()

    def e2e_step(i):
        hv, ht, hs = host[i % R2]
        f = ref.wrap(w, hv.to(dev, non_blocking=True), ht.to(dev, non_blocking=True), hs.to(dev, non_blocking=True))
        return ref.sr_fitness(f, hX.to(dev, non_blocking=True), hy.to(dev, non_blocking=True)).cpu()

    for i in range(max(2, min(args.warmup, 5))):
        e2e_step(i)
    torch.cuda.synchronize()
    sampler.active = True
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    sampler.active = False
    e2e_value = P * N * args.steps / e2e_s

    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "tree-evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": w["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(cfg_id, world),
            "cpu_baseline": {"value": value, "unit": "tree-evals/s", "cores": 1, "kind": "reference",
                             "sample": "whole population (%d trees x %d datapoints) per step" % (P, N),
                             "what": "the reference ships NO CPU implementation of this path (torch_wrapper.cu:301-307 registers "
                                     "CUDA only): this is its own CUDA path, Forest.SR_fitness(execute_mode='auto'), on ONE B200 "
                                     "(it has no multi-GPU form), one host thread driving it"},
            "e2e": {"value": e2e_value, "unit": "tree-evals/s", "h2d_bytes_per_step": P * L * 8 + N * (V + O) * 4,
                    "d2h_bytes_per_step": P * 4,
                    "path": "pinned host arrays -> .to(cuda) -> reference Forest.SR_fitness -> .cpu(), every step"},
            "reference_build": ref.build, "gpus_used": 1, "fitness_mean_check": check, "clocks": sampler.summary()}
    if not args.quick and isinstance(ref, ReferencePackage):
        try:
            line["config5_loop"] = reference_config5_loop(ref, dev)
        except Exception as e:
            line["config5_loop"] = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
    sampler.stop_flag = True
    out.emit(json.dumps(line))


def reference_config5_loop(ref, dev, generations=10, warm=2):
    """The reference's own GP loop (its GeneticProgramming + default operators + SymbolicRegression) on one GPU."""
    import torch
    c = CONFIG5
    torch.manual_seed(1)
    X, y = dataset(c, dev)
    forest, d = ref.forest(c["pop"], c, keys_for(99, dev))
    ra, rp = ref.ra, ref.rp
    algo = ra.GeneticProgramming(initial_forest=forest, crossover=ra.DefaultCrossover(),
                                 mutation=ra.DefaultMutation(mutation_rate=c["mutation_rate"], descriptor=d.update(max_layer_cnt=3)),
                                 selection=ra.DefaultSelection(survival_rate=c["survival_rate"], elite_rate=c["elite_rate"]))
    prob = rp.SymbolicRegression(datapoints=X, labels=y)

    def one():
        fit = prob.evaluate(algo.forest)
        fit = torch.where(torch.isnan(fit), torch.full_like(fit, float("-inf")), fit)
        algo.step(fit)

    for _ in range(warm):
        one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(generations):
        one()
    torch.cuda.synchronize()
    t = time.perf_counter() - t0
    return {"value": c["pop"] * c["N"] * generations / t, "unit": "tree-evals/s (P*N*G / t_total)", "generations": generations,
            "ms_per_generation": t / generations * 1e3, "gpus_used": 1,
            "mean_tree_len_after": float(algo.forest.batch_subtree_size[:, 0].float().mean()),
            "what": "reference GeneticProgramming(DefaultSelection 0.3/0.01, DefaultCrossover, DefaultMutation 0.2) + SymbolicRegression, "
                    "pop 500000, generations %d..%d of a run (trees bloat with the generations: early ones are the cheap ones)" % (warm, warm + generations)}


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def contiguous_forest(Forest, f, lo, hi):
    return Forest(f.input_len, f.output_len, f.batch_node_value[lo:hi].contiguous(), f.batch_node_type[lo:hi].contiguous(),
                  f.batch_subtree_size[lo:hi].contiguous())


def hbm_kernel_report(dev, peak):
    """Achieved GB/s of the HBM-bound genetic kernels at config-5 sizes (rank 0, N = 1 line): CUDA events around
    `reps` back-to-back launches on rotating outputs.  `moved` = bytes the kernel actually reads + writes (full-width
    zero-filled rows are written); `algorithmic` = SURVEY.md §8d (valid prefixes only)."""
    import torch
    from evogp_b200.tree import Forest, GenerateDescriptor
    _ops = torch.ops.evogp_cuda
    c = CONFIG5
    L = c["L"]
    d = GenerateDescriptor(**descriptor_args(c))
    dm = d.update(max_layer_cnt=3)
    rep = {}

    def timed(fn, reps=20, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e-3

    def entry(name, t, moved, algo, what):
        rep[name] = {"us": t * 1e6, "moved_GBps": moved / t / 1e9, "moved_frac_of_hbm_peak": moved / t / 1e9 / peak,
                     "algorithmic_GBps": algo / t / 1e9, "algorithmic_frac_of_hbm_peak": algo / t / 1e9 / peak, "what": what}

    # generate: a fresh population (config 2 size) and a batch of mutation donors (config 5: 0.2 * 495000)
    for name, P, desc in (("generate_pop100000", 100000, d), ("generate_donors99000", 99000, dm)):
        keys = keys_for(5, dev)
        f = Forest.generate_with_keys(P, desc, keys)
        nodes = float(f.batch_subtree_size[:, 0].float().sum())
        t = timed(lambda: Forest.generate_with_keys(P, desc, keys))
        entry(name, t, P * L * 8, nodes * 8, "evogp_generate: %d trees, mean length %.1f; writes %d full rows" % (P, nodes / P, P))
    # crossover: 150000 survivors -> 495000 children
    pop = Forest.generate_with_keys(c["pop"], d, keys_for(6, dev))
    surv = contiguous_forest(Forest, pop, 0, 150000)
    n_new = 495000
    g = torch.Generator(device=dev).manual_seed(3)
    li = torch.randint(0, 150000, (n_new,), dtype=torch.int32, device=dev, generator=g)
    ri = torch.randint(0, 150000, (n_new,), dtype=torch.int32, device=dev, generator=g)
    sizes = surv.batch_subtree_size[:, 0].int()
    lp = torch.randint(0, 2**31 - 1, (n_new,), dtype=torch.int32, device=dev, generator=g) % sizes[li.long()]
    rp = torch.randint(0, 2**31 - 1, (n_new,), dtype=torch.int32, device=dev, generator=g) % sizes[ri.long()]
    child = surv.crossover(li, ri, lp, rp)
    clen = float(child.batch_subtree_size[:, 0].float().sum())
    t = timed(lambda: surv.crossover(li, ri, lp, rp))
    entry("crossover_150000_to_495000", t, clen * 8 + n_new * L * 8 + 16 * n_new, 2 * clen * 8 + 16 * n_new,
          "evogp_crossover: reads the spans that form the child (~child length), writes 495000 full rows")
    # mutate: 99000 mutants with whole-tree donors
    Pm = 99000
    mutants = contiguous_forest(Forest, child, 0, Pm)
    donors = Forest.generate_with_keys(Pm, dm, keys_for(7, dev))
    pos = torch.randint(0, 1024, (Pm,), dtype=torch.int32, device=dev, generator=g) % mutants.batch_subtree_size[:, 0].int()
    res = mutants.mutate(pos, donors)
    rlen = float(res.batch_subtree_size[:, 0].float().sum())
    t = timed(lambda: mutants.mutate(pos, donors))
    entry("mutate_99000", t, rlen * 8 + Pm * L * 8 + 4 * Pm, 2 * rlen * 8 + 4 * Pm, "evogp_mutate: 99000 rows, donors of <= 7 nodes")
    # the fused generation step at pop 500000
    fit = torch.rand(c["pop"], device=dev, generator=g)
    order = torch.sort(fit, descending=True, stable=True).indices
    elite, survivors = int(c["pop"] * c["elite_rate"]), int(c["pop"] * c["survival_rate"])
    keys = keys_for(8, dev)

    def nextgen():
        return _ops.tree_next_generation(c["pop"], L, pop.batch_node_value, pop.batch_node_type, pop.batch_subtree_size, order,
                                         elite, survivors, c["mutation_rate"], c["V"], c["O"], dm.out_prob, dm.const_prob,
                                         dm.depth2leaf_probs, dm.roulette_funcs, dm.const_samples, keys)
    nv, nt, ns = nextgen()
    nlen = float(ns[:, 0].float().sum())
    t = timed(nextgen)
    entry("nextgen_pop500000", t, nlen * 8 + c["pop"] * L * 8 + 8 * c["pop"], 2 * nlen * 8 + 8 * c["pop"],
          "evogp_next_generation: elitism + crossover + mutation of a whole generation in one kernel")
    return rep


def config5_loop(dev, world, rank, exch_cls):
    """BASELINE configs[4]: full GP loop, 100 generations, pop 500000, mutation_rate 0.2: every rank evaluates its row
    shard (fitness exchange over peer memory), then runs the identical fused generation step on the replicated
    population.  Value = P * N * G / t_total (max over ranks)."""
    import torch
    import torch.distributed as dist
    from evogp_b200.algorithm import FusedGeneticProgramming
    from evogp_b200.parallel import shard_bounds
    from evogp_b200.tree import Forest, GenerateDescriptor

    c = CONFIG5
    P, G = c["pop"], c["generations"]
    X, y = dataset(c, dev)
    d = GenerateDescriptor(**descriptor_args(c))
    forest = Forest.generate_with_keys(P, d, keys_for(99, dev))
    algo = FusedGeneticProgramming(forest, d.update(max_layer_cnt=3), c["mutation_rate"], c["survival_rate"], elite_rate=c["elite_rate"])
    lo, hi, _ = shard_bounds(P, world, rank)
    exch = exch_cls(P, dev) if world > 1 else None
    gen_keys = torch.stack([keys_for(200 + g, dev) for g in range(G + 3)])

    def one(g):
        f = algo.forest
        if exch is not None:
            fit = exch.sr_fitness(contiguous_forest(Forest, f, lo, hi), X, y)
        else:
            fit = f.SR_fitness(X, y)
        algo.step(-fit, keys=gen_keys[g])

    for g in range(3):
        one(g)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for g in range(G):
        one(3 + g)
    e1.record()
    torch.cuda.synchronize()
    tms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    digest = algo.forest.batch_subtree_size[:, 0].long().sum().reshape(1)
    same = True
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        got = [torch.empty_like(digest) for _ in range(world)]
        dist.all_gather(got, digest)
        same = all(bool(torch.equal(a, got[0])) for a in got)
    t = float(tms) * 1e-3
    return {"value": P * c["N"] * G / t, "unit": "tree-evals/s (P*N*G / t_total)", "generations": G, "ms_per_generation": t / G * 1e3,
            "n_gpus": world, "mean_tree_len_after": float(algo.forest.batch_subtree_size[:, 0].float().mean()),
            "populations_identical_on_all_ranks": same,
            "what": "pop 500000, V 10, mutation_rate 0.2, selection 0.3 / elite 0.01: sharded evaluation (fitness exchange over peer memory) + "
                    "evogp_next_generation (one kernel) + torch.sort per generation; device-timed, max over ranks"}


def run_ours(args, out):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from evogp_b200 import _native
    from evogp_b200.parallel import FitnessExchange, shard_bounds
    from evogp_b200.tree import Forest, GenerateDescriptor

    dev = torch.device("cuda", local)
    cfg_id = args.config or (2 if world == 1 else 3)
    w = WORKLOADS[cfg_id]
    P_total, L, N, V, O = w["pop"], w["L"], w["N"], w["V"], w["O"]
    X, y = dataset(w, dev)
    desc = GenerateDescriptor(**descriptor_args(w))
    lo, hi, _ = shard_bounds(P_total, world, rank)
    pops, fulls = [], []
    for r in range(ROTATE):
        full = Forest.generate_with_keys(P_total, desc, keys_for(r, dev))   # replicated population; this rank evaluates [lo, hi)
        pops.append(contiguous_forest(Forest, full, lo, hi) if world > 1 else full)
        if world > 1 and r < 2:
            fulls.append(full)              # kept for the exchange check below
        del full
    torch.cuda.synchronize()
    mean_len = float(torch.stack([p.batch_subtree_size[:, 0].float().mean() for p in pops]).mean())

    exch = FitnessExchange(P_total, dev) if world > 1 else None
    exchange_kind = ("none (1 GPU)" if world == 1 else
                     ({"push": "evaluation kernel, then evogp_push_fitness: coalesced stores into every rank's buffer over peer-mapped symmetric memory, then one inter-GPU barrier",
                       "fused": "fused into the evaluation kernel (evogp_SR_fitness_scatter) over peer-mapped symmetric memory"}.get(exch.mode, exch.mode)
                      if exch.available else "NCCL all_gather (symmetric memory unavailable: %s)" % exch.why))

    def step(i):
        if exch is not None:
            return exch.sr_fitness(pops[i % ROTATE], X, y)
        return pops[i % ROTATE].SR_fitness(X, y)

    abi = _native.abi()
    sampler = ClockSampler(local); sampler.start()
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    sampler.ready.wait(timeout=10)

    # ---- N > 1: the exchanged fitness is what a single-GPU evaluation of the whole population gives (bit for bit),
    #      on both alternating buffers, on every rank — outside the timed region ----
    exchange_check = None
    if world > 1:
        ok = True
        for r in range(2):
            got = exch.sr_fitness(pops[r], X, y).clone()
            want = fulls[r].SR_fitness(X, y)
            ok = ok and bool(torch.equal(got.view(torch.int32), want.view(torch.int32)))
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        exchange_check = {"bit_equal_to_single_gpu_evaluation": bool(flag.item()), "ranks_checked": world, "buffers_checked": 2,
                          "what": "every rank compares its exchanged full-population fitness with its own evaluation of all %d trees" % P_total}
        del fulls
        assert exchange_check["bit_equal_to_single_gpu_evaluation"], "fitness exchange delivered wrong values"
        dist.barrier()

    # ---- device-timed steps ----
    launches0 = _native.launch_count()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in kev:
        a.record(); b.record()     # materialise the handles
    ev_t0 = torch.cuda.Event(enable_timing=True); ev_t1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    sampler.active = True
    ev_t0.record()
    for i in range(args.steps):
        abi.evogp_eval_set_timing_events(ctypes.c_void_p(kev[i][0].cuda_event), ctypes.c_void_p(kev[i][1].cuda_event))
        fit = step(i)
    ev_t1.record()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    sampler.active = False
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fitness=fit.cpu().numpy())     # N > 1: the exchanged fitness of the whole population
    abi.evogp_eval_set_timing_events(None, None)
    kern_ms = [a.elapsed_time(b) for a, b in kev]
    launches = _native.launch_count() - launches0
    total_ms = torch.tensor([ev_t0.elapsed_time(ev_t1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.barrier()
    total_s = float(total_ms) / 1e3
    value = P_total * N * args.steps / total_s

    # ---- e2e: host buffers through the C ABI (H2D of the forest + dataset, D2H of fitness, every step) ----
    R2 = 2
    hv = [p.batch_node_value.cpu().pin_memory() for p in pops[:R2]]
    ht = [p.batch_node_type.cpu().pin_memory() for p in pops[:R2]]
    hs = [p.batch_subtree_size.cpu().pin_memory() for p in pops[:R2]]
    hX, hy = X.cpu().pin_memory(), y.cpu().pin_memory()
    hfit = torch.empty(hi - lo, dtype=torch.float32).pin_memory()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())

    def e2e_step(i):
        r = i % R2
        rc = abi.evogp_SR_fitness_host(hi - lo, N, L, V, O, 1, vp(hv[r]), vp(ht[r]), vp(hs[r]), vp(hX), vp(hy), vp(hfit), local)
        _native.check(rc, "evogp_SR_fitness_host")

    for i in range(max(2, min(args.warmup, 5))):
        e2e_step(i)
    if world > 1:
        dist.barrier()
    sampler.active = True
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    e2e_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    sampler.active = False
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = P_total * N * args.steps / float(e2e_t)
    # what evogp_SR_fitness_host actually uploads: valid prefixes of node_value + node_type (6 B per node), one 32-bit
    # offset per tree, the dataset
    nodes = int(sum(int(p.batch_subtree_size[:, 0].long().sum()) for p in pops[:R2]) // R2)
    h2d = nodes * 6 + (hi - lo + 9) * 4 + N * (V + O) * 4
    d2h = (hi - lo) * 4
    fit_host_check = float(np.nanmean(np.clip(np.nan_to_num(hfit.numpy(), nan=0.0, posinf=0.0, neginf=0.0), None, 1e6)))
    del hv, ht, hs

    # ---- extra legs (outside every timed region above) ----
    extras = {}
    if not args.quick:
        extras["config5_loop"] = config5_loop(dev, world, rank, FitnessExchange)
        if world == 1 and cfg_id == 2:
            w3 = WORKLOADS[3]
            X3, y3 = dataset(w3, dev)
            d3 = GenerateDescriptor(**descriptor_args(w3))
            f3 = [Forest.generate_with_keys(w3["pop"], d3, keys_for(r, dev)) for r in range(2)]
            for i in range(3):
                f3[i % 2].SR_fitness(X3, y3)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            a.record()
            for i in range(reps):
                f3[i % 2].SR_fitness(X3, y3)
            b.record(); torch.cuda.synchronize()
            ms3 = a.elapsed_time(b) / reps
            extras["config3_single_gpu"] = {"value": w3["pop"] * w3["N"] / (ms3 * 1e-3), "unit": "tree-evals/s", "ms_per_step": ms3,
                                            "what": "configs[2] (pop 1000000, V 10) evaluated whole on ONE GPU: the N = 1 point of the "
                                                    "strong-scaling series that --gpus 2/4/8 run"}
            del f3

    line = None
    if rank == 0:
        peak, peak_src = measured_peak()
        kms = float(np.mean(kern_ms))
        ms_step = total_s * 1e3 / args.steps
        ach = algorithmic_bytes(hi - lo, L, N, V, O) / (kms * 1e-3) / 1e9
        facts = ncu_facts(cfg_id) or {}
        line = {"metric": METRIC, "value": value, "unit": "tree-evals/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": w["scaling"],
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": make_config(cfg_id, world),
                "e2e": {"value": e2e_value, "unit": "tree-evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "path": "evogp_SR_fitness_host (C ABI, pinned host buffers: valid prefixes packed by a host thread pool, chunked copy/compute overlap), every rank on its shard"},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "kernel": "replay_kernel", "achieved": ach, "peak": peak,
                             "unit": "GB/s", "frac": ach / peak,
                             "traffic": (facts["replay_dram_bytes_per_tree"] * (hi - lo)) if "replay_dram_bytes_per_tree" in facts else None,
                             "traffic_source": facts.get("source"),
                             "algorithmic_bytes": algorithmic_bytes(hi - lo, L, N, V, O), "peak_source": peak_src,
                             "kernel_ms": kms, "kernel_share_of_step": kms / ms_step,
                             "issue_slots_busy_pct": facts.get("replay_issue_slots_busy_pct"),
                             "note": "interpreter kernel: bound by instruction issue, not HBM (DESIGN.md 3.2); kernel_ms is measured "
                                     "live (CUDA events recorded around the replay launch inside the C ABI)"},
                "mean_tree_len": round(mean_len, 2), "fitness_exchange": exchange_kind,
                "wall_s_timed_region": t_wall, "fitness_mean_check": fit_host_check}
        if exchange_check is not None:
            line["exchange_check"] = exchange_check
        line.update(extras)
        if world == 1 and not args.quick:
            line["hbm_kernels"] = hbm_kernel_report(dev, peak)
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline_leg(w)
        line["clocks"] = sampler.summary()
        out.emit(json.dumps(line))
    sampler.stop_flag = True
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=0, choices=[0, 2, 3], help="0: configs[1] at --gpus 1, configs[2] strong-scaled otherwise")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--quick", action="store_true", help="skip the extra legs (config-5 loop, HBM kernels, config 3 on one GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the fitness the last timed step computed to DIR/fitness.npy (finite values) and DIR/fitness_nonfinite.npy (which were NaN / inf)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    with StdoutGuard() as out:
        if args.impl == "reference":
            run_reference(args, out)
        else:
            run_ours(args, out)


if __name__ == "__main__":
    main()
