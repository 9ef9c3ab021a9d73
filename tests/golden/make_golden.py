#!/usr/bin/env python
"""Regenerates the reference's results stored under tests/golden/.  The reference's own code is built by
__graft_entry__.build() where its sources are present (oracle/build_ref.sh -> oracle/_ref/, its python package ->
baseline/_ref/); copy the .npz files this writes into tests/golden/.

    python tests/golden/make_golden.py kernels OUTDIR   ref_{arith,allfuncs,multi}.npz: its CUDA kernels on a GPU
    python tests/golden/make_golden.py parity OUTDIR    ref_parity.npz: every reference call of tests/test_gpu_parity.py
    python tests/golden/make_golden.py dropin OUTDIR    ref_dropin.npz: its python front-end over its own extension
    python tests/golden/make_golden.py rng OUTDIR       ref_rng.npz: its hash() and taus88 draws, on the host

Inputs are seeded numpy / fixed keys, so the files are reproducible.  The reference leaves row tails undefined;
buffers are pre-zeroed here so the files are deterministic (consumers compare valid prefixes only)."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle  # noqa: E402
from conftest import ALL_FUNCS, ARITH_FUNCS, depth2leaf, make_data, roulette  # noqa: E402


def dev(*arrs):
    out = tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs)
    return out if len(out) > 1 else out[0]


def kernels(outdir):
    ref = oracle.ref_gpu()
    cases = {
        "arith": dict(pop=512, L=32, V=3, O=1, funcs=ARITH_FUNCS, layers=5, keys=(42, 0), consts=(-1.0, 0.0, 1.0), N=200),
        "allfuncs": dict(pop=384, L=64, V=4, O=1, funcs=ALL_FUNCS, layers=4, keys=(7, 9), consts=(-1.0, 0.5, 2.0), N=64),
        "multi": dict(pop=384, L=64, V=5, O=3, funcs=ALL_FUNCS, layers=4, keys=(123456, 654321), consts=(-1.0, 0.5, 2.0), N=33),
    }
    for name, c in cases.items():
        d2l, roul, consts = depth2leaf(c["layers"]), roulette(c["funcs"]), np.array(c["consts"], np.float32)
        keys = np.array(c["keys"], np.uint32)
        v, t, s = ref.generate(c["pop"], c["L"], c["V"], c["O"], 0.5, 0.5, *dev(keys, d2l, roul, consts))
        torch.cuda.synchronize()
        ev_v, ev_t, ev_s = v, t, s
        X, y = make_data(c["N"], c["V"], c["O"], seed=11)
        dX, dy = dev(X, y)
        fit_mse = ref.sr_fitness(v, t, s, dX, dy, True, 4)
        fit_abs = ref.sr_fitness(v, t, s, dX, dy, False, 4)
        fit_mode0 = ref.sr_fitness(v, t, s, dX, dy, True, 0)
        rng = np.random.default_rng(5)
        Xrow = rng.uniform(-2, 2, (c["pop"], c["V"])).astype(np.float32)
        ev = ref.evaluate(v, t, s, dev(Xrow), c["O"])
        # splice fixtures use a forest WITHOUT ternary nodes: the reference's _gpTreeReplace reads an
        # uninitialised stack slot when the splice point is the middle child of an IF (mutation.cu:69-73),
        # which is undefined behaviour (observed: illegal memory access on B200), so it cannot define a golden
        no_if = [f for f in c["funcs"] if f != "if"]
        if no_if != list(c["funcs"]):
            v, t, s = ref.generate(c["pop"], c["L"], c["V"], c["O"], 0.5, 0.5, *dev(np.array([77, 78], np.uint32), d2l, roulette(no_if), consts))
            roul = roulette(no_if)
        sp_v, sp_t, sp_s = v, t, s
        lens = s[:, 0].cpu().numpy().astype(np.int64)
        n_new = 700
        li = rng.integers(0, c["pop"], n_new).astype(np.int32)
        ri = rng.integers(0, c["pop"], n_new).astype(np.int32)
        lp = (rng.integers(0, 1 << 30, n_new) % lens[li]).astype(np.int32)
        rp = (rng.integers(0, 1 << 30, n_new) % lens[ri]).astype(np.int32)
        ri[:8] = -1
        ri[8:16] = c["pop"]
        cv, ct, cs = ref.crossover(v, t, s, *dev(li, ri, lp, rp))
        # mutation donors: small trees from the same generator
        nv, nt, ns = ref.generate(c["pop"], c["L"], c["V"], c["O"], 0.5, 0.5, *dev(np.array([5, 6], np.uint32), depth2leaf(3), roul, consts))
        pos = (rng.integers(0, 1024, c["pop"]) % lens).astype(np.int32)
        pos[:4] = -1
        pos[4:8] = lens[4:8]
        mv, mt, ms = ref.mutate(v, t, s, dev(pos), nv, nt, ns)
        torch.cuda.synchronize()
        g = lambda a: a.cpu().numpy()
        np.savez_compressed(os.path.join(outdir, f"ref_{name}.npz"),
                            keys=keys, d2l=d2l, roul=roulette(c["funcs"]), consts=consts, V=c["V"], O=c["O"],
                            value=g(ev_v), type=g(ev_t), size=g(ev_s), sp_value=g(sp_v), sp_type=g(sp_t), sp_size=g(sp_s), X=X, y=y, fit_mse=g(fit_mse), fit_abs=g(fit_abs),
                            fit_mode0=g(fit_mode0), Xrow=Xrow, evaluate=g(ev), li=li, ri=ri, lp=lp, rp=rp,
                            cx_value=g(cv), cx_type=g(ct), cx_size=g(cs), donor_value=g(nv), donor_type=g(nt),
                            donor_size=g(ns), mut_pos=pos, mut_value=g(mv), mut_type=g(mt), mut_size=g(ms))
        print(name, "ok", float(np.nanmean(g(fit_mse)[np.isfinite(g(fit_mse))])))


def parity(outdir):
    env = dict(os.environ, EVOGP_RECORD_REFERENCE=os.path.abspath(os.path.join(outdir, "ref_parity.npz")))
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-m", "gpu", os.path.join(ROOT, "tests", "test_gpu_parity.py")],
                          cwd=ROOT, env=env)


def dropin(outdir):
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tests", "dropin_run.py"), "reference",
                           os.path.abspath(os.path.join(outdir, "ref_dropin.npz"))], cwd=outdir)


def rng(outdir):
    import ctypes as C

    shim = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_shim.so"))
    shim.ref_hash.restype = C.c_uint32
    shim.ref_hash.argtypes = [C.c_uint32] * 3
    hash_args = np.random.default_rng(1).integers(0, 2**32, size=(200, 3), dtype=np.uint64).astype(np.uint32)
    hashes = np.array([shim.ref_hash(int(n), int(k1), int(k2)) for n, k1, k2 in hash_args], np.uint32)
    seeds = np.array([0, 1, 341, 746587583, 0xFFFFFFFF, 123456789], np.uint32)
    draws = np.zeros((len(seeds), 64), np.uint32)
    uniforms = np.zeros((len(seeds), 64), np.float32)
    for i, seed in enumerate(seeds):
        shim.ref_engine_draws(C.c_uint32(int(seed)), 64, draws[i].ctypes.data_as(C.c_void_p))
        shim.ref_engine_uniforms(C.c_uint32(int(seed)), 64, uniforms[i].ctypes.data_as(C.c_void_p))
    np.savez_compressed(os.path.join(outdir, "ref_rng.npz"), hash_args=hash_args, hash=hashes, seeds=seeds, draws=draws,
                        uniforms=uniforms)


if __name__ == "__main__":
    what, outdir = sys.argv[1], sys.argv[2]
    os.makedirs(outdir, exist_ok=True)
    {"kernels": kernels, "parity": parity, "dropin": dropin, "rng": rng}[what](outdir)
