"""Helpers for the -m gpu tests: call the C ABI (include/evogp_b200.h) through ctypes with torch
device pointers, move oracle/numpy data to the GPU, and replay the reference's recorded results."""
import ctypes as C
import hashlib

import numpy as np
import torch


def dev():
    return torch.device("cuda", torch.cuda.current_device())


def to_dev(*arrs):
    out = tuple(torch.from_numpy(np.ascontiguousarray(a)).to(dev()) for a in arrs)
    return out if len(out) > 1 else out[0]


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ws(native, P, L):
    n = native.abi().evogp_eval_workspace_bytes(P, L)
    return torch.empty(n, dtype=torch.uint8, device=dev()), n


def abi_sr_fitness(native, v, t, s, X, y, use_mse=True):
    P, L = v.shape
    N, V = X.shape
    O = y.shape[1]
    fit = torch.empty(P, dtype=torch.float32, device=v.device)
    ws, n = _ws(native, P, L)
    rc = native.abi().evogp_SR_fitness(P, N, L, V, O, int(use_mse), _p(v), _p(t), _p(s), _p(X), _p(y), _p(fit), 4,
                                       _p(ws), n, _stream())
    native.check(rc, "evogp_SR_fitness")
    return fit


def abi_evaluate(native, v, t, s, X, O):
    P, L = v.shape
    V = X.shape[1]
    res = torch.empty((P, O), dtype=torch.float32, device=v.device)
    ws, n = _ws(native, P, L)
    native.check(native.abi().evogp_evaluate(P, L, V, O, _p(v), _p(t), _p(s), _p(X), _p(res), _p(ws), n, _stream()),
                 "evogp_evaluate")
    return res


def abi_batch_forward(native, v, t, s, X, O):
    P, L = v.shape
    N, V = X.shape
    res = torch.empty((P, N, O), dtype=torch.float32, device=v.device)
    ws, n = _ws(native, P, L)
    native.check(native.abi().evogp_batch_forward(P, N, L, V, O, _p(v), _p(t), _p(s), _p(X), _p(res), _p(ws), n,
                                                  _stream()), "evogp_batch_forward")
    return res


def abi_generate(native, pop, L, V, O, out_prob, const_prob, keys, d2l, roul, consts):
    v = torch.empty((pop, L), dtype=torch.float32, device=dev())
    t = torch.empty((pop, L), dtype=torch.int16, device=dev())
    s = torch.empty((pop, L), dtype=torch.int16, device=dev())
    rc = native.abi().evogp_generate(pop, L, V, O, consts.shape[0], out_prob, const_prob, _p(keys), _p(d2l), _p(roul),
                                     _p(consts), _p(v), _p(t), _p(s), _stream())
    native.check(rc, "evogp_generate")
    return v, t, s


def abi_crossover(native, v, t, s, li, ri, lp, rp):
    P, L = v.shape
    Pn = li.shape[0]
    ov = torch.empty((Pn, L), dtype=torch.float32, device=v.device)
    ot = torch.empty((Pn, L), dtype=torch.int16, device=v.device)
    os_ = torch.empty((Pn, L), dtype=torch.int16, device=v.device)
    rc = native.abi().evogp_crossover(P, Pn, L, _p(v), _p(t), _p(s), _p(li), _p(ri), _p(lp), _p(rp), _p(ov), _p(ot),
                                      _p(os_), _stream())
    native.check(rc, "evogp_crossover")
    return ov, ot, os_


def abi_mutate(native, v, t, s, pos, nv, nt, ns):
    P, L = v.shape
    ov, ot, os_ = torch.empty_like(v), torch.empty_like(t), torch.empty_like(s)
    rc = native.abi().evogp_mutate(P, L, _p(v), _p(t), _p(s), _p(pos), _p(nv), _p(nt), _p(ns), _p(ov), _p(ot),
                                   _p(os_), _stream())
    native.check(rc, "evogp_mutate")
    return ov, ot, os_


def same_bits(a, b):
    a, b = a.cpu().numpy(), b if isinstance(b, np.ndarray) else b.cpu().numpy()
    if a.dtype.kind == "f":
        return np.array_equal(a.view(np.uint32), b.view(np.uint32))
    return np.array_equal(a, b)


def assert_close_fitness(got, want, rtol=1e-5, atol=0.0, what=""):
    """NaN == NaN, +-inf == +-inf, otherwise relative tolerance (north star: 1e-5 on fp32 fitness)."""
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    want = want.cpu().numpy() if hasattr(want, "cpu") else np.asarray(want)
    assert got.shape == want.shape
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), f"{what}: NaN pattern differs at {np.nonzero(gn != wn)[0][:10]}"
    gi, wi = np.isinf(got), np.isinf(want)
    assert np.array_equal(gi, wi) and np.array_equal(got[gi], want[wi]), f"{what}: inf pattern differs"
    m = ~(gn | gi)
    err = np.abs(got[m].astype(np.float64) - want[m]) - atol
    tol = rtol * np.abs(want[m].astype(np.float64))
    bad = err > tol
    assert not bad.any(), (f"{what}: {bad.sum()} of {m.sum()} beyond rtol={rtol}; worst rel "
                           f"{(err[bad] / np.maximum(np.abs(want[m][bad]), 1e-30)).max():.3e}")


def _host(a):
    return np.ascontiguousarray(a.cpu().numpy() if isinstance(a, torch.Tensor) else a)


def prefix_digest(v, t, s):
    """SHA-256 of a forest's valid prefixes (row tails zeroed, each row's length from its own size[:, 0]): two forests
    have the same digest when their prefixes agree bit for bit."""
    v, t, s = _host(v), _host(t), _host(s)
    L = v.shape[1]
    valid = np.arange(L)[None, :] < np.clip(s[:, 0].astype(np.int64), 0, L)[:, None]
    h = hashlib.sha256()
    for a in (v.view(np.uint32), t, s):
        h.update(np.where(valid, a, 0).astype(a.dtype).tobytes())
    return h.hexdigest()


def call_key(op, *args):
    """Digest of an operator name and its inputs (arrays by dtype, shape and bytes; scalars by value)."""
    h = hashlib.sha256(op.encode())
    for a in args:
        if isinstance(a, (torch.Tensor, np.ndarray)):
            a = _host(a)
            h.update(f"{a.dtype.str}{a.shape}".encode())
            h.update(a.tobytes())
        else:
            h.update(repr(a).encode())
    return h.hexdigest()


class GoldenReference:
    """The reference's own CUDA kernels (forward.cu / generate.cu / mutation.cu compiled unmodified), replayed from
    results recorded on a B200 (tests/golden/make_golden.py parity).  Each result is stored under call_key of its
    inputs, so a test whose inputs changed finds no result rather than a wrong one.  Fitness and evaluation results
    are stored as values; the tree producers, whose outputs are too large to store, as prefix_digest of their output."""

    def __init__(self, path):
        with np.load(path) as f:
            self.results = {k: f[k] for k in f.files}

    def _get(self, *call):
        key = call_key(*call)
        assert key in self.results, f"no recorded reference result for these {call[0]} inputs (key {key[:16]})"
        r = self.results[key]
        return str(r) if r.dtype.kind == "U" else r

    def generate(self, pop, gp_len, var_len, out_len, out_prob, const_prob, keys, depth2leaf, roulette, const_samples):
        return self._get("generate", pop, gp_len, var_len, out_len, out_prob, const_prob, keys, depth2leaf, roulette, const_samples)

    def crossover(self, value, ntype, size, left_idx, right_idx, left_node, right_node):
        return self._get("crossover", value, ntype, size, left_idx, right_idx, left_node, right_node)

    def mutate(self, value, ntype, size, mut_idx, nvalue, ntype_new, nsize):
        return self._get("mutate", value, ntype, size, mut_idx, nvalue, ntype_new, nsize)

    def sr_fitness(self, value, ntype, size, variables, labels, use_mse=True, kernel_type=4):
        return self._get("sr_fitness", value, ntype, size, variables, labels, bool(use_mse), kernel_type)

    def evaluate(self, value, ntype, size, variables, out_len):
        return self._get("evaluate", value, ntype, size, variables, out_len)


class RecordingReference(GoldenReference):
    """Runs the reference's kernels (oracle.ref_gpu()) and records what GoldenReference replays."""

    def __init__(self, live):
        self.live, self.results = live, {}

    def _get(self, op, *args):
        out = getattr(self.live, op)(*args)
        torch.cuda.synchronize()
        r = np.array(prefix_digest(*out)) if isinstance(out, tuple) else out.cpu().numpy()
        self.results[call_key(op, *args)] = r
        return str(r) if r.dtype.kind == "U" else r

    def save(self, path):
        np.savez_compressed(path, **self.results)
