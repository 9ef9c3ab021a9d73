"""-m gpu: parity of the sm_100a kernels, called through the C ABI, against
  (a) the CPU oracle (oracle/evogp_oracle.c) — bit-exact for integer/index work,
  (b) the reference's own CUDA kernels compiled unmodified, as recorded on a B200 in tests/golden/ref_parity.npz
      (tests/golden/make_golden.py parity) — bit-exact valid prefixes, fp32 fitness within 1e-5 relative
      (BASELINE.json north_star).
"""
import os

import numpy as np
import pytest
import torch

import gpu_util as G
from conftest import ALL_FUNCS, ARITH_FUNCS, EXACT_FUNCS, depth2leaf, make_data, make_forest, roulette

pytestmark = pytest.mark.gpu
RTOL = 1e-5   # north star: fp32 fitness within 1e-5 relative
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_parity.npz")


@pytest.fixture(scope="module")
def ref(orc):
    """The reference's results replayed from GOLDEN; with EVOGP_RECORD_REFERENCE=<path.npz> (make_golden.py parity)
    its kernels run live from oracle/_ref and the results are written to that file instead."""
    record = os.environ.get("EVOGP_RECORD_REFERENCE")
    if not record:
        yield G.GoldenReference(GOLDEN)
        return
    rec = G.RecordingReference(orc.ref_gpu())
    yield rec
    rec.save(record)


def gen_args(funcs, layers, consts=(-1.0, 0.0, 1.0), leaf_prob=0.2):
    return depth2leaf(layers, leaf_prob), roulette(funcs), np.array(consts, np.float32)


# --------------------------------------------------------------------------- generate
GEN_CASES = [
    # pop, L, V, O, funcs, layers, keys
    (5000, 32, 3, 1, ARITH_FUNCS, 4, (42, 0)),
    (20000, 64, 3, 1, ARITH_FUNCS, 6, (1, 2)),
    (3000, 64, 10, 1, ALL_FUNCS, 4, (123456, 654321)),
    (3000, 128, 13, 3, ALL_FUNCS, 4, (7, 7)),
    (1000, 33, 2, 2, ARITH_FUNCS + ["sin"], 5, (9, 8)),      # odd row width
    (64, 1024, 5, 1, ARITH_FUNCS, 9, (3, 1)),               # widest rows
    (1, 16, 1, 1, ["neg"], 3, (0, 0)),
    (100000, 64, 3, 1, ARITH_FUNCS, 6, (1000, 7)),            # configs[1]: one full wave of the one-tree-per-lane kernel
    # populations large enough for the lane-re-arming kernel (generate.cu generate_balanced_kernel): spans of ~85 trees
    (300001, 64, 10, 1, ALL_FUNCS, 4, (5, 6)),                # ragged last span
    (290001, 33, 2, 1, ARITH_FUNCS + ["sin"], 5, (9, 8)),     # odd row width
]


@pytest.mark.parametrize("case", GEN_CASES)
def test_generate_bit_exact(native, orc, ref, case):
    pop, L, V, O, funcs, layers, keys = case
    d2l, roul, consts = gen_args(funcs, layers)
    want = orc.generate(pop, L, V, O, 0.5, 0.5, np.array(keys, np.uint32), d2l, roul, consts)
    k, a, r, c = G.to_dev(np.array(keys, np.uint32), d2l, roul, consts)
    got = G.abi_generate(native, pop, L, V, O, 0.5, 0.5, k, a, r, c)
    torch.cuda.synchronize()
    for g, w in zip(got, want):
        assert G.same_bits(g, w)           # whole rows: oracle and kernel both zero-fill tails
    assert G.prefix_digest(*got) == ref.generate(pop, L, V, O, 0.5, 0.5, k, a, r, c)   # reference defines prefixes only
    orc.check_forest(*[g.cpu().numpy() for g in got], input_len=V, output_len=O)


# --------------------------------------------------------------------------- splice
def splice_inputs(orc, pop, L, V, funcs, layers, n_new, seed):
    v, t, s = make_forest(orc, pop, L, V, 1, funcs, layers, keys=(seed, seed + 1), leaf_prob=0.1)
    lens = s[:, 0].astype(np.int64)
    rng = np.random.default_rng(seed)
    li = rng.integers(0, pop, n_new).astype(np.int32)
    ri = rng.integers(0, pop, n_new).astype(np.int32)
    lp = (rng.integers(0, 1 << 30, n_new) % lens[li]).astype(np.int32)
    rp = (rng.integers(0, 1 << 30, n_new) % lens[ri]).astype(np.int32)
    ri[: n_new // 50] = -1
    ri[n_new // 50: n_new // 25] = pop
    return (v, t, s), (li, ri, lp, rp), lens


@pytest.mark.parametrize("pop,L,funcs,layers,n_new", [(2000, 32, ARITH_FUNCS, 5, 7001), (3000, 64, ARITH_FUNCS + ["sin", "neg"], 6, 5000),
                                                      (500, 128, ALL_FUNCS, 4, 999), (300, 33, ARITH_FUNCS, 5, 1000)])
def test_crossover_bit_exact(native, orc, ref, pop, L, funcs, layers, n_new):
    forest, idx, lens = splice_inputs(orc, pop, L, 3, funcs, layers, n_new, seed=11)
    want = orc.crossover(*forest, *idx)
    df, di = G.to_dev(*forest), G.to_dev(*idx)
    got = G.abi_crossover(native, *df, *di)
    torch.cuda.synchronize()
    for g, w in zip(got, want):
        assert G.same_bits(g, w)
    assert G.prefix_digest(*got) == ref.crossover(*df, *di)
    orc.check_forest(*[g.cpu().numpy() for g in got], input_len=3)
    assert (want[2][:, 0] == lens[idx[0]]).sum() > n_new // 25      # fallbacks were exercised


@pytest.mark.parametrize("pop,L,layers", [(4000, 32, 5), (4000, 64, 6), (500, 31, 4)])
def test_mutate_bit_exact(native, orc, ref, pop, L, layers):
    v, t, s = make_forest(orc, pop, L, 3, 1, ARITH_FUNCS, layers, keys=(5, 5), leaf_prob=0.1)
    nv, nt, ns = make_forest(orc, pop, L, 3, 1, ARITH_FUNCS, 3, keys=(6, 6))
    lens = s[:, 0].astype(np.int64)
    rng = np.random.default_rng(0)
    pos = (rng.integers(0, 1024, pop) % lens).astype(np.int32)
    pos[:20] = -1
    pos[20:40] = lens[20:40]
    want = orc.mutate(v, t, s, pos, nv, nt, ns)
    dargs = G.to_dev(v, t, s, pos, nv, nt, ns)
    got = G.abi_mutate(native, *dargs)
    torch.cuda.synchronize()
    for g, w in zip(got, want):
        assert G.same_bits(g, w)
    assert G.prefix_digest(*got) == ref.mutate(*dargs)


# --------------------------------------------------------------------------- SR fitness
FIT_CASES = [
    # pop, L, V, O, funcs, layers, N
    (3000, 64, 3, 1, ARITH_FUNCS, 6, 1024),
    (3000, 64, 10, 1, ARITH_FUNCS, 6, 1000),
    (2000, 32, 3, 1, ARITH_FUNCS, 5, 8),
    (2000, 32, 2, 1, ARITH_FUNCS + ["sin", "cos", "tan"], 5, 100),
    (2000, 64, 4, 1, ALL_FUNCS, 4, 300),
    (1500, 128, 13, 3, ALL_FUNCS, 4, 257),
    (1500, 64, 5, 2, ARITH_FUNCS, 6, 1024),
    (700, 33, 3, 1, EXACT_FUNCS, 3, 1),
]


@pytest.mark.parametrize("case", FIT_CASES)
@pytest.mark.parametrize("use_mse", [True, False])
def test_sr_fitness_vs_reference_cuda(native, orc, ref, case, use_mse):
    pop, L, V, O, funcs, layers, N = case
    v, t, s = make_forest(orc, pop, L, V, O, funcs, layers, keys=(2, 3), consts=(-1.0, 0.5, 2.0))
    X, y = make_data(N, V, O, seed=1)
    dv, dt, ds, dX, dy = G.to_dev(v, t, s, X, y)
    got = G.abi_sr_fitness(native, dv, dt, ds, dX, dy, use_mse)
    want = ref.sr_fitness(dv, dt, ds, dX, dy, use_mse, kernel_type=4)
    torch.cuda.synchronize()
    G.assert_close_fitness(got, want, rtol=RTOL, what=f"vs reference CUDA {case}")
    # determinism: same bits on a second run
    again = G.abi_sr_fitness(native, dv, dt, ds, dX, dy, use_mse)
    torch.cuda.synchronize()
    assert G.same_bits(got, again)


# division is div.approx (2 ulp) on the GPU and exact on the CPU; cancellation inside random trees amplifies that,
# so the CPU comparison of "/" trees is loose — the tight 1e-5 check is the one against the reference CUDA kernels
@pytest.mark.parametrize("funcs,rtol", [(EXACT_FUNCS, 1e-5), (ARITH_FUNCS, 2e-3)])
@pytest.mark.parametrize("N", [1, 31, 1024, 1500])
def test_sr_fitness_vs_cpu_oracle(native, orc, funcs, rtol, N):
    layers = 4 if "if" in funcs else 6
    v, t, s = make_forest(orc, 1500, 64, 3, 1, funcs, layers, keys=(8, 1))
    X, y = make_data(N, 3, 1, seed=2)
    want = orc.sr_fitness(v, t, s, X, y, nthreads=8)
    got = G.abi_sr_fitness(native, *G.to_dev(v, t, s, X, y))
    torch.cuda.synchronize()
    if funcs is ARITH_FUNCS:   # division is approximate on the GPU: compare well-conditioned rows only
        ok = np.isfinite(want) & (want < 1e6)
        G.assert_close_fitness(got[torch.from_numpy(ok)], want[ok], rtol=rtol, what="vs CPU oracle")
        assert np.array_equal(np.isnan(got.cpu().numpy()), np.isnan(want))
    else:
        G.assert_close_fitness(got, want, rtol=rtol, what="vs CPU oracle")


@pytest.mark.parametrize("funcs,layers,N", [(ALL_FUNCS, 4, 1024), (ARITH_FUNCS + ["max", "pow", "sinh", "cosh", "loose_pow", "tan"], 5, 700),
                                            (ARITH_FUNCS, 6, 1024), (ARITH_FUNCS + ["sin", "cos", "tan"], 6, 1000)])
def test_replay_width_is_a_speed_knob_only(native, orc, ref, funcs, layers, N):
    """evogp_eval_set_replay_width: both kernel widths against the reference's kernels, every function on the table
    (in the 8-datapoint loop the rare operators share one body per operator behind a second dispatch - gen_fastpath.py).
    A lane owns the same datapoints at either width and adds their errors in the same order: with whole passes
    (N a multiple of 512) the fitness is the same bit for bit; a ragged last pass takes the bounds-checked path, whose
    multiply and add are not contracted, at different datapoints for the two widths (last-bit differences)."""
    v, t, s = make_forest(orc, 3000, 64, 4, 1, funcs, layers, keys=(77, 5), consts=(-1.0, 0.5, 2.0))
    X, y = make_data(N, 4, 1, seed=3)
    dv, dt, ds, dX, dy = G.to_dev(v, t, s, X, y)
    want = ref.sr_fitness(dv, dt, ds, dX, dy, True, kernel_type=4)
    got = {}
    try:
        for width in (8, 16):
            native.set_replay_width(width)
            got[width] = G.abi_sr_fitness(native, dv, dt, ds, dX, dy, True).clone()
            torch.cuda.synchronize()
    finally:
        native.set_replay_width(0)
    for width in (8, 16):
        G.assert_close_fitness(got[width], want, rtol=RTOL, what=f"width {width} vs reference CUDA")
    a, b = got[8].cpu().numpy(), got[16].cpu().numpy()
    assert np.array_equal(np.isnan(a), np.isnan(b))
    if N % 512 == 0:
        assert np.array_equal(a.view(np.uint32)[~np.isnan(a)], b.view(np.uint32)[~np.isnan(b)])
    else:
        G.assert_close_fitness(got[8], b, rtol=1e-6, what="width 8 vs width 16")
    with pytest.raises(RuntimeError, match="replay width"):
        native.set_replay_width(12)


def test_front_end_sets_the_width_from_the_descriptor(native):
    native.load_ops()
    from evogp_b200.tree import Forest, GenerateDescriptor
    common = dict(max_tree_len=32, input_len=2, output_len=1, max_layer_cnt=4, const_samples=[-1.0, 0.0, 1.0])
    d_wide = GenerateDescriptor(using_funcs=["+", "*", "max", "exp"], **common)
    d_hot = GenerateDescriptor(using_funcs={"+": 2.0, "-": 1.0, "sin": 1.0, "tan": 0.0}, **common)
    assert d_wide.func_names == ("+", "*", "max", "exp") and d_hot.func_names == ("+", "-", "sin")
    d_raw = GenerateDescriptor(roulette_funcs=d_wide.roulette_funcs, depth2leaf_probs=d_wide.depth2leaf_probs, **{k: v for k, v in common.items() if k != "max_layer_cnt"})
    assert set(d_raw.func_names) == set(d_wide.func_names)
    X = torch.rand(300, 2, device=G.dev()); y = X[:, :1] * 2
    f = Forest.random_generate(500, d_wide)            # width 8 from here on
    a = f.SR_fitness(X, y)
    native.set_replay_width(16)
    b = f.SR_fitness(X, y)
    torch.cuda.synchronize()
    assert torch.allclose(a, b, rtol=1e-5, atol=1e-6, equal_nan=True)
    Forest.random_generate(10, d_hot)                  # back to the automatic choice
    c = f.SR_fitness(X, y)
    torch.cuda.synchronize()
    assert torch.equal(torch.nan_to_num(b), torch.nan_to_num(c))     # N = 300: the automatic choice is 16 as well


def test_fix_bug_tree_all_modes(native):
    native.load_ops()
    # reference test/fix_bug.py: fitness 0.5 whatever the execute mode
    t = torch.tensor([[3, 3, 0, 0, 3, 0, 0, 0]], dtype=torch.int16, device=G.dev())
    v = torch.tensor([[3, 2, 0, 2, 2, 0, 2, 0]], dtype=torch.float32, device=G.dev())
    s = torch.tensor([[7, 3, 1, 1, 3, 1, 1, 0]], dtype=torch.int16, device=G.dev())
    X = torch.tensor([[0, 0, 0], [0, 0, 1], [0, 1, 0], [0, 1, 1]], dtype=torch.float32, device=G.dev())
    y = torch.tensor([[0], [1], [1], [0]], dtype=torch.float32, device=G.dev())
    for kt in (0, 1, 2, 3, 4):
        fit = torch.ops.evogp_cuda.tree_SR_fitness(1, 4, 8, 3, 1, True, v, t, s, X, y, kt)
        assert float(fit[0]) == 0.5


# --------------------------------------------------------------------------- forward paths
@pytest.mark.parametrize("funcs,O,L,layers", [(EXACT_FUNCS, 1, 40, 4), (ALL_FUNCS, 1, 64, 4), (ALL_FUNCS, 3, 64, 4)])
def test_evaluate_rowwise(native, orc, ref, funcs, O, L, layers):
    pop, V = 4000, 5
    v, t, s = make_forest(orc, pop, L, V, O, funcs, layers, keys=(4, 4), consts=(-2.0, 0.25, 3.0))
    X = np.random.default_rng(5).uniform(-2, 2, (pop, V)).astype(np.float32)
    dv, dt, ds, dX = G.to_dev(v, t, s, X)
    got = G.abi_evaluate(native, dv, dt, ds, dX, O)
    want = ref.evaluate(dv, dt, ds, dX, O)
    torch.cuda.synchronize()
    G.assert_close_fitness(got, want, rtol=RTOL, what="evaluate vs reference CUDA")
    if funcs is EXACT_FUNCS:
        assert G.same_bits(got, orc.evaluate(v, t, s, X, O))


@pytest.mark.parametrize("O,N", [(1, 100), (1, 1024), (3, 64), (2, 7)])
def test_batch_forward(native, orc, O, N):
    pop, V, L = 800, 4, 64
    v, t, s = make_forest(orc, pop, L, V, O, EXACT_FUNCS, 4, keys=(6, 1))
    X, _ = make_data(N, V, seed=3)
    got = G.abi_batch_forward(native, *G.to_dev(v, t, s, X), O)
    torch.cuda.synchronize()
    want = orc.batch_forward(v, t, s, X, O, nthreads=8)
    assert G.same_bits(got, want)   # exact ops only; out nodes accumulate in the reference's order


@pytest.mark.parametrize("pop,L,V,O,N,funcs,layers", [(600, 128, 13, 3, 4096, ALL_FUNCS, 4),      # configs[3] shape (Wine-like)
                                                       (800, 64, 40, 1, 3000, ARITH_FUNCS, 6),     # wide single-output dataset
                                                       (300, 64, 100, 2, 2500, EXACT_FUNCS, 4)])
def test_datasets_larger_than_shared_memory_are_tiled(native, orc, ref, pop, L, V, O, N, funcs, layers):
    """(V + O) * N * 4 bytes exceeds the staging area: the launcher walks the datapoints in tiles and carries the
    running error sum between launches; batch_forward tiles write disjoint slices."""
    v, t, s = make_forest(orc, pop, L, V, O, funcs, layers, keys=(17, 4), consts=(-1.0, 0.5, 2.0))
    X, y = make_data(N, V, O, seed=6)
    dv, dt, ds, dX, dy = G.to_dev(v, t, s, X, y)
    for use_mse in (True, False):
        got = G.abi_sr_fitness(native, dv, dt, ds, dX, dy, use_mse)
        want = ref.sr_fitness(dv, dt, ds, dX, dy, use_mse, kernel_type=4)
        torch.cuda.synchronize()
        G.assert_close_fitness(got, want, rtol=RTOL, what=f"tiled fitness V={V} N={N}")
    bf = G.abi_batch_forward(native, dv, dt, ds, dX, O)
    torch.cuda.synchronize()
    if funcs is EXACT_FUNCS:
        assert G.same_bits(bf, orc.batch_forward(v, t, s, X, O, nthreads=8))
    else:
        sub = slice(0, 64)
        want_bf = orc.batch_forward(v[sub], t[sub], s[sub], X, O, nthreads=8)
        G.assert_close_fitness(bf[sub], want_bf, rtol=5e-3, atol=1e-5, what="tiled batch_forward")


@pytest.mark.parametrize("pop,L,V,O,N,funcs,layers", [(200, 64, 300, 1, 200, ARITH_FUNCS, 6),       # one 512-datapoint pass of 301 floats does not fit
                                                       (150, 64, 512, 1, 129, ARITH_FUNCS, 6),       # the reference's var_len bound
                                                       (100, 32, 256, 8, 77, EXACT_FUNCS, 4)])       # wide multi-output
def test_wide_datasets_fall_back_to_fewer_datapoints_per_lane(native, orc, ref, pop, L, V, O, N, funcs, layers):
    """Hundreds of inputs: 32*K datapoints x (V + O) floats must fit shared memory, so K drops to 4 / 1 instead of
    the call failing (the reference accepts var_len <= 512, forward.cu:318-324)."""
    v, t, s = make_forest(orc, pop, L, V, O, funcs, layers, keys=(23, 9), consts=(-1.0, 0.5, 2.0))
    X, y = make_data(N, V, O, seed=8)
    dv, dt, ds, dX, dy = G.to_dev(v, t, s, X, y)
    got = G.abi_sr_fitness(native, dv, dt, ds, dX, dy, True)
    want = ref.sr_fitness(dv, dt, ds, dX, dy, True, kernel_type=4)
    torch.cuda.synchronize()
    G.assert_close_fitness(got, want, rtol=RTOL, what=f"wide dataset V={V} O={O}")
    vars_used = v[(t & 0x7F) == 0]
    assert vars_used.max() >= V // 2      # the trees do read far columns


@pytest.mark.parametrize("V,N", [(10, 100000), (20, 70000)])
def test_more_than_64_datapoint_tiles(native, orc, V, N):
    """N far beyond 64 tiles of the staging area (the ticket words are reused round-robin): compared with the CPU
    oracle on exact ops, and with the mean of chunk-wise fitness (linearity of the error sum)."""
    pop, L = 64, 64
    v, t, s = make_forest(orc, pop, L, V, 1, EXACT_FUNCS, 4, keys=(3, 30))
    X, y = make_data(N, V, 1, seed=12)
    dv, dt, ds, dX, dy = G.to_dev(v, t, s, X, y)
    got = G.abi_sr_fitness(native, dv, dt, ds, dX, dy, True)
    torch.cuda.synchronize()
    want = orc.sr_fitness(v, t, s, X, y, nthreads=8)
    G.assert_close_fitness(got, want, rtol=1e-4, what=f"{N} datapoints")
    half = N // 2
    a = G.abi_sr_fitness(native, dv, dt, ds, dX[:half].contiguous(), dy[:half].contiguous(), True)
    b = G.abi_sr_fitness(native, dv, dt, ds, dX[half:].contiguous(), dy[half:].contiguous(), True)
    torch.cuda.synchronize()
    comb = (a.double() * half + b.double() * (N - half)) / N
    G.assert_close_fitness(got, comb.float(), rtol=1e-4, what="chunk linearity")


# --------------------------------------------------------------------------- edge cases
def _chain_forest(L, kind):
    """Degenerate shapes: 'unary' = neg(neg(...x0)), 'left' = ((x0+x1)+x1)+..., 'right' = x0+(x1+(x1+...)),
    'bushy' = complete binary tree (deepest operand stack)."""
    t = np.zeros((1, L), np.int16); v = np.zeros((1, L), np.float32); s = np.zeros((1, L), np.int16)
    if kind == "unary":
        t[0, : L - 1] = 2; v[0, : L - 1] = 25; t[0, L - 1] = 0
        s[0] = np.arange(L, 0, -1)
    elif kind == "left":
        n = (L - 1) // 2
        t[0, :n] = 3; v[0, :n] = 1
        t[0, n: 2 * n + 1] = 0; v[0, n] = 0; v[0, n + 1: 2 * n + 1] = 1
        for i in range(n):
            s[0, i] = 2 * (n - i) + 1
        s[0, n: 2 * n + 1] = 1
    elif kind == "right":
        n = (L - 1) // 2
        for i in range(n):
            t[0, 2 * i] = 3; v[0, 2 * i] = 2; s[0, 2 * i] = 2 * (n - i) + 1
            t[0, 2 * i + 1] = 0; v[0, 2 * i + 1] = i % 2; s[0, 2 * i + 1] = 1
        t[0, 2 * n] = 0; v[0, 2 * n] = 1; s[0, 2 * n] = 1
    else:
        depth = int(np.log2(L + 1))
        n = 2**depth - 1
        pos = 0

        def build(d):
            nonlocal pos
            me = pos; pos += 1
            if d == depth - 1:
                t[0, me] = 0; v[0, me] = me % 2; s[0, me] = 1
            else:
                t[0, me] = 3; v[0, me] = 1 + (me % 3)
                build(d + 1); build(d + 1)
                s[0, me] = pos - me
        build(0)
        assert pos == n
    return v, t, s


@pytest.mark.parametrize("L", [7, 64, 127, 1024])
@pytest.mark.parametrize("kind", ["unary", "left", "right", "bushy"])
def test_degenerate_shapes(native, orc, kind, L):
    v, t, s = _chain_forest(L, kind)
    orc.check_forest(v, t, s, input_len=2)
    X, y = make_data(70, 2, seed=9)
    want = orc.sr_fitness(v, t, s, X, y)
    got = G.abi_sr_fitness(native, *G.to_dev(v, t, s, X, y))
    torch.cuda.synchronize()
    G.assert_close_fitness(got, want, rtol=1e-5, what=f"{kind} L={L}")


def _ternary_forest(depth):
    """IF of IFs of ... of leaves: the shape that needs the deepest operand stack per node (2 slots per level)."""
    nodes = []

    def rec(d):
        nodes.append((4, 0.0))
        if d == 0:
            nodes.extend([(0, 0.0), (1, 1.0), (0, 1.0)])
        else:
            rec(d - 1); rec(d - 1); rec(d - 1)
    rec(depth)
    n = len(nodes)
    L = n + (n & 1)
    t = np.zeros((1, L), np.int16); v = np.zeros((1, L), np.float32); s = np.zeros((1, L), np.int16)
    sizes = [0] * n
    for i, (ty, val) in enumerate(nodes):
        t[0, i], v[0, i] = ty, val
    for i in range(n - 1, -1, -1):
        ar = 0 if t[0, i] <= 1 else t[0, i] - 1
        sz, c = 1, i + 1
        for _ in range(ar):
            sz += sizes[c]; c += sizes[c]
        sizes[i] = sz
    s[0, :n] = sizes
    return v, t, s


@pytest.mark.parametrize("N", [256, 1024])   # 8 datapoints per lane (whole stack in tensor memory while depth <= 8) and
                                             # 16 (slots >= 4 in shared memory, reached through the deep opcodes)
@pytest.mark.parametrize("shape", ["bushy127", "bushy1023", "ternary2", "ternary3"])
def test_deep_operand_stacks(native, orc, shape, N):
    if shape.startswith("bushy"):
        v, t, s = _chain_forest(int(shape[5:]) + 1, "bushy")
    else:
        v, t, s = _ternary_forest(int(shape[7:]))
    v, t, s = (np.repeat(a, 40, axis=0) for a in (v, t, s))      # several warps, same tree
    orc.check_forest(v, t, s, input_len=2)
    X, y = make_data(N, 2, seed=12)
    want = orc.sr_fitness(v, t, s, X, y)
    got = G.abi_sr_fitness(native, *G.to_dev(v, t, s, X, y))
    torch.cuda.synchronize()
    G.assert_close_fitness(got, want, rtol=1e-5, what=f"{shape} N={N}")
    out = G.abi_batch_forward(native, *G.to_dev(v, t, s, X), 1).cpu().numpy().reshape(len(v), N)
    ref_out = orc.batch_forward(v, t, s, X, 1).reshape(len(v), N)
    assert np.allclose(out, ref_out, rtol=1e-5, atol=1e-6, equal_nan=True)


def test_fitness_scatter_into_peer_buffers(native, orc):
    """evogp_SR_fitness_scatter: the fused all-gather.  On one GPU the 'peers' are three buffers of this device."""
    import ctypes
    v, t, s = make_forest(orc, 3001, 64, 3, 1, ARITH_FUNCS, 6, keys=(5, 9))
    X, y = make_data(1024, 3, seed=3)
    dv, dt, ds, dX, dy = G.to_dev(v, t, s, X, y)
    want = G.abi_sr_fitness(native, dv, dt, ds, dX, dy)
    abi = native.abi()
    P, L = v.shape
    total, off, world = 5000, 1234, 3
    bufs = [torch.full((total,), -7.0, device="cuda") for _ in range(world)]
    table = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
    local = torch.empty(P, device="cuda")
    nbytes = abi.evogp_eval_workspace_bytes(P, L)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    vp = lambda a: ctypes.c_void_p(a.data_ptr())
    for N in (1024, 100):     # 16 and 4 datapoints per lane
        rc = abi.evogp_SR_fitness_scatter(P, N, L, 3, 1, 1, vp(dv), vp(dt), vp(ds), vp(dX), vp(dy), vp(local), vp(table), world, off,
                                          vp(ws), ctypes.c_size_t(nbytes), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, abi.evogp_last_error()
        torch.cuda.synchronize()
        ref = want if N == 1024 else G.abi_sr_fitness(native, dv, dt, ds, dX[:N].contiguous(), dy[:N].contiguous())
        same = lambda a, b: torch.equal(torch.nan_to_num(a, nan=-1.0), torch.nan_to_num(b, nan=-1.0))
        assert same(local, ref)
        for b in bufs:
            assert same(b[off:off + P], ref) and bool((b[:off] == -7.0).all()) and bool((b[off + P:] == -7.0).all())


def test_if_heavy_trees(native, orc):
    funcs = ["if", "if", "+", "<", "neg"]   # roulette normalises duplicates away; IF share is 1/4
    v, t, s = make_forest(orc, 4000, 121, 3, 1, ["if", "+", "<", "neg"], 5, keys=(13, 13), leaf_prob=0.1)
    orc.check_forest(v, t, s, input_len=3)
    X, y = make_data(200, 3, seed=4)
    want = orc.sr_fitness(v, t, s, X, y, nthreads=8)
    got = G.abi_sr_fitness(native, *G.to_dev(v, t, s, X, y))
    torch.cuda.synchronize()
    G.assert_close_fitness(got, want, rtol=1e-5, what="IF-heavy")


def test_malformed_rows_give_nan_not_a_crash(native, orc):
    v, t, s = make_forest(orc, 64, 32, 3, 1, ARITH_FUNCS, 4, keys=(1, 1))
    s2 = s.copy(); s2[0, 0] = 0; s2[1, 0] = 33; s2[2, 0] = -5      # bad lengths
    t2 = t.copy(); t2[3, : s[3, 0]] = 3                             # all-binary prefix never closes
    X, y = make_data(40, 3)
    got = G.abi_sr_fitness(native, *G.to_dev(v, t2, s2, X, y)).cpu().numpy()
    assert np.isnan(got[:4]).all()
    want = orc.sr_fitness(v, t, s, X, y)
    G.assert_close_fitness(got[4:], want[4:], rtol=2e-4, atol=1e-6, what="untouched rows")


def test_argument_errors_raise(native):
    native.load_ops()
    d = G.dev()
    v = torch.zeros((4, 8), dtype=torch.float32, device=d); t = torch.zeros((4, 8), dtype=torch.int16, device=d)
    s = torch.ones((4, 8), dtype=torch.int16, device=d); X = torch.zeros((5, 2), device=d); y = torch.zeros((5, 1), device=d)
    ops = torch.ops.evogp_cuda
    with pytest.raises(RuntimeError):
        ops.tree_SR_fitness(4, 5, 2000, 2, 1, True, v, t, s, X, y, 4)          # gp_len > MAX_STACK
    with pytest.raises(RuntimeError):
        ops.tree_SR_fitness(4, 5, 8, 3, 1, True, v, t, s, X, y, 4)             # variables shape mismatch
    with pytest.raises(RuntimeError):
        ops.tree_SR_fitness(4, 5, 8, 2, 1, True, v.cpu(), t, s, X, y, 4)       # CPU tensor
    with pytest.raises(RuntimeError):
        ops.tree_crossover(4, 2, 8, v, t, s, torch.zeros(2, dtype=torch.int64, device=d), torch.zeros(2, dtype=torch.int32, device=d),
                           torch.zeros(2, dtype=torch.int32, device=d), torch.zeros(2, dtype=torch.int32, device=d))   # int64 indices
    rc = native.abi().evogp_SR_fitness(4, 5, 8, 2, 1, 1, None, None, None, None, None, None, 4, None, 0, None)
    assert rc == 3 and b"workspace" in native.abi().evogp_last_error()


# --------------------------------------------------------------------------- BASELINE sizes: properties
def test_config2_size_properties(native, orc, ref):
    """configs[1]: pop=100000, L=64, N=1024, V=3.  The oracle cannot run this in seconds, so check
    size-independent properties: permutation equivariance over rows, agreement with the reference CUDA
    kernels on a strided sample, and invariance to how the population is chunked."""
    pop, L, V, N = 100000, 64, 3, 1024
    d2l, roul, consts = gen_args(ARITH_FUNCS, 6)
    k, a, r, c = G.to_dev(np.array([0, 1], np.uint32), d2l, roul, consts)
    v, t, s = G.abi_generate(native, pop, L, V, 1, 0.5, 0.5, k, a, r, c)
    X, y = G.to_dev(*make_data(N, V, seed=0))
    fit = G.abi_sr_fitness(native, v, t, s, X, y)
    perm = torch.randperm(pop, device=G.dev(), generator=torch.Generator(device=G.dev()).manual_seed(0))
    fit_p = G.abi_sr_fitness(native, v[perm].contiguous(), t[perm].contiguous(), s[perm].contiguous(), X, y)
    assert G.same_bits(fit[perm], fit_p)
    half = pop // 2
    f1 = G.abi_sr_fitness(native, v[:half].contiguous(), t[:half].contiguous(), s[:half].contiguous(), X, y)
    f2 = G.abi_sr_fitness(native, v[half:].contiguous(), t[half:].contiguous(), s[half:].contiguous(), X, y)
    assert G.same_bits(fit, torch.cat([f1, f2]))
    sample = torch.arange(0, pop, 37, device=G.dev())
    want = ref.sr_fitness(v[sample].contiguous(), t[sample].contiguous(), s[sample].contiguous(), X, y)
    torch.cuda.synchronize()
    G.assert_close_fitness(fit[sample], want, rtol=RTOL, what="config-2 sample vs reference CUDA")
    # datapoint-order invariance up to summation order
    pd = torch.randperm(N, device=G.dev(), generator=torch.Generator(device=G.dev()).manual_seed(1))
    fit_d = G.abi_sr_fitness(native, v, t, s, X[pd].contiguous(), y[pd].contiguous())
    G.assert_close_fitness(fit_d, fit, rtol=1e-5, what="datapoint permutation")


def test_config5_shape_genetic_ops_properties(native, orc):
    """Full-size crossover + mutation (config 5's per-GPU shape: 150k survivors -> 495k children, L=64):
    children are structurally valid, lengths follow the splice arithmetic, and a no-op splice is the identity."""
    P_src, P_new, L = 150000, 495000, 64
    d2l, roul, consts = gen_args(ARITH_FUNCS, 6)
    k, a, r, c = G.to_dev(np.array([5, 6], np.uint32), d2l, roul, consts)
    v, t, s = G.abi_generate(native, P_src, L, 10, 1, 0.5, 0.5, k, a, r, c)
    g = torch.Generator(device=G.dev()).manual_seed(0)
    li = torch.randint(0, P_src, (P_new,), dtype=torch.int32, device=G.dev(), generator=g)
    ri = torch.randint(0, P_src, (P_new,), dtype=torch.int32, device=G.dev(), generator=g)
    lens = s[:, 0].int()
    lp = torch.randint(0, 2**31 - 1, (P_new,), dtype=torch.int32, device=G.dev(), generator=g) % lens[li.long()]
    rp = torch.randint(0, 2**31 - 1, (P_new,), dtype=torch.int32, device=G.dev(), generator=g) % lens[ri.long()]
    cv, ct, cs = G.abi_crossover(native, v, t, s, li, ri, lp, rp)
    sub_l = s[li.long(), lp.long()].int(); sub_r = s[ri.long(), rp.long()].int()
    want_len = lens[li.long()] + torch.where(lens[li.long()] + sub_r - sub_l <= L, sub_r - sub_l, torch.zeros_like(sub_l))
    assert torch.equal(cs[:, 0].int(), want_len)
    # tails are zero, prefixes closed: check a strided sample with the structural validator
    idx = torch.arange(0, P_new, 97, device=G.dev())
    orc.check_forest(cv[idx].cpu().numpy(), ct[idx].cpu().numpy(), cs[idx].cpu().numpy(), input_len=10)
    cols = torch.arange(L, device=G.dev())[None, :]
    assert not (cs[cols.expand_as(cs) >= cs[:, :1]].any() or ct[cols.expand_as(ct) >= cs[:, :1]].any())
    # identity: replacing a subtree by itself
    same = torch.arange(P_src, dtype=torch.int32, device=G.dev())
    pos = torch.randint(0, 2**31 - 1, (P_src,), dtype=torch.int32, device=G.dev(), generator=g) % lens
    iv, it, is_ = G.abi_crossover(native, v, t, s, same, same, pos, pos)
    assert torch.equal(iv.view(torch.int32), v.view(torch.int32)) and torch.equal(it, t) and torch.equal(is_, s)
