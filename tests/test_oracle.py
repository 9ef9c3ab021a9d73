"""CPU suite, part 1: pin the oracle (no GPU needed).

Known answers:  thrust's documented taus88 KAT, the hash/seed/draw values probed from the
reference's kernel.h with keys=(42,0) (SURVEY.md §8c), the hand tree of the reference's
test/fix_bug.py, the descriptor tensors printed in tutorial/evogp_intro.ipynb, hand-derived
operator semantics, and structural invariants of every producer."""
import os

import numpy as np
import pytest

from conftest import ALL_FUNCS, ARITH_FUNCS, depth2leaf, make_data, make_forest, roulette

HERE = os.path.dirname(os.path.abspath(__file__))


def test_taus88_thrust_kat(orc):
    # thrust/random.h:87 — 10000th draw of a default-constructed taus88 (seed 341)
    assert orc.taus88_nth(341, 10000) == 3535848941


def test_hash_and_draws_keys_42_0(orc):
    # probed from the reference's own hash() + thrust taus88 (SURVEY.md §8c item 3)
    expect = {0: (746587583, [3274878540, 509073243, 2395345521]),
              1: (3518090510, [2647108157, 2985584162, 2335719075]),
              2: (1915868893, [2479674156, 43975335, 399991473])}
    for n, (seed, draws) in expect.items():
        assert orc.hash32(n, 42, 0) == seed
        assert orc.taus88_draws(seed, 3).tolist() == draws
    u = orc.taus88_draws(746587583, 3).astype(np.float32) / np.float32(4294967296.0)
    np.testing.assert_allclose(u, [0.762492061, 0.118527852, 0.557709813], rtol=1e-7)


def test_rng_against_reference_headers(orc):
    """The restated hash / taus88 / uniform against the reference's kernel.h + thrust, compiled as is; their outputs
    are stored in tests/golden/ref_rng.npz (tests/golden/make_golden.py rng)."""
    g = np.load(os.path.join(HERE, "golden", "ref_rng.npz"))
    for (n, k1, k2), want in zip(g["hash_args"], g["hash"]):
        assert orc.hash32(int(n), int(k1), int(k2)) == want
    for seed, draws, uniforms in zip(g["seeds"], g["draws"], g["uniforms"]):
        assert np.array_equal(draws, orc.taus88_draws(int(seed), 64))
        mine = orc.taus88_draws(int(seed), 64).astype(np.float32) / np.float32(4294967296.0)
        assert np.array_equal(uniforms, mine)


def fix_bug_tree(L=8):
    # reference test/fix_bug.py:7-10: (x0 - x2) * (x0 - x2)
    t = np.array([[3, 3, 0, 0, 3, 0, 0, 0]], np.int16)
    v = np.array([[3, 2, 0, 2, 2, 0, 2, 0]], np.float32)
    s = np.array([[7, 3, 1, 1, 3, 1, 1, 0]], np.int16)
    return v, t, s


def test_fix_bug_tree_fitness_is_half(orc):
    v, t, s = fix_bug_tree()
    X = np.array([[0, 0, 0], [0, 0, 1], [0, 1, 0], [0, 1, 1]], np.float32)   # fix_bug.py:14-27 (first 4 XOR rows)
    y = np.array([[0], [1], [1], [0]], np.float32)
    out = orc.batch_forward(v, t, s, X, 1)[0, :, 0]
    assert out.tolist() == [0.0, 1.0, 0.0, 1.0]
    assert orc.sr_fitness(v, t, s, X, y)[0] == 0.5
    assert orc.sr_fitness(v, t, s, X, y, use_mse=False)[0] == 0.5


def test_descriptor_tensors_from_tutorial():
    # tutorial/evogp_intro.ipynb cells 3/5: using_funcs=+,-,*,/ and max_layer_cnt=5
    r = roulette(["+", "-", "*", "/"])
    assert r[:6].tolist() == [0.0, 0.25, 0.5, 0.75, 1.0, 1.0] and (r[4:] == 1.0).all()
    assert depth2leaf(5).tolist() == pytest.approx([0.2] * 4 + [1.0] * 6)


def _row(nodes, L=16):
    """nodes: list of (type, value) in prefix order -> packed single-row forest with sizes computed."""
    n = len(nodes)
    t = np.zeros((1, L), np.int16)
    v = np.zeros((1, L), np.float32)
    s = np.zeros((1, L), np.int16)
    for i, (ty, val) in enumerate(nodes):
        t[0, i], v[0, i] = ty, val
    sizes = [0] * n
    for i in range(n - 1, -1, -1):
        ar = 0 if (t[0, i] & 0x7F) <= 1 else (t[0, i] & 0x7F) - 1
        sz, c = 1, i + 1
        for _ in range(ar):
            sz += sizes[c]
            c += sizes[c]
        sizes[i] = sz
    s[0, :n] = sizes
    return v, t, s


VAR, CONST, U, B, T = 0, 1, 2, 3, 4


def test_operator_semantics_hand_cases(orc):
    x = np.array([[2.0, 0.0, -3.0]], np.float32)

    def ev(nodes):
        return orc.evaluate(*_row(nodes), x, 1)[0, 0]

    assert ev([(B, 2), (VAR, 0), (VAR, 2)]) == 5.0                   # SUB: first child is the left operand
    assert ev([(B, 4), (VAR, 0), (VAR, 2)]) == pytest.approx(-2 / 3)  # DIV
    assert np.isnan(ev([(B, 4), (VAR, 0), (VAR, 1)]))                # DIV by zero -> NaN (forward.cu:183-187)
    assert ev([(B, 5), (VAR, 0), (VAR, 1)]) == pytest.approx(2e9)    # LOOSE_DIV clamps |b|<=1e-9
    assert np.isnan(ev([(B, 6), (VAR, 2), (CONST, 2.0)]))            # fast-math pow(x<0, y) is NaN
    assert ev([(B, 7), (VAR, 2), (CONST, 2.0)]) == pytest.approx(9.0, rel=1e-6)   # LOOSE_POW = |a|^b
    assert ev([(B, 7), (VAR, 1), (VAR, 1)]) == 0.0                   # LOOSE_POW(0,0) = 0
    assert ev([(B, 8), (VAR, 0), (VAR, 2)]) == 2.0 and ev([(B, 9), (VAR, 0), (VAR, 2)]) == -3.0
    assert ev([(B, 10), (VAR, 0), (VAR, 2)]) == -1.0 and ev([(B, 11), (VAR, 0), (VAR, 2)]) == 1.0
    assert ev([(T, 0), (VAR, 2), (CONST, 10.0), (CONST, 20.0)]) == 20.0   # IF a>0 ? b : c
    assert ev([(T, 0), (VAR, 0), (CONST, 10.0), (CONST, 20.0)]) == 10.0
    assert ev([(U, 21), (VAR, 1)]) == -1e9                           # LOOSE_LOG(0)
    assert np.isnan(ev([(U, 23), (VAR, 1)]))                         # INV(0) -> NaN
    assert ev([(U, 24), (VAR, 1)]) == pytest.approx(1e9)             # LOOSE_INV clamps
    assert ev([(U, 28), (VAR, 2)]) == pytest.approx(np.sqrt(3.0))    # LOOSE_SQRT = sqrt|a|
    assert np.isnan(ev([(U, 27), (VAR, 2)]))                         # SQRT(<0)
    assert ev([(U, 29), (VAR, 0)]) == 0.0                            # unknown function id evaluates to 0 (G5)
    assert ev([(CONST, 7.5)]) == 7.5 and ev([(VAR, 2)]) == -3.0      # single-leaf trees


def test_multi_output_semantics(orc):
    # out node adds its value to outs[idx] and forwards its RIGHT-most child (forward.cu:236-242)
    def outval(f, idx):
        return np.array([f | (idx << 16)], np.uint32).view(np.float32)[0]

    x = np.array([[2.0, 5.0]], np.float32)
    # root ADD(out) -> outs[1] += (x0 + inner);  inner = MUL(out idx 0)(x0, x1) -> outs[0] += 10, forwards x1 = 5
    nodes = [(B | 0x80, outval(1, 1)), (VAR, 0), (B | 0x80, outval(3, 0)), (VAR, 0), (VAR, 1)]
    res = orc.evaluate(*_row(nodes), x, 2)[0]
    assert res.tolist() == [10.0, 7.0]
    # out index beyond out_len is dropped, value still forwarded
    nodes = [(B, 1), (VAR, 0), (U | 0x80, outval(25, 7)), (VAR, 1)]
    assert orc.evaluate(*_row(nodes), x, 2)[0].tolist() == [0.0, 0.0]


@pytest.mark.parametrize("funcs,layers,L,O", [(ARITH_FUNCS, 5, 32, 1), (ALL_FUNCS, 4, 64, 1), (ALL_FUNCS, 4, 128, 3)])
def test_generate_invariants_and_determinism(orc, funcs, layers, L, O):
    v, t, s = make_forest(orc, 3000, L, 4, O, funcs, layers, keys=(7, 9))
    lens = orc.check_forest(v, t, s, input_len=4, output_len=O)
    assert lens.max() <= L and lens.min() >= 1 and len(np.unique(lens)) > 3
    v2, t2, s2 = make_forest(orc, 3000, L, 4, O, funcs, layers, keys=(7, 9))
    assert np.array_equal(v.view(np.uint32), v2.view(np.uint32)) and np.array_equal(t, t2) and np.array_equal(s, s2)
    v3, _, _ = make_forest(orc, 3000, L, 4, O, funcs, layers, keys=(7, 10))
    assert not np.array_equal(v.view(np.uint32), v3.view(np.uint32))
    # tree n depends on (n, keys) only: a prefix of a bigger population is the same trees
    v4, t4, s4 = make_forest(orc, 100, L, 4, O, funcs, layers, keys=(7, 9))
    assert np.array_equal(v[:100].view(np.uint32), v4.view(np.uint32)) and np.array_equal(s[:100], s4)
    if O > 1:
        assert ((t & 0x80) != 0).any()


def test_generate_first_tree_keys_42_0(orc):
    """Tree 0 of keys=(42,0), +-*/ roulette, layers=5: derived by hand from the pinned draws
    u = .7625, .1185, ... : root is a function (u >= .2) with r=.1185 -> k=1 (ADD)."""
    v, t, s = make_forest(orc, 4, 32, 3, 1, ARITH_FUNCS, 5, keys=(42, 0))
    assert t[0, 0] == B and v[0, 0] == 1.0
    assert s[0, 0] == np.count_nonzero(s[0])


def test_splice_invariants_and_fallbacks(orc):
    rng = np.random.default_rng(3)
    v, t, s = make_forest(orc, 500, 32, 3, 1, ARITH_FUNCS + ["sin"], 5, keys=(1, 2), leaf_prob=0.05, consts=(0.5,))
    lens = s[:, 0].astype(np.int64)
    n = 2000
    li = rng.integers(0, 500, n).astype(np.int32)
    ri = rng.integers(0, 500, n).astype(np.int32)
    lp = (rng.integers(0, 1 << 30, n) % lens[li]).astype(np.int32)
    rp = (rng.integers(0, 1 << 30, n) % lens[ri]).astype(np.int32)
    ri[:10] = -1            # invalid donor -> copy of the recipient (mutation.cu:256-266)
    ri[10:20] = 500
    cv, ct, cs = orc.crossover(v, t, s, li, ri, lp, rp)
    clens = orc.check_forest(cv, ct, cs, input_len=3)
    for k in range(20):
        assert np.array_equal(cs[k], s[li[k]]) and np.array_equal(cv[k].view(np.uint32), v[li[k]].view(np.uint32))
    sub_l = s[li, lp].astype(np.int64)
    sub_r = np.where((ri >= 0) & (ri < 500), s[np.clip(ri, 0, 499), rp], 0).astype(np.int64)
    want = lens[li] + np.where((ri >= 0) & (ri < 500) & (lens[li] + sub_r - sub_l <= 32), sub_r - sub_l, 0)
    assert np.array_equal(clens, want)
    assert (lens[li] + sub_r - sub_l > 32).any(), "test should exercise the too-long fallback"
    # mutation: donor = whole new tree
    nv, nt, ns = make_forest(orc, 500, 32, 3, 1, ARITH_FUNCS, 3, keys=(5, 6))
    pos = (rng.integers(0, 1024, 500) % lens).astype(np.int32)
    pos[:5] = -1
    pos[5:10] = lens[5:10]   # == len: invalid
    mv, mt, ms = orc.mutate(v, t, s, pos, nv, nt, ns)
    mlens = orc.check_forest(mv, mt, ms, input_len=3)
    assert np.array_equal(ms[:10], s[:10])
    k = 20
    assert mlens[k] == lens[k] - s[k, pos[k]] + ns[k, 0] or mlens[k] == lens[k]


def test_splice_hand_case(orc):
    # recipient (x0 + x1) * x2, replace "x1" (pos 3) by donor subtree (x0 - 1) taken at pos 1 of  neg(x0 - 1)
    rv, rt, rs = _row([(B, 3), (B, 1), (VAR, 0), (VAR, 1), (VAR, 2)], L=8)
    dv, dt, ds = _row([(U, 25), (B, 2), (VAR, 0), (CONST, 1.0)], L=8)
    v = np.concatenate([rv, dv]); t = np.concatenate([rt, dt]); s = np.concatenate([rs, ds])
    cv, ct, cs = orc.crossover(v, t, s, [0], [1], [3], [1])
    assert cs[0].tolist() == [7, 5, 1, 3, 1, 1, 1, 0]
    assert ct[0].tolist() == [3, 3, 0, 3, 0, 1, 0, 0]
    assert cv[0].tolist() == [3, 1, 0, 2, 0, 1, 2, 0]
    x = np.array([[2.0, 9.0, 4.0]], np.float32)
    assert orc.evaluate(cv, ct, cs, x, 1)[0, 0] == (2 + (2 - 1)) * 4


def test_fitness_matches_batch_forward(orc):
    v, t, s = make_forest(orc, 200, 64, 3, 1, ARITH_FUNCS, 6, keys=(3, 4))
    X, y = make_data(50, 3)
    out = orc.batch_forward(v, t, s, X, 1)[:, :, 0].astype(np.float64)
    want = ((y[None, :, 0] - out) ** 2).mean(axis=1)
    got = orc.sr_fitness(v, t, s, X, y)
    m = np.isfinite(want)
    np.testing.assert_allclose(got[m], want[m], rtol=1e-5)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    got2 = orc.sr_fitness(v, t, s, X, y, nthreads=4)
    assert np.array_equal(got, got2, equal_nan=True)


def test_philox_known_answer(orc):
    """Random123 KAT: philox4x32-10, counter 0, key 0 (Salmon et al., SC'11 reference implementation kat_vectors)."""
    assert [int(x) for x in orc.philox(0, 0, 0, 0)] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


def test_own_operator_restatements_are_well_formed(orc):
    """The restatements of this library's own operators produce structurally valid forests / permutations (their GPU
    counterparts are compared with them bit for bit in tests/test_gpu_variants.py)."""
    from conftest import ARITH_FUNCS, depth2leaf, roulette
    d2l, roul, consts = depth2leaf(5), roulette(ARITH_FUNCS), np.array([-1.0, 0.0, 1.0], np.float32)
    pv = orc.generate_philox(3000, 64, 3, 1, 0.5, 0.5, np.array([9, 9], np.uint32), d2l, roul, consts)
    lens = orc.check_forest(*pv, input_len=3)
    tv = orc.generate(3000, 64, 3, 1, 0.5, 0.5, np.array([9, 9], np.uint32), d2l, roul, consts)
    assert abs(lens.mean() - tv[2][:, 0].mean()) < 0.1 * tv[2][:, 0].mean()        # same growth distribution
    order = np.random.default_rng(0).permutation(3000).astype(np.int64)
    nv = orc.next_generation(*pv, order, 30, 900, 0.3, 3, 1, 0.5, 0.5, depth2leaf(3), roul, consts, np.array([1, 2], np.uint32))
    orc.check_forest(*nv, input_len=3)
    assert np.array_equal(nv[1][:30], pv[1][order[:30]])
    perm = orc.feistel_perm(1001, 2, np.array([3, 4], np.uint32))
    assert sorted(perm.tolist()) == list(range(1001))
    fit = np.random.default_rng(1).normal(size=1001).astype(np.float32)
    w = orc.tournament(fit, 1, 1.0, False, 1001, np.array([3, 4], np.uint32))
    assert sorted(w.tolist()) == list(range(1001))                                # size-1 tournaments without replacement = a permutation
    sub = orc.extract_subtree(*pv, np.zeros(3000, np.int32))
    assert all(np.array_equal(a, b) for a, b in zip(sub, pv))                     # the subtree at the root is the tree
