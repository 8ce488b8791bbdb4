"""CPU tests (-m "not gpu"): the oracle port against the reference's golden vectors and the compiled reference's stored results,
plus known-answer properties of the TV-L1 prox (SURVEY.md section 8c)."""
import numpy as np

from conftest import digest
from oracle import oracle as O

METHODS = ["hybrid", "linearized", "classic", "condat"]


def test_port_matches_golden_1d(golden, port):
    for k in range(int(golden["d1_count"])):
        y = golden["d1_%02d_y" % k]; lam = float(golden["d1_%02d_lam" % k])
        for m in METHODS:
            got = getattr(port, "tv1_" + m)(y, lam)
            assert np.array_equal(got, golden["d1_%02d_%s" % (k, m)]), (k, m)
        if y.size >= 2:
            assert np.array_equal(port.tv1_weighted(y, golden["d1_%02d_w" % k]), golden["d1_%02d_weighted" % k]), k


def test_port_matches_golden_cfg1_digest(golden, port):
    y = O.gen_cfg1(200_000, seed=0)
    x = port.tv1_hybrid(y, 0.5)
    d = golden["cfg1_200k_digest"]
    assert x.sum() == d[0] and (x * x).sum() == d[1] and np.count_nonzero(np.diff(x)) == d[2]
    assert np.array_equal(x[:: 200_000 // 64][:64], golden["cfg1_200k_samples"])


def test_port_matches_golden_2d(golden, port):
    for k in range(int(golden["dr_count"])):
        Y = golden["dr_%d_Y" % k]; lam = float(golden["dr_%d_lam" % k]); it = int(golden["dr_%d_it" % k])
        o, info = port.dr2_tv(Y, lam, maxit=it)
        assert np.array_equal(o, golden["dr_%d_out" % k]) and np.array_equal(info, golden["dr_%d_info" % k])
        o, info = port.pd2_tv(Y, [lam, 1.5 * lam], [1, 2], maxit=it)
        assert np.array_equal(o, golden["pd2_%d_out" % k]) and np.array_equal(info, golden["pd2_%d_info" % k])


def test_port_matches_golden_weighted_2d(golden, port):
    for k in range(int(golden["drw_count"])):
        o, info = port.dr2l1w_tv(golden["drw_%d_Y" % k], golden["drw_%d_W1" % k], golden["drw_%d_W2" % k], maxit=int(golden["drw_%d_it" % k]))
        assert np.array_equal(o, golden["drw_%d_out" % k]) and np.array_equal(info, golden["drw_%d_info" % k]), k


def test_port_matches_golden_nd(golden, port):
    o, info = port.pd_tv(golden["pd3_V"], [0.2, 0.2, 0.2], [1, 2, 3])
    assert np.array_equal(o, golden["pd3_out"]) and np.array_equal(info, golden["pd3_info"])
    o, info = port.pd_tv(golden["pd4_V"], [0.3, 0.1, 0.2, 0.4, 0.05], [1, 2, 3, 4, 2])
    assert np.array_equal(o, golden["pd4_out"]) and np.array_equal(info, golden["pd4_info"])
    o, info = port.pd_tv(golden["d1_05_y"], [0.7], [1])
    assert np.array_equal(o, golden["pd1_out"]) and np.array_equal(info, golden["pd1_info"])


# ---- the port against the compiled reference.  Each helper computes, for either implementation (the port here, the reference in
#      tests/golden/make_golden.py), every result its test compares; the reference's side is stored in tests/golden/reference_checks.npz
#      (digests for bit-identical comparisons, values otherwise) ----
def _mismatches(got, refcheck, prefix):
    return {k: np.nonzero(v != refcheck[prefix + k])[0][:10].tolist() for k, v in got.items() if not np.array_equal(v, refcheck[prefix + k])}


def random_1d_digests(impl):
    """Seeded random 1D signals: digests of the input, of every method's result, of the hybrid forced to switch to the classic
    method, and of the weighted result (0 for signals of one sample)."""
    out = {k: [] for k in ["y"] + METHODS + ["hybrid_e0.5", "hybrid_e0.9", "weighted"]}
    rng = np.random.default_rng(5)
    for trial in range(150):
        n = int(rng.integers(1, 300))
        y = rng.normal(0, rng.choice([0.1, 1, 100]), n)
        if trial % 5 == 0:
            y = np.round(y)
        lam = float(rng.choice([0, 0.01, 0.5, 2, 20, 1000]) * rng.uniform(0.5, 1.5))
        out["y"].append(digest(y))
        for m in METHODS:
            out[m].append(digest(getattr(impl, "tv1_" + m)(y, lam)))
        for e in (0.5, 0.9):        # force the hybrid's switch to the classic method
            out["hybrid_e%s" % e].append(digest(impl.tv1_hybrid(y, lam, e)))
        out["weighted"].append(digest(impl.tv1_weighted(y, rng.uniform(0, 2, n - 1))) if n >= 2 else np.uint64(0))
    return {k: np.array(v, dtype=np.uint64) for k, v in out.items()}


def test_port_matches_compiled_reference_random(port, refcheck):
    assert not _mismatches(random_1d_digests(port), refcheck, "rand1d_")      # {result: trials that differ}


def dr2_digests(impl):
    Y = O.gen_cfg2(70, 45, seed=11, block=8)
    a, ia = impl.dr2_tv(Y, 0.25, n_threads=2)
    p, ip = impl.pd2_tv(Y, [0.2, 0.3], [2, 1])
    return {"Y": np.array([digest(Y)]), "dr": np.array([digest(a)]), "dr_info": ia, "pd2": np.array([digest(p)]), "pd2_iters": ip[:1]}


def test_port_matches_compiled_reference_2d(port, refcheck):
    assert not _mismatches(dr2_digests(port), refcheck, "dr2_")


def weighted_2d_digests(impl):
    rng = np.random.default_rng(12)
    out = {"in": [], "out": [], "info": []}
    for (M, N, it) in [(2, 2, 0), (4, 2, 5), (33, 47, 0), (70, 45, 0), (64, 64, 3)]:
        Y = np.asfortranarray(rng.normal(0, 1, (M, N)))
        W1 = rng.uniform(0, 0.6, (M - 1, N)); W2 = rng.uniform(0, 0.6, (M, N - 1))
        a, ia = impl.dr2l1w_tv(Y, W1, W2, maxit=it, n_threads=3)
        out["in"].append(digest(np.concatenate([Y.ravel(), W1.ravel(), W2.ravel()]))); out["out"].append(digest(a)); out["info"].append(ia)
    return {"in": np.array(out["in"], dtype=np.uint64), "out": np.array(out["out"], dtype=np.uint64), "info": np.array(out["info"])}


def test_port_matches_compiled_reference_weighted_2d(port, refcheck):
    assert not _mismatches(weighted_2d_digests(port), refcheck, "w2d_")        # {result: shapes that differ}
    # uniform weights: the weighted iteration is the unweighted one up to rounding (prox_tv_test.py:129-153 allows 1e-3)
    Y = O.gen_cfg2(64, 48, seed=3, block=8)
    a, _ = port.dr2l1w_tv(Y, np.full((63, 48), 0.2), np.full((64, 47), 0.2)); b, _ = port.dr2_tv(Y, 0.2)
    assert np.abs(a - b).max() <= 1e-12


# reference solver -> (weighted, tolerance against the exact scan)
ALT_SOLVERS = {"PN_TV1": (False, 1e-9), "SolveTVConvexQuadratic_a1_nw": (False, 1e-9), "dp": (False, 1e-9),
               "TV1D_denoise_tautstring": (False, 1e-5), "SolveTVConvexQuadratic_a1": (True, 1e-9), "PN_TV1_Weighted": (True, 1e-9)}


def alt_solver_cases():
    """(y, lam, edge weights) of test_reference_alternative_1d_solvers_share_the_minimiser."""
    rng = np.random.default_rng(17)
    for _ in range(25):
        n = int(rng.integers(2, 300)); y = rng.normal(0, 1, n); lam = float(rng.choice([0.05, 0.5, 5]))
        yield y, lam, rng.uniform(0, 2, n - 1)


def test_reference_alternative_1d_solvers_share_the_minimiser(port, refcheck):
    """PN, Kolmogorov, Johnson's DP and Condat's taut-string variant of the reference agree with the exact scan (the C ABI maps
    all of them onto the one kernel, include/proxtv_b200.h).  The reference's results are stored case after case."""
    cases = list(alt_solver_cases())
    assert np.array_equal([digest(np.concatenate([y, w])) for y, _, w in cases], refcheck["alt_in"])
    ends = np.cumsum([y.size for y, _, _ in cases])
    for k, (y, lam, w) in enumerate(cases):
        want = {False: port.tv1_linearized(y, lam), True: port.tv1_weighted(y, w)}
        for name, (weighted, tol) in ALT_SOLVERS.items():
            x = refcheck["alt_" + name][ends[k] - y.size:ends[k]]
            assert np.abs(x - want[weighted]).max() < tol, (k, name)


# ---- known-answer properties (hold for the exact minimiser, any implementation) ----
def test_lambda_zero_is_identity(port):
    y = np.random.default_rng(0).normal(size=333)
    for m in METHODS:
        assert np.allclose(getattr(port, "tv1_" + m)(y, 0.0), y, rtol=0, atol=1e-15)


def test_large_lambda_gives_mean(port):
    y = np.random.default_rng(1).normal(size=200)
    for m in METHODS:
        assert np.allclose(getattr(port, "tv1_" + m)(y, 1e6), y.mean(), rtol=0, atol=1e-9)


def test_weighted_uniform_equals_unweighted(port):
    rng = np.random.default_rng(2)
    for n in (2, 3, 50, 777):
        y = rng.normal(size=n); lam = 0.37
        assert np.allclose(port.tv1_weighted(y, np.full(n - 1, lam)), port.tv1_linearized(y, lam), rtol=0, atol=1e-12)


def test_methods_agree_and_share_jump_set(port):
    y = O.gen_cfg1(50_000, seed=3)
    a = port.tv1_linearized(y, 0.5); b = port.tv1_classic(y, 0.5); c = port.tv1_condat(y, 0.5)
    assert np.abs(a - b).max() < 1e-9 and np.array_equal(a, c)
    assert np.array_equal(port.jump_set(a), port.jump_set(b))


def test_optimality_conditions(port):
    """KKT of the prox: u = cumsum(y - x) satisfies |u_i| <= lam, u_i = -lam*sign(jump) exactly where x jumps, u_{n-1} = 0."""
    y = O.gen_cfg1(20_000, seed=4); lam = 0.5
    x = port.tv1_linearized(y, lam)
    u = np.cumsum(y - x)
    assert np.abs(u).max() <= lam + 1e-9 and abs(u[-1]) < 1e-8
    j = np.nonzero(np.diff(x))[0]
    assert np.allclose(u[j], -lam * np.sign(np.diff(x)[j]), atol=1e-8)


def test_pd_single_term_equals_tv1_1d(port):
    y = np.random.default_rng(6).normal(size=500)
    o, info = port.pd_tv(y, [0.8], [1])
    assert np.array_equal(o.ravel(), port.tv1_hybrid(y, 0.8))


def pdr_digests(impl):
    rng = np.random.default_rng(4)
    out = {"in": [], "out": [], "info": []}
    for shp, ws, ds in [((20, 17), [0.3, 0.2], [1, 2]), ((9, 8, 7), [0.2, 0.2, 0.2], [1, 2, 3]),
                        ((6, 5, 4, 3), [0.3, 0.1, 0.2, 0.4, 0.05], [1, 2, 3, 4, 2]), ((40,), [0.7], [1])]:
        V = np.asfortranarray(rng.normal(size=shp))
        for it in (0, 3, 50):
            a, ia = impl.pdr_tv(V, ws, ds, maxit=it)
            out["in"].append(digest(V)); out["out"].append(digest(a)); out["info"].append(ia)
    return {"in": np.array(out["in"], dtype=np.uint64), "out": np.array(out["out"], dtype=np.uint64), "info": np.array(out["info"])}


def test_pdr_port_equals_reference(port, refcheck):
    """PDR_TV (src/TVNDopt.cpp:280-500, SURVEY.md 8f N4): the port must be bit-identical to the compiled reference, including
    info[] and the in-place scaling of the weights."""
    assert not _mismatches(pdr_digests(port), refcheck, "pdr_")               # {result: (shape, iterations) runs that differ}
