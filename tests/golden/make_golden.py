"""Generates tests/golden/golden_v1.npz from the UNMODIFIED reference (oracle/_ref/libproxtv_ref.so, compiled from
/root/reference/src by oracle/build_ref.sh).  The reference ships no golden vectors (SURVEY.md section 4), so these
fixtures -- inputs (seeded) and the reference's outputs -- are the portable pin for the oracle port and the CUDA path.

Run from the repo root in a container that has /root/reference:  python tests/golden/make_golden.py
tests/golden/reference_checks.npz (the reference's side of the tests that compare with it):  python tests/golden/make_golden.py reference_checks
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import digest  # noqa: E402
from oracle import oracle as O  # noqa: E402


def main():
    R = O.Ref()
    out = {}

    def generated(name, x, call):
        """An input made by synth_inputs is stored as its call (the golden fixture in tests/conftest.py regenerates it) and a digest."""
        out[name + "_" + call[0]] = np.array(call[1:], dtype=np.int64); out[name + "_digest"] = digest(x)
        return x
    rng = np.random.default_rng(20260924)
    # ---- 1D: (name, y, lam) ----
    cases = []
    for n, lam, scale in [(1, 0.5, 1), (2, 0.3, 1), (3, 10.0, 1), (17, 0.0, 1), (64, 0.2, 0.3), (200, 1.0, 1.0),
                          (257, 5.0, 1.0), (1000, 0.5, 0.5), (1000, 50.0, 0.5), (4096, 0.2, 0.3)]:
        y = np.repeat(rng.normal(0, 2, n // 16 + 1), 16)[:n] + rng.normal(0, scale, n)
        cases.append((y, lam))
    cases.append((np.round(rng.normal(0, 3, 300)), 2.0))          # integer data: exact ties
    cases.append((np.full(100, 1.25), 0.7))                       # constant
    cases.append((np.linspace(-3, 3, 500), 0.4))                  # ramp
    cases.append((np.sin(np.linspace(0, 20, 2000)) * 3, 0.3))     # smooth: long hull
    for k, (y, lam) in enumerate(cases):
        out["d1_%02d_y" % k] = y
        out["d1_%02d_lam" % k] = np.float64(lam)
        out["d1_%02d_hybrid" % k] = R.tv1_hybrid(y, lam)
        out["d1_%02d_linearized" % k] = R.tv1_linearized(y, lam)
        out["d1_%02d_classic" % k] = R.tv1_classic(y, lam)
        out["d1_%02d_condat" % k] = R.tv1_condat(y, lam)
        if y.size >= 2:
            w = rng.uniform(0.0, 2 * max(lam, 0.1), y.size - 1)
            out["d1_%02d_w" % k] = w
            out["d1_%02d_weighted" % k] = R.tv1_weighted(y, w)
    out["d1_count"] = np.int64(len(cases))
    # cfg-1 style long signal, stored as a digest only (sum, sumsq, jump count, 64 samples) to keep the file small
    y = O.gen_cfg1(200_000, seed=0)
    x = R.tv1_hybrid(y, 0.5)
    out["cfg1_200k_digest"] = np.array([x.sum(), (x * x).sum(), np.count_nonzero(np.diff(x))])
    out["cfg1_200k_samples"] = x[:: 200_000 // 64][:64]
    # ---- 2D DR / PD2 ----
    for k, (M, N, lam, it) in enumerate([(2, 2, 0.3, 0), (3, 5, 0.5, 0), (37, 53, 0.2, 0), (64, 48, 0.2, 7), (96, 128, 1.0, 0)]):
        Y = generated("dr_%d_Y" % k, O.gen_cfg2(M, N, seed=100 + k, block=8), ("cfg2", M, N, 100 + k, 8))
        o, info = R.dr2_tv(Y, lam, maxit=it)
        out["dr_%d_lam" % k] = np.float64(lam); out["dr_%d_it" % k] = np.int64(it)
        out["dr_%d_out" % k] = o; out["dr_%d_info" % k] = info
        o, info = R.pd2_tv(Y, [lam, 1.5 * lam], [1, 2], maxit=it)
        out["pd2_%d_out" % k] = o; out["pd2_%d_info" % k] = info
    out["dr_count"] = np.int64(5)
    # ---- ND PD ----
    V = generated("pd3_V", O.gen_cfg4((24, 20, 12), seed=2, block=4), ("cfg4", 24, 20, 12, 2, 4))
    o, info = R.pd_tv(V, [0.2, 0.2, 0.2], [1, 2, 3])
    out["pd3_out"] = o; out["pd3_info"] = info
    V4 = np.asfortranarray(rng.normal(0, 1, (6, 5, 4, 3)))
    o, info = R.pd_tv(V4, [0.3, 0.1, 0.2, 0.4, 0.05], [1, 2, 3, 4, 2])
    out["pd4_V"] = V4; out["pd4_out"] = o; out["pd4_info"] = info
    o, info = R.pd_tv(cases[5][0], [0.7], [1])                     # 1 term on a 1D signal (tvgen_1d)
    out["pd1_out"] = o; out["pd1_info"] = info
    # ---- weighted 2D DR (DR2L1W_TV); its own generator so that everything above keeps its draws ----
    rw = np.random.default_rng(20260925)
    shapes = [(2, 2, 0), (3, 4, 0), (5, 2, 4), (37, 53, 0), (64, 48, 7), (96, 128, 0), (130, 100, 0)]
    for k, (M, N, it) in enumerate(shapes):
        if min(M, N) >= 8:
            Y = generated("drw_%d_Y" % k, O.gen_cfg2(M, N, seed=300 + k, block=8), ("cfg2", M, N, 300 + k, 8))
        else:
            Y = out["drw_%d_Y" % k] = np.asfortranarray(rw.normal(0, 1, (M, N)))
        W1 = np.asfortranarray(rw.uniform(0.02, 0.6, (M - 1, N))); W2 = np.asfortranarray(rw.uniform(0.02, 0.6, (M, N - 1)))
        if k == 4: W1[::3] = 0.0                                   # some zero weights (no coupling across those edges)
        o, info = R.dr2l1w_tv(Y, W1, W2, maxit=it)
        out["drw_%d_W1" % k] = W1; out["drw_%d_W2" % k] = W2; out["drw_%d_it" % k] = np.int64(it)
        out["drw_%d_out" % k] = o; out["drw_%d_info" % k] = info
    out["drw_count"] = np.int64(len(shapes))
    path = os.path.join(ROOT, "tests", "golden", "golden_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")


def reference_checks(n_threads=os.cpu_count() or 1):
    """Writes tests/golden/reference_checks.npz: what the compiled reference computes in the tests that compare with it
    (tests/test_oracle.py, tests/test_gpu_fullsize.py), computed here through the tests' own helpers and seeded inputs.  Digests
    stand for results a test requires to be bit-identical; the full-size results are sampled (fixed seeds) to keep the file small."""
    import ctypes as C
    import test_gpu_fullsize as G
    import test_oracle as T
    R = O.Ref()
    out = {}
    for prefix, fn in (("rand1d_", T.random_1d_digests), ("dr2_", T.dr2_digests), ("w2d_", T.weighted_2d_digests), ("pdr_", T.pdr_digests)):
        out.update({prefix + k: v for k, v in fn(R).items()})
    # the reference's other 1D solvers, results stored case after case
    L = R.lib; dp = C.POINTER(C.c_double)
    ptr = lambda a: a.ctypes.data_as(dp)  # noqa: E731
    for f in (L.TV1D_denoise_tautstring, L.SolveTVConvexQuadratic_a1_nw, L.SolveTVConvexQuadratic_a1, L.dp):
        f.restype = None
    calls = {"PN_TV1": lambda y, lam, w, x, n: L.PN_TV1(ptr(y), C.c_double(lam), ptr(x), ptr(np.zeros(3)), n, C.c_double(0.05), None),
             "SolveTVConvexQuadratic_a1_nw": lambda y, lam, w, x, n: L.SolveTVConvexQuadratic_a1_nw(n, ptr(y), C.c_double(lam), ptr(x)),
             "dp": lambda y, lam, w, x, n: L.dp(n, ptr(y), C.c_double(lam), ptr(x)),
             "TV1D_denoise_tautstring": lambda y, lam, w, x, n: L.TV1D_denoise_tautstring(ptr(y), ptr(x), n, C.c_double(lam)),
             "SolveTVConvexQuadratic_a1": lambda y, lam, w, x, n: L.SolveTVConvexQuadratic_a1(n, ptr(y), ptr(w), ptr(x)),
             "PN_TV1_Weighted": lambda y, lam, w, x, n: L.PN_TV1_Weighted(ptr(y), ptr(w), ptr(x), ptr(np.zeros(3)), n, C.c_double(0.05), None)}
    assert set(calls) == set(T.ALT_SOLVERS)
    res = {name: [] for name in calls}
    cases = list(T.alt_solver_cases())
    for y, lam, w in cases:
        wpad = np.append(w, 0.0)
        for name, call in calls.items():
            x = np.zeros(y.size); call(y, lam, wpad, x, y.size); res[name].append(x)
    out["alt_in"] = np.array([digest(np.concatenate([y, w])) for y, _, w in cases], dtype=np.uint64)
    out.update({"alt_" + name: np.concatenate(v) for name, v in res.items()})
    # full size (tests/test_gpu_fullsize.py)
    Y = O.gen_cfg2(4096, 4096, seed=0)
    want = R.dr2_tv(Y, 0.2, n_threads=n_threads)[0]
    rows = np.sort(np.random.default_rng(2).choice(4096, 8, replace=False))
    jr, jc = G.jump_maps(want)
    out.update(cfg2_Y=digest(Y), cfg2_rows=rows, cfg2_want_rows=want[rows], cfg2_absmax=np.abs(want).max(),
               cfg2_row_jumps=jr.sum(axis=1), cfg2_col_jumps=jc.sum(axis=0), cfg2_row_jump_map=digest(jr), cfg2_col_jump_map=digest(jc))
    del Y, want, jr, jc
    imgs = np.stack([np.ascontiguousarray(O.gen_cfg2(2048, 2048, seed=s)).astype(np.float32) for s in range(3)])
    rows = np.sort(np.random.default_rng(3).choice(2048, 4, replace=False))
    want = [R.dr2_tv(np.asfortranarray(im.astype(np.float64)), 0.2, n_threads=n_threads)[0] for im in imgs]
    out.update(cfg5_imgs=digest(imgs), cfg5_rows=rows, cfg5_want_rows=np.stack([w[rows] for w in want]),
               cfg5_absmax=np.array([np.abs(w).max() for w in want]))
    del imgs, want
    V32 = np.asfortranarray(O.gen_cfg4((512, 512, 256), seed=0).astype(np.float32))
    want, winfo = R.pd_tv(np.asfortranarray(V32.astype(np.float64)), [0.2, 0.2, 0.2], [1, 2, 3], n_threads=n_threads)
    idx = np.sort(np.random.default_rng(4).choice(V32.size, 8192, replace=False))
    out.update(cfg4_V32=digest(V32), cfg4_info=winfo, cfg4_index=idx, cfg4_want=want.ravel("F")[idx], cfg4_absmax=np.abs(want).max())
    path = os.path.join(ROOT, "tests", "golden", "reference_checks.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    reference_checks() if sys.argv[1:] == ["reference_checks"] else main()
