"""CPU test (-m "not gpu") of the lane-per-fiber engine: tests/emu/emu_lane.cu runs proxtv_b200/csrc/lane_core.cuh -- the code the
CUDA kernel of kernels_lane.cu executes (scan steps in slope form, circular window management, start marks, sweep, chunk records,
verification and repair) -- on the host, one warp task at a time with the 32 lanes in a plain loop, and the result must agree
with the oracle's sequential taut-string to rounding (<= 1e-9 relative; observed ~1e-15; the slope form is not bit-identical to the
reference's incremental form, jump sets are compared with the 1e-9 threshold used everywhere else).

Covered on purpose: both layouts (contiguous fibers / fibers adjacent in memory), whole-fiber and chunked modes with several halo
lengths (0 = every chunk boundary must be repaired), tiny windows (32 rows: lanes retire because a segment does not fit and the
repair path takes over), the boxed drain of the contiguous layout, partial fiber groups, fibers of 1..3 samples, flat / ramp /
alternating / integer-valued data, lambda from 0 to 1e4, float32 storage, and the fused Douglas-Rachford pass arithmetic driven
through a complete DR2_TV solve against the oracle."""
import ctypes as C

import numpy as np
import pytest

from emu import lane_emu

dp = C.POINTER(C.c_double)
fp = C.POINTER(C.c_float)


@pytest.fixture(scope="module")
def emu():
    return lane_emu.load(required=False)


def _p(a, t=dp):
    return a.ctypes.data_as(t) if a is not None else None


def lane(lib, op, A, B, Cc, nf, ln, inc, lam, clen=0, halo=32, boxed=0, config=0, X2=None):
    f32 = A.dtype == np.float32
    X = np.full_like(A, np.nan); st = (C.c_longlong * 8)()
    t = fp if f32 else dp
    (lib.emu_lane_f32 if f32 else lib.emu_lane_f64)(op, _p(A, t), _p(B, t), _p(Cc, t), _p(X, t), _p(X2, t), nf, ln, inc, lam, clen, halo, boxed, config, st)
    return X, dict(tasks=st[0], epochs=st[1], retire_events=st[2], tails=st[3], rows_fed=st[4], repairs=st[5], retired_lanes=st[6], iters=st[7])


def fibers(A, nf, ln, inc):
    A = np.asarray(A).ravel()
    for j in range(nf):
        base = (j // inc) * inc * ln + j % inc if inc > 1 else j * ln
        yield j, base + np.arange(ln) * (inc if inc > 1 else 1)


def check(lib, port, A, nf, ln, inc, lam, **kw):
    X, st = lane(lib, 0, A, None, None, nf, ln, inc, lam, **kw)
    Af = np.asarray(A, dtype=np.float64).ravel(); Xf = X.ravel()
    for j, idx in fibers(A, nf, ln, inc):
        want = port.tv1_linearized(Af[idx], lam)
        got = Xf[idx]
        assert not np.isnan(got).any(), (j, kw)
        tol = 1e-9 if A.dtype == np.float64 else 3e-6
        assert np.abs(got - want).max() <= tol * max(1.0, np.abs(want).max()), (j, kw, st)
        if A.dtype == np.float64:
            assert np.array_equal(np.nonzero(np.abs(np.diff(got)) > 1e-9)[0], np.nonzero(np.abs(np.diff(want)) > 1e-9)[0]), (j, kw)
    return st


def test_slope_form_sequential_matches_reference_scan(emu, port):
    """The arithmetic alone (no window, no chunks): same minimiser, same jump sets, 1.8 steps per sample on config-2 data."""
    rng = np.random.default_rng(0)
    for t in range(200):
        n = int(rng.integers(1, 3000)); y = rng.normal(0, rng.choice([0.1, 1, 100]), n)
        if t % 4 == 0:
            y = np.round(y)
        lam = float(rng.choice([0, 0.01, 0.5, 2, 20, 1000]) * rng.uniform(0.5, 1.5))
        x = np.empty_like(y); st = C.c_longlong(0)
        emu.emu_slope_seq_f64(_p(y), n, lam, _p(x), C.byref(st))
        w = port.tv1_linearized(y, lam)
        assert np.abs(x - w).max() <= 1e-9 * max(1.0, np.abs(w).max()), (t, n, lam)
        assert np.array_equal(np.nonzero(np.abs(np.diff(x)) > 1e-9)[0], np.nonzero(np.abs(np.diff(w)) > 1e-9)[0]), (t, n, lam)


def test_layouts_chunking_windows(emu, port):
    from oracle import oracle as O
    Y = O.gen_cfg2(256, 200, seed=1, block=16)
    A = np.asfortranarray(Y).ravel("F")
    for cfg in (0, 1):                                       # window 64 / 32 rows
        for clen, halo in ((0, 0), (64, 32), (48, 16), (32, 8), (64, 0)):
            for boxed in (0, 1):
                st = check(emu, port, A, 256, 200, 256, 0.2, clen=clen, halo=halo, boxed=boxed, config=cfg)      # rows: strided fibers
                if halo == 0 and clen:
                    assert st["repairs"] >= 256            # a cold start exactly at the boundary can never be verified
                if halo >= 16 and cfg == 0:
                    assert st["repairs"] == 0
    for clen, halo in ((0, 0), (64, 32)):
        check(emu, port, A, 200, 256, 1, 0.2, clen=clen, halo=halo, boxed=1)                                     # columns: contiguous fibers


def test_adversarial_inputs(emu, port):
    rng = np.random.default_rng(5)

    def mk(kind, nf, ln):
        if kind == 0: return np.repeat(rng.normal(0, 1, (nf, ln // 16 + 1)), 16, axis=1)[:, :ln] + rng.normal(0, 0.3, (nf, ln))
        if kind == 1: return np.full((nf, ln), 2.5)
        if kind == 2: return np.tile(np.linspace(-3, 3, ln), (nf, 1)) + rng.normal(0, 0.01, (nf, 1))
        if kind == 3: return np.round(rng.normal(0, 3, (nf, ln)))
        if kind == 4: return np.sin(np.linspace(0, 20, ln))[None, :] * 3 + rng.normal(0, 0.05, (nf, ln))
        if kind == 5:
            a = rng.normal(0, 1, (nf, ln)); a[:, ln // 3:2 * ln // 3] = 0.3; return a
        return np.where(np.arange(ln) % 2 == 0, 1.0, -1.0)[None, :] * np.ones((nf, 1))

    repairs = 0
    for trial in range(250):
        nf = int(rng.choice([1, 5, 31, 32, 33, 64, 70])); ln = int(rng.choice([1, 2, 3, 7, 31, 32, 33, 63, 64, 65, 100, 129, 257, 500, 1000]))
        kind = int(rng.integers(0, 7)); lam = float(rng.choice([0.0, 0.05, 0.2, 1.0, 5.0, 50.0, 1e4]))
        data = mk(kind, nf, ln)
        clen = int(rng.choice([0, 16, 32, 48, 64, 128])); halo = int(rng.choice([0, 8, 16, 32])); boxed = int(rng.integers(0, 2)); cfg = int(rng.integers(0, 3))
        if rng.integers(0, 2):
            A = np.ascontiguousarray(data).ravel(); inc = 1
        else:
            A = np.ascontiguousarray(data.T).ravel(); inc = nf
        repairs += check(emu, port, A, nf, ln, inc, lam, clen=clen, halo=halo, boxed=boxed, config=cfg)["repairs"]
    assert repairs > 500                                     # the repair path was exercised, not just the fast path


def test_float32_storage(emu, port):
    from oracle import oracle as O
    Y = O.gen_cfg2(96, 300, seed=3, block=16).astype(np.float32)
    A = np.asfortranarray(Y).ravel("F")
    for clen, halo in ((0, 0), (128, 32)):
        check(emu, port, A, 96, 300, 96, np.float32(0.2), clen=clen, halo=halo, config=0)
        check(emu, port, A, 300, 96, 1, np.float32(0.2), clen=0, halo=0, boxed=1, config=0)


def test_douglas_rachford_through_the_lane_passes(emu, port):
    """Whole DR2_TV solves made of lane passes, exactly as solver.cu issues them, against the oracle.
    (a) the staged schedule: column pass plain (contiguous fibers), row pass with the three operands combined at landing;
    (b) the transposed schedule (the default): BOTH passes strided, each over its own copy (columns over the row-major arrays, rows
        over the column-major ones), arithmetic in the drain, results written transposed into the other layout."""
    from oracle import oracle as O
    M, N = 96, 80
    Y = O.gen_cfg2(M, N, seed=2, block=8)
    want = port.dr2_tv(Y, 0.2)[0]
    Yf = Y.ravel("F").copy()
    t = np.full_like(Yf, 2 * Yf.mean())
    out = None
    for it in range(36):
        final = it == 35
        x1 = t.copy() if it == 0 else lane(emu, 0, t, None, None, N, M, 1, 0.2, clen=32, halo=16, boxed=1)[0]
        out = lane(emu, 2 if final else 1, Yf, x1, t, M, N, M, 0.2, clen=32, halo=16)[0]
        if not final:
            t = out
    got = out.reshape(N, M).T
    assert np.abs(got - want).max() / np.abs(want).max() <= 1e-9
    staged = got

    Yr = np.ascontiguousarray(Y).ravel()                     # row-major copy: column fibers have stride N, adjacent columns are adjacent
    t0 = 2 * Yf.mean()
    Uc = Yf - (2.0 * (t0 - t0) - t0); Dc = np.zeros_like(Yf)   # first column pass: prox of the constant image is that constant
    Tr = None
    for it in range(36):
        final = it == 35
        if it > 0:                                           # column pass over the row-major copies -> u, d in column-major
            Dc = np.full_like(Yf, np.nan)
            Uc = lane(emu, 4 if final else 3, Tr, Yr, Tr, N, M, N, 0.2, clen=32, halo=16, X2=None if final else Dc)[0]
        if final:
            out = lane(emu, 0, Uc, None, None, M, N, M, 0.2, clen=32, halo=16)[0]
        else:                                                # row pass over the column-major arrays -> t' in row-major
            Tr = lane(emu, 5, Uc, Dc, None, M, N, M, 0.2, clen=32, halo=16)[0]
    got = out.reshape(N, M).T
    assert np.abs(got - want).max() / np.abs(want).max() <= 1e-9
    assert np.array_equal(got, staged)                       # same arithmetic, other data movement: bit-identical


def test_chunk_and_task_plans(emu):
    """ChunkPlan: boundaries start at 0, end at n, strictly increase, fall on the feed's tile rows, every chunk owns at least two tile
    rows more than its halo costs, cold starts are aligned and never negative, and the work (owned rows + halo) is balanced to within
    one tile row.  TaskPlan: task index -> (group, chunk) is a bijection, also when the last groups have one chunk fewer."""
    rng = np.random.default_rng(11)
    for _ in range(3000):
        gran = int(rng.choice([8, 16, 32])); halo = gran * int(rng.integers(0, 5)); n = int(rng.integers(1, 20000)); want = int(rng.integers(1, 80))
        cs = (C.c_int * 128)(); p0 = (C.c_int * 128)()
        nc = emu.emu_plan(n, want, halo, gran, cs, p0)
        assert 1 <= nc <= want, (n, want, halo, gran, nc)
        b = [cs[c] for c in range(nc + 1)]
        assert b[0] == 0 and b[-1] == n and all(x < y for x, y in zip(b, b[1:])), (n, want, halo, gran, b)
        assert all(x % gran == 0 for x in b[:-1])
        if nc > 1:
            work = [b[1]] + [b[c + 1] - b[c] + halo for c in range(1, nc)]
            assert max(work) - min(work) <= 2 * gran, (n, nc, halo, gran, work)      # rounding moves a boundary by less than one tile row
            assert min(b[c + 1] - b[c] for c in range(nc)) >= gran
        for c in range(nc):
            assert p0[c] == max(0, b[c] - halo) and p0[c] % gran == 0
    for nmax, gfull, groups in ((1, 7, 7), (14, 112, 128), (13, 128, 128), (2, 0, 5), (3, 5, 5), (9, 1, 1000)):
        want = gfull * nmax + (groups - gfull) * (nmax - 1)
        assert emu.emu_taskplan(nmax, gfull, groups) == want


def test_transposed_result_ops(emu, port):
    """Ops that write fiber-major (transposed) results, one by one against the plain pass: 6 (plain), 5 (B + x), 4 (B - (C - x)),
    3 (two results), on strided fibers with a partial last group and chunked fibers."""
    rng = np.random.default_rng(8)
    M, N = 72, 90                                            # fibers = rows of the column-major M x N image: nf = M, len = N, inc = M
    A = np.asfortranarray(rng.normal(0, 1, (M, N))).ravel("F"); Bv = rng.normal(0, 1, M * N); Cv = rng.normal(0, 1, M * N)
    x = lane(emu, 0, A, None, None, M, N, M, 0.3, clen=32, halo=16)[0]
    T = lambda v: v.reshape(N, M).T.copy().ravel()           # position (row r of fiber f) -> f * N + r
    assert np.array_equal(lane(emu, 6, A, None, None, M, N, M, 0.3, clen=32, halo=16)[0], T(x))
    assert np.array_equal(lane(emu, 5, A, Bv, None, M, N, M, 0.3, clen=32, halo=16)[0], T(Bv + x))
    assert np.array_equal(lane(emu, 4, A, Bv, Cv, M, N, M, 0.3, clen=32, halo=16)[0], T(Bv - (Cv - x)))
    X2 = np.full_like(A, np.nan)
    u = lane(emu, 3, A, Bv, Cv, M, N, M, 0.3, clen=32, halo=16, X2=X2)[0]
    d = Cv - x
    assert np.array_equal(X2, T(d)) and np.array_equal(u, T(Bv - (2.0 * d - Cv)))
