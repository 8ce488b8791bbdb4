"""GPU tests (-m gpu) of the lane engine's CUDA kernel (kernels_lane.cu), pass by pass, BIT FOR BIT.

Reference: the plain sequential slope-form scan of one fiber (emu_slope_seq_f64 of tests/emu/emu_lane.cu, compiled from
lane_core.cuh) with the pass's fused arithmetic (PassOp, kernels_lane.cu) composed around it in numpy, in the storage type and
with PassOp's association.  Every chunk of the lane engine either verifies or is repaired into exactly the sequential scan's state
(DESIGN.md section 3), and both sides are built without FMA contraction, so the kernel must reproduce that scan exactly -- for
every op, layout, storage type, chunk plan, tuning variant and data set.  float32 storage: the scan runs in float64 on the
float32 input and rounds its result once, so the reference is seq_f64(in.astype(f64), float(np.float32(lam))).astype(float32)
and all arithmetic around it is float32.

Because that reference shares lane_core.cuh with the kernel, every plain (op 0) case is also checked independently: the dual
certificate of the TV prox in extended precision, and the oracle's linearized taut string within 1e-12 relative with the same
jump sets.  Whole Douglas-Rachford solves are composed from the reference passes on inputs whose 2 * mean is exact in any
summation order, and must match bit for bit as well.

Every device array is an interior, 16-byte aligned view of a larger buffer whose margins hold a NaN canary; margins, inputs and
operands must come back unchanged, and result arrays start as canary so that an element the kernel does not write fails.
"""
import ctypes as C

import numpy as np
import pytest

from emu import lane_emu
from oracle import oracle as O

pytestmark = pytest.mark.gpu
vp = C.c_void_p
MARGIN = 512                                              # canary elements on each side of every device array (2 / 4 KB)
CANARY = {np.float64: np.uint64(0x7FF8DEADBEEF0001), np.float32: np.uint32(0x7FC0BEEF)}
LENGTHS = (2, 6, 7, 8, 14, 16, 18, 62, 63, 64, 65, 66, 129, 130, 1000)
LAMS = (1e-6, 0.2, 5.0, 1e4)
KINDS = ("cfg2", "noise", "const", "plateau", "alt", "int")


@pytest.fixture(scope="module")
def emu():
    return lane_emu.load(required=True)


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


@pytest.fixture
def lib(ptv):
    """The library, with the lane tuning and the engine restored to their defaults after the test (PTV_LANE_VARIANT is assumed unset)."""
    lib = ptv.load()
    lib.proxtv_lane_stats(1)
    prev = ptv.set_engine("auto")
    try:
        yield lib
    finally:
        lib.proxtv_lane_tuning(0, 32, -1)
        ptv.set_engine(prev)


# ---------------------------------------------------------------- layouts
def fibers_of(a, nf, ln, inc):
    """Flat array in a pass's own layout -> (nf, ln), fiber-major.  STRIDED: element (slab s, fiber i, row r) at s*inc*ln + r*inc + i."""
    if inc == 1:
        return a.reshape(nf, ln)
    return a.reshape(nf // inc, ln, inc).transpose(0, 2, 1).reshape(nf, ln)


def own_layout(F, nf, ln, inc):
    """(nf, ln) fiber-major -> flat array in the pass's own layout."""
    if inc == 1:
        return np.ascontiguousarray(F).ravel()
    return np.ascontiguousarray(F.reshape(nf // inc, inc, ln).transpose(0, 2, 1)).ravel()


def pitch_ok(dtype, ln, inc, op):
    sz = np.dtype(dtype).itemsize
    if (ln if inc == 1 else inc) * sz % 16:
        return False
    return op < 3 or ln * sz % 16 == 0


# ---------------------------------------------------------------- reference
def seq(emu, F, lam):
    """Sequential slope-form scan of every row of F (nf, ln); returns (result in F's dtype, the float64 scan values)."""
    F64 = np.ascontiguousarray(F, dtype=np.float64)
    X = np.empty_like(F64)
    lam64 = float(np.float32(lam)) if F.dtype == np.float32 else float(lam)
    emu.emu_slope_seq_rows_f64(F64.ctypes.data_as(lane_emu.dp), F64.shape[0], F64.shape[1], lam64, X.ctypes.data_as(lane_emu.dp))
    return X.astype(F.dtype), X


def ref_pass(emu, op, A, B, Cc, nf, ln, inc, lam):
    """What pass `op` must write: (X, X2 or None, scan input (nf, ln), float64 scan values (nf, ln)).  PassOp's forms and association."""
    T = A.dtype.type
    fa = fibers_of(A, nf, ln, inc)
    fb = fibers_of(B, nf, ln, inc) if B is not None else None
    fc = fibers_of(Cc, nf, ln, inc) if Cc is not None else None
    if op == 1:
        d = fc - fb
        inp = fa - (T(2) * d - fc)
    elif op == 2:
        inp = fa - (fc - fb)
    else:
        inp = fa
    x, x64 = seq(emu, inp, lam)
    o2 = None
    if op == 1:
        o = (fc - fb) + x
    elif op == 3:
        d = fc - x
        o, o2 = fb - (T(2) * d - fc), d
    elif op == 4:
        o = fb - (fc - x)
    elif op == 5:
        o = fb + x
    else:
        o = x
    if op <= 2:                                           # results in the pass's own layout; ops 3-6 write them fiber-major
        o = own_layout(o, nf, ln, inc)
    return o.ravel(), (o2.ravel() if o2 is not None else None), inp, x64


def ulps(a, b):
    ia = np.asarray(a).view(np.int64 if a.dtype == np.float64 else np.int32).astype(np.int64)
    ib = np.asarray(b).view(np.int64 if b.dtype == np.float64 else np.int32).astype(np.int64)
    top = np.int64(-(1 << 63)) if a.dtype == np.float64 else np.int64(-(1 << 31))
    oa = np.where(ia < 0, top - ia, ia); ob = np.where(ib < 0, top - ib, ib)
    return np.abs(oa - ob)


def assert_bits(got, want, nf, ln, what):
    """Bit-for-bit equality of two fiber-major (nf, ln) results; on a mismatch name the fiber, the first row and the ulps."""
    if np.array_equal(got, want):
        return
    G = got.reshape(nf, ln); W = want.reshape(nf, ln)
    bad = ~((G == W) | (np.isnan(G) & np.isnan(W)))
    j = int(np.nonzero(bad.any(axis=1))[0][0]); r = int(np.nonzero(bad[j])[0][0])
    raise AssertionError("%s: %d of %d elements differ; first: fiber %d row %d got %r want %r (%s ulp)"
                         % (what, int(bad.sum()), bad.size, j, r, G[j, r], W[j, r],
                            "nan" if np.isnan(G[j, r]) else int(ulps(G[j, r:r + 1], W[j, r:r + 1])[0])))


def check_independent(port, Y, X64, lam, what):
    """Op-0 checks that do not rest on lane_core.cuh.  Y: scan input, X64: float64 scan values, both (nf, ln).
    Both taut-string forms add and subtract 2 lam to running sums of y, so their rounding scales with s = max(|y|, |x|, lam) per
    fiber, and a segment of k samples carries at most ~k eps s of it per sample.
    (a) the dual certificate in extended precision: S_k = sum_{i<=k} (y_i - x_i) satisfies |S_k| <= lam, S_{n-1} = 0, and
        S_k = -lam sign(x_{k+1} - x_k) at every jump, each up to tiny = 4 eps s sum(k^2) over the fiber's segments;
    (b) the oracle's linearized taut string (the reference's own form) within 1e-12 s, and the same jump sets at the suite's
        1e-9 threshold (scaled by max|y| for data above unit scale, where 1e-9 is below the rounding of the values)."""
    Y = np.asarray(Y, dtype=np.float64)
    nf, ln = Y.shape
    scale = np.maximum(np.maximum(np.abs(Y).max(axis=1), np.abs(X64).max(axis=1)), lam)
    dx = np.diff(X64, axis=1)
    seg2 = np.empty(nf)
    for j in range(nf):
        b = np.concatenate(([0], np.nonzero(dx[j])[0] + 1, [ln]))
        seg2[j] = float((np.diff(b).astype(np.float64) ** 2).sum())
    tiny = (4 * np.finfo(np.float64).eps * scale * seg2)[:, None]
    S = np.cumsum(Y.astype(np.longdouble) - X64.astype(np.longdouble), axis=1)
    assert np.all(np.abs(S[:, :-1]) <= lam * (1 + 1e-12) + tiny), (what, "dual certificate: |S_k| > lam")
    assert np.all(np.abs(S[:, -1:]) <= tiny), (what, "dual certificate: S_{n-1} != 0")
    at_jump = np.abs(S[:, :-1] + lam * np.sign(dx)) <= lam * 1e-12 + tiny
    assert np.all(at_jump | (dx == 0)), (what, "dual certificate at a jump")
    for j in range(nf):
        w = port.tv1_linearized(Y[j], float(lam))
        assert np.abs(X64[j] - w).max() <= 1e-12 * scale[j], (what, j, "linearized taut string")
        thr = 1e-9 * max(1.0, np.abs(Y[j]).max())
        assert np.array_equal(np.nonzero(np.abs(dx[j]) > thr)[0], np.nonzero(np.abs(np.diff(w)) > thr)[0]), (what, j, "jump set")


# ---------------------------------------------------------------- device side
class Buf:
    """Interior view of a larger device buffer whose margins (and, unless `data` is given, interior) hold the NaN canary."""
    def __init__(self, torch, n, dtype, data=None, offset=0):
        self.dtype = np.dtype(dtype)
        self.itype = torch.int64 if self.dtype == np.float64 else torch.int32
        self.canary = CANARY[self.dtype.type]
        self.store = torch.empty(n + 2 * MARGIN + offset, dtype=torch.float64 if self.dtype == np.float64 else torch.float32, device="cuda")
        self.store.view(self.itype).fill_(int(self.canary.view(np.int64 if self.dtype == np.float64 else np.int32)))
        self.lo, self.n = MARGIN + offset, n
        self.t = self.store[self.lo:self.lo + n]
        self.init = None
        if data is not None:
            self.init = np.ascontiguousarray(data, dtype=self.dtype).ravel()
            self.t.copy_(torch.from_numpy(self.init))

    def ptr(self):
        return vp(self.t.data_ptr())

    def get(self):
        return self.t.cpu().numpy()

    def check(self, what):
        """Margins still canary; an input still holds its data, bit for bit."""
        s = self.store.cpu().numpy().view(self.canary.dtype)
        assert np.all(s[:self.lo] == self.canary) and np.all(s[self.lo + self.n:] == self.canary), (what, "canary margin overwritten")
        if self.init is not None:
            assert np.array_equal(s[self.lo:self.lo + self.n], self.init.view(self.canary.dtype)), (what, "input or operand modified")


def stream(torch):
    return vp(torch.cuda.current_stream().cuda_stream)


def lane_call(lib, torch, op, bufs, nf, ln, inc, lam):
    """One pass through the C ABI on the current stream; bufs = (A, B, C, X, X2) of Buf or None.  Returns the return code."""
    A, B, Cc, X, X2 = bufs
    f32 = A.dtype == np.float32
    p = lambda b: b.ptr() if b is not None else None       # noqa: E731
    if X2 is not None:
        fn = lib.proxtv_lane_prox2_dev_f32 if f32 else lib.proxtv_lane_prox2_dev_f64
        rc = fn(op, p(A), p(B), p(Cc), p(X), p(X2), nf, ln, inc, float(np.float32(lam)) if f32 else lam, stream(torch))
    else:
        fn = lib.proxtv_lane_prox_dev_f32 if f32 else lib.proxtv_lane_prox_dev_f64
        rc = fn(op, p(A), p(B), p(Cc), p(X), nf, ln, inc, float(np.float32(lam)) if f32 else lam, stream(torch))
    torch.cuda.synchronize()
    return rc


def run_pass(lib, torch, emu, port, op, A, B, Cc, nf, ln, inc, lam, what, independent=True):
    """Run pass `op` on the GPU and hold it bit for bit to the reference (plus the independent checks for op 0).  A, B, C: flat
    arrays in the pass's own layout.  Returns the number of fibers compared."""
    what = "%s op=%d %s nf=%d len=%d inc=%d lam=%g" % (what, op, A.dtype, nf, ln, inc, lam)
    n = nf * ln
    bufs = [Buf(torch, n, A.dtype, A), Buf(torch, n, A.dtype, B) if B is not None else None, Buf(torch, n, A.dtype, Cc) if Cc is not None else None,
            Buf(torch, n, A.dtype), Buf(torch, n, A.dtype) if op == 3 else None]
    rc = lane_call(lib, torch, op, bufs, nf, ln, inc, lam)
    assert rc == 1, (what, lib.proxtv_last_error())
    for b in bufs:
        if b is not None:
            b.check(what)
    want, want2, inp, x64 = ref_pass(emu, op, A, B, Cc, nf, ln, inc, lam)
    tr = (lambda v: v) if op >= 3 else (lambda v: fibers_of(v, nf, ln, inc))
    assert_bits(tr(bufs[3].get()), tr(want), nf, ln, what)
    if op == 3:
        assert_bits(bufs[4].get(), want2, nf, ln, what + " (X2)")
    if op == 0 and independent:
        check_independent(port, inp, x64, float(np.float32(lam)) if A.dtype == np.float32 else lam, what)
    return nf


def make_data(rng, kind, nf, ln, scale=1.0):
    if kind == "cfg2":                                    # blocks of 16 samples + noise (config 2's statistics)
        y = np.repeat(rng.normal(0, 1, (nf, ln // 16 + 1)), 16, axis=1)[:, :ln] + rng.normal(0, 0.3, (nf, ln))
    elif kind == "noise":
        y = rng.normal(0, 1, (nf, ln))
    elif kind == "const":                                 # no break anywhere: every lane retires, every fiber is repaired
        y = np.repeat(rng.normal(0, 1, (nf, 1)), ln, axis=1)
    elif kind == "plateau":                               # a long flat stretch in the middle
        y = rng.normal(0, 1, (nf, ln)); y[:, ln // 4:3 * ln // 4] = 0.3
    elif kind == "alt":                                   # +-1: ties in the slope comparisons
        y = np.where(np.arange(ln) % 2 == 0, 1.0, -1.0)[None, :] * np.ones((nf, 1))
    else:                                                 # integer-valued: ties
        y = np.round(rng.normal(0, 3, (nf, ln)))
    return y * scale


def operands(rng, nf, ln, op, dtype):
    B = rng.normal(0, 1, nf * ln).astype(dtype) if op >= 1 and op != 6 else None
    Cc = rng.normal(0, 1, nf * ln).astype(dtype) if op in (1, 2, 3, 4) else None
    return B, Cc


# ---------------------------------------------------------------- tests
# fiber sets: (fibers per slab, slabs); STRIDED: inc = fibers per slab, nf = slabs * inc (the slab is the TMA map's third coordinate)
STRIDED_SETS = {np.float64: ((32, 1), (64, 1), (34, 1), (40, 2), (32, 3)), np.float32: ((32, 1), (64, 1), (40, 1), (36, 2), (32, 3))}
CONTIG_NF = (1, 32, 40, 64, 97)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_plain_pass_shapes(lib, torch, emu, port, dtype):
    """Op 0 in both layouts at the kernel's edges: full / partial / single groups, 1-3 slabs, lengths around the 8-row tiles of the
    STRIDED feed and the 16 (f64) / 32 (f32) row boxes of the CONTIG feed, odd lengths where the pitch allows them."""
    rng = np.random.default_rng(1)
    cases = 0
    for k, ln in enumerate(LENGTHS):
        for per, slabs in STRIDED_SETS[dtype]:
            if not pitch_ok(dtype, ln, per, 0):
                continue
            nf = per * slabs
            y = make_data(rng, KINDS[(k + per) % len(KINDS)], nf, ln).astype(dtype)
            cases += run_pass(lib, torch, emu, port, 0, own_layout(y, nf, ln, per), None, None, nf, ln, per, LAMS[(k + slabs) % 4], "strided")
        for nf in CONTIG_NF:
            if not pitch_ok(dtype, ln, 1, 0):
                continue
            y = make_data(rng, KINDS[(k + nf) % len(KINDS)], nf, ln).astype(dtype)
            cases += run_pass(lib, torch, emu, port, 0, y.ravel(), None, None, nf, ln, 1, LAMS[(k + nf) % 4], "contig")
    assert cases > 1000


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_fused_ops_strided(lib, torch, emu, port, dtype):
    """Ops 1-6 (STRIDED only): staged input forms 1, 2; drain forms with results written fiber-major 3 (two results), 4, 5, 6."""
    rng = np.random.default_rng(2)
    for op in range(1, 7):
        for k, ln in enumerate((6, 7, 8, 16, 18, 63, 64, 66, 130, 1000)):
            for per, slabs in STRIDED_SETS[dtype]:
                if not pitch_ok(dtype, ln, per, op):
                    continue
                nf = per * slabs
                y = make_data(rng, KINDS[(k + op) % len(KINDS)], nf, ln).astype(dtype)
                B, Cc = operands(rng, nf, ln, op, dtype)
                run_pass(lib, torch, emu, port, op, own_layout(y, nf, ln, per), B, Cc, nf, ln, per, LAMS[(k + per) % 4], "fused")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_data_sets(lib, torch, emu, port, dtype):
    """Every data kind at every penalty and at three scales, in both layouts, with a partial last group and a chunked plan."""
    rng = np.random.default_rng(3)
    per, ln_s = (40, 130) if dtype == np.float64 else (40, 129)
    ln_c = 130 if dtype == np.float64 else 132
    lib.proxtv_lane_tuning(64, 16, -1)
    for kind in KINDS:
        for lam in LAMS:
            for scale in (1.0, 1e8, 1e-8):
                y = make_data(rng, kind, 2 * per, ln_s, scale).astype(dtype)
                run_pass(lib, torch, emu, port, 0, own_layout(y, 2 * per, ln_s, per), None, None, 2 * per, ln_s, per, lam, "data %s x%g" % (kind, scale))
                y = make_data(rng, kind, per, ln_c, scale).astype(dtype)
                run_pass(lib, torch, emu, port, 0, y.ravel(), None, None, per, ln_c, 1, lam, "data %s x%g" % (kind, scale))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_forced_chunks_and_repair(lib, torch, emu, port, dtype):
    """Fixed chunk lengths with halo 0, 8, 16.  Halo 0 puts every chunk boundary through verification, and a cold start exactly at
    a boundary cannot be verified: the GPU repair path must run (and reproduce the sequential scan).  The staged ops 1 and 2
    recompute their scan input from global memory during repair."""
    rng = np.random.default_rng(4)
    nf, ln = 72, 1000
    y = make_data(rng, "cfg2", nf, ln).astype(dtype)
    for clen in (64, 128):
        for halo in (0, 8, 16):
            lib.proxtv_lane_tuning(clen, halo, -1)
            lib.proxtv_lane_stats(1)
            run_pass(lib, torch, emu, port, 0, own_layout(y, nf, ln, 36), None, None, nf, ln, 36, 0.2, "clen=%d halo=%d" % (clen, halo))
            run_pass(lib, torch, emu, port, 0, y.ravel(), None, None, nf, ln, 1, 0.2, "clen=%d halo=%d" % (clen, halo))
            for op in (1, 2):
                B, Cc = operands(rng, nf, ln, op, dtype)
                run_pass(lib, torch, emu, port, op, own_layout(y, nf, ln, 36), B, Cc, nf, ln, 36, 0.2, "clen=%d halo=%d" % (clen, halo))
            reps = lib.proxtv_lane_stats(1)
            if halo == 0:
                assert reps > 0, "halo 0: no fiber went through the GPU repair path"
                print("%s clen=%d halo=0: %d repaired fibers" % (np.dtype(dtype), clen, reps))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("variant", [0, 1, 5, 6, 7])
def test_tuning_variants(lib, torch, emu, port, dtype, variant):
    """Window / epoch / CTA variants (kernels_lane.cu launch_variant), one-wave plan and forced chunks, both layouts, ops 0 and 3."""
    rng = np.random.default_rng(10 + variant)
    ln = 1000
    for clen, halo in ((0, 32), (128, 8)):
        lib.proxtv_lane_tuning(clen, halo, variant)
        y = make_data(rng, "cfg2", 80, ln).astype(dtype)
        run_pass(lib, torch, emu, port, 0, own_layout(y, 80, ln, 40), None, None, 80, ln, 40, 0.2, "variant %d" % variant)
        run_pass(lib, torch, emu, port, 0, y.ravel(), None, None, 80, ln, 1, 0.2, "variant %d" % variant)
        B, Cc = operands(rng, 80, ln, 3, dtype)
        run_pass(lib, torch, emu, port, 3, own_layout(y, 80, ln, 40), B, Cc, 80, ln, 40, 0.2, "variant %d" % variant)
        y = make_data(rng, "const", 40, 200).astype(dtype)                   # every lane retires
        run_pass(lib, torch, emu, port, 0, own_layout(y, 40, 200, 40), None, None, 40, 200, 40, 0.2, "variant %d const" % variant)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_production_plan(lib, torch, emu, port, dtype):
    """One 4096 x 4096 pass at default tuning in each layout (one wave of chunked tasks with halo 32), and a batch of 3 images
    2048 x 2048 (three slabs) with whole fibers (one task per fiber group)."""
    Y = O.gen_cfg2(4096, 4096, seed=11).astype(dtype)                     # column-major: columns contiguous, rows strided
    A = Y.ravel("F")
    run_pass(lib, torch, emu, port, 0, A, None, None, 4096, 4096, 1, 0.2, "4096^2 contig")
    run_pass(lib, torch, emu, port, 0, A, None, None, 4096, 4096, 4096, 0.2, "4096^2 strided")
    if dtype == np.float32:
        lib.proxtv_lane_tuning(2048, 32, -1)                              # whole fibers: one chunk per fiber
        Z = np.concatenate([O.gen_cfg2(2048, 2048, seed=s).astype(dtype).ravel("F") for s in (1, 2, 3)])
        run_pass(lib, torch, emu, port, 0, Z, None, None, 3 * 2048, 2048, 2048, 0.2, "3 x 2048^2 strided")
        run_pass(lib, torch, emu, port, 0, Z, None, None, 3 * 2048, 2048, 1, 0.2, "3 x 2048^2 contig")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_refusals(lib, torch, dtype):
    """Shapes and arguments the engine does not take: return 0, say why, and leave every array untouched."""
    nf, ln = 64, 64
    y = np.random.default_rng(5).normal(0, 1, 80 * ln)          # enough for the largest case
    cases = [("base misaligned by 8 bytes", 0, nf, ln, 32, 0.2, 8 // np.dtype(dtype).itemsize, False),
             ("odd pitch", 0, 33 * 2, ln, 33, 0.2, 0, False),
             ("len < 2", 0, nf, 1, 32, 0.2, 0, False),
             ("lam = 0", 0, nf, ln, 32, 0.0, 0, False),
             ("lam < 0", 0, nf, ln, 32, -0.2, 0, False),
             ("contig with op 1", 1, nf, ln, 1, 0.2, 0, False),
             ("nf % inc != 0", 0, 80, ln, 32, 0.2, 0, False),
             ("op 3 without X2", 3, nf, ln, 32, 0.2, 0, False),
             ("op 3 with a misaligned X2", 3, nf, ln, 32, 0.2, 0, True)]
    if dtype == np.float32:
        cases[1] = ("odd pitch", 0, 34 * 2, ln, 34, 0.2, 0, False)            # 136-byte rows
    for what, op, nf_, ln_, inc, lam, off, bad_x2 in cases:
        n = nf_ * ln_
        bufs = [Buf(torch, n, dtype, y[:n], offset=off), Buf(torch, n, dtype, y[:n]), Buf(torch, n, dtype, y[:n]), Buf(torch, n, dtype, offset=off),
                Buf(torch, n, dtype, offset=8 // np.dtype(dtype).itemsize) if bad_x2 else None]
        rc = lane_call(lib, torch, op, bufs, nf_, ln_, inc, lam)
        assert rc == 0, what
        assert lib.proxtv_last_error().decode(), what
        for b in bufs:
            if b is not None:
                b.check(what)
        assert np.all(bufs[3].store.cpu().numpy().view(bufs[3].canary.dtype) == bufs[3].canary), (what, "X written")


# ---------------------------------------------------------------- whole solves
def dyadic_image(rng, M, N):
    """Multiples of 2^-10 with |y| < 2^8 whose sum is exactly M N c for a dyadic c (a few pixels adjusted by at most 64): 2 * mean
    is then exact in any summation order (ew_image_means_x2 accumulates in double, also for float32 images)."""
    Y = rng.integers(-(1 << 17), 1 << 17, (M, N)).astype(np.float64) / 1024.0
    c = np.round(Y.sum() / Y.size * 1024.0) / 1024.0
    d = c * Y.size - Y.sum()
    k = max(1, int(np.ceil(abs(d) / 64)))
    step = np.trunc(d / k * 1024.0) / 1024.0
    Y.ravel()[:k] += step
    Y[0, 0] += d - step * k
    assert Y.sum() == c * Y.size and np.abs(Y).max() < 256
    return Y


def dr_compose(emu, Y, lam, maxit=35):
    """DR2_TV made of reference passes, as the lane schedules issue them (solver.cu dr2_lane_body / dr2_lane_t_body, the same
    expressions in both): t = 2 mean; x1 = t in the first iteration (the prox of a constant fiber is that constant), else
    prox of the columns of t; d = t - x1; t' = d + prox_rows(Y - (2 d - t)); final: prox_rows(Y - (t - x1))."""
    T = Y.dtype.type
    M, N = Y.shape
    t = np.full((M, N), T(2 * Y.astype(np.float64).sum() / Y.size), dtype=Y.dtype)
    cols = lambda Z: seq(emu, np.ascontiguousarray(Z.T), lam)[0].T          # noqa: E731
    rows = lambda Z: seq(emu, np.ascontiguousarray(Z), lam)[0]               # noqa: E731
    for it in range(maxit + 1):
        x1 = t.copy() if it == 0 else cols(t)
        if it == maxit:
            return rows(Y - (t - x1))
        d = t - x1
        t = d + rows(Y - (T(2) * d - t))


SOLVE_SHAPES = {np.float64: ((96, 80), (130, 66)), np.float32: ((96, 80), (132, 68))}


def test_dr2_lane_schedules_bit_exact(ptv, lib, torch, emu):
    """tv1_2d under 'lane' (staged schedule) and 'lane-t' (transposed schedule) on numpy input; the same solves on torch tensors
    in both memory orders and float32; tv1_2d_batched on row-major tensors: all equal the composition of reference passes."""
    rng = np.random.default_rng(6)
    for dtype in (np.float64, np.float32):
        for M, N in SOLVE_SHAPES[dtype]:
            Y = dyadic_image(rng, M, N).astype(dtype)
            want = dr_compose(emu, Y, 0.2)
            for eng in ("lane", "lane-t"):
                ptv.set_engine(eng)
                if dtype == np.float64:
                    assert_bits(ptv.tv1_2d(Y, 0.2).T.ravel(), want.T.ravel(), N, M, "tv1_2d %s %dx%d" % (eng, M, N))
                tr = torch.tensor(np.ascontiguousarray(Y), device="cuda")                 # row-major: always the transposed schedule
                tc = torch.tensor(np.ascontiguousarray(Y.T), device="cuda").T             # column-major view
                for name, x in (("row-major", tr), ("column-major", tc)):
                    got = ptv.tv1_2d(x, 0.2).cpu().numpy()
                    assert_bits(np.ascontiguousarray(got).ravel(), want.ravel(), M, N, "torch %s %s %s %dx%d" % (dtype.__name__, name, eng, M, N))
        ptv.set_engine("lane")
        M, N = SOLVE_SHAPES[dtype][1]
        imgs = np.stack([dyadic_image(rng, M, N) for _ in range(3)]).astype(dtype)
        got = ptv.tv1_2d_batched(torch.tensor(imgs, device="cuda"), 0.2).cpu().numpy()
        for b in range(3):
            assert_bits(got[b].ravel(), dr_compose(emu, imgs[b], 0.2).ravel(), M, N, "tv1_2d_batched %s image %d" % (dtype.__name__, b))


def test_dr2_chunked_family_bit_exact(ptv, lib, port):
    """The bit-faithful schedules run the reference's own arithmetic: with 2 * mean exact they equal the oracle bit for bit."""
    rng = np.random.default_rng(7)
    for M, N in ((96, 80), (130, 66), (1024, 1026)):
        Y = dyadic_image(rng, M, N)
        want = port.dr2_tv(Y, 0.2)[0]
        for eng in ("chunked", "pipelined", "tspace", "tpose"):
            ptv.set_engine(eng)
            assert_bits(ptv.tv1_2d(Y, 0.2).T.ravel(), want.T.ravel(), N, M, "tv1_2d %s %dx%d" % (eng, M, N))


# ---------------------------------------------------------------- the 1D batched route
def test_prox_fibers_route(ptv, lib, torch, emu, port):
    """tv1_1d_batched with >= 1024 rows of >= 64 samples runs the lane engine under 'auto' (its guard accepts the data): rows equal
    the sequential slope-form scan bit for bit.  proxtv_prox_fibers_f64 with strided fibers likewise.  Under 'chunked' the same
    calls equal the reference's linearized taut string bit for bit."""
    rng = np.random.default_rng(9)
    X = make_data(rng, "cfg2", 2048, 256)
    for dtype in (np.float64, np.float32):
        Xd = X.astype(dtype)
        want = seq(emu, Xd, 0.2)[0]
        for name, fn in (("numpy", lambda a: ptv.tv1_1d_batched(a, 0.2)),
                         ("torch", lambda a: ptv.tv1_1d_batched(torch.tensor(a, device="cuda"), 0.2).cpu().numpy())):
            ptv.set_engine("auto")
            got = fn(Xd)
            assert lib.proxtv_lane_guard_last() == 1, (name, dtype)
            assert_bits(np.ascontiguousarray(got).ravel(), want.ravel(), 2048, 256, "tv1_1d_batched %s %s auto" % (name, dtype.__name__))
            if dtype == np.float64:
                ptv.set_engine("chunked")
                got = fn(Xd)
                for j in range(0, 2048, 61):
                    assert np.array_equal(got[j], port.tv1_linearized(X[j], 0.2)), (name, j)
    # strided fibers: two slabs of 1024 fibers, element (slab s, fiber i, row r) at s*1024*256 + r*1024 + i
    A = own_layout(X, 2048, 256, 1024)
    out = np.full_like(A, np.nan)
    ptv.set_engine("auto")
    assert lib.proxtv_prox_fibers_f64(vp(A.ctypes.data), vp(out.ctypes.data), 2048, 256, 1024, 0.2, None) == 1
    assert lib.proxtv_lane_guard_last() == 1
    assert_bits(fibers_of(out, 2048, 256, 1024).ravel(), seq(emu, X, 0.2)[0].ravel(), 2048, 256, "proxtv_prox_fibers_f64 strided auto")
    ptv.set_engine("chunked")
    assert lib.proxtv_prox_fibers_f64(vp(A.ctypes.data), vp(out.ctypes.data), 2048, 256, 1024, 0.2, None) == 1
    F = fibers_of(out, 2048, 256, 1024)
    for j in range(0, 2048, 61):
        assert np.array_equal(F[j], port.tv1_linearized(X[j], 0.2)), j
