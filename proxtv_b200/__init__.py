"""proxtv_b200 -- B200-native Total-Variation (TV-L1) proximity operators behind proxTV's Python surface.

Drop-in for the hot path of ``prox_tv`` (reference: prox_tv/__init__.py): ``tv1_1d`` (:124), ``tv1w_1d`` (:218),
``tv1_2d`` (:355) and ``tvgen`` (:533) keep the reference's names, argument meaning, dtype/layout coercion, assertion
behaviour and return conventions; the computation runs in hand-written sm_100a CUDA kernels reached through the C ABI of
``libproxtv_b200.so`` (include/proxtv_b200.h).  There is NO CPU fallback: without the built extension or a CUDA
device the calls raise.

Extensions the reference lacks (SURVEY.md section 8b): a leading batch dimension (``tv1_1d_batched``,
``tv1w_1d_batched``, ``tv1_2d_batched``), float32, and torch CUDA tensors as inputs (device-resident path: no PCIe
traffic, no host transposes -- a C-ordered tensor is handled by swapping the kernels' stride roles).
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import ProxTVError, load, require_device  # noqa: F401

__all__ = ["tv1_1d", "tv1w_1d", "tv1_2d", "tv1w_2d", "tvgen", "tvgen_pdr", "tv1_1d_batched", "tv1w_1d_batched", "tv1_2d_batched",
           "set_engine", "set_pinned_results", "ProxTVError"]

_N_INFO = 3                      # prox_tv/__init__.py:67
ENGINES = {"auto": 0, "seq": 1, "chunked": 2, "chunked-strided": 3, "pipelined": 4, "tspace": 5, "tpose": 6, "lane": 7, "lane-t": 8}


def set_engine(name):
    """Select the kernel family / DR schedule ('auto' | 'seq' | 'chunked' | 'chunked-strided' | 'pipelined' | 'tspace' |
    'tpose', see include/proxtv_b200.h); returns the previous one.  Only measurements and tests need this."""
    prev = load().proxtv_set_engine(ENGINES[name])
    return [k for k, v in ENGINES.items() if v == prev][0]


# ---- argument coercion, as the reference does it (prox_tv/__init__.py:80-121) ----
def force_float_scalar(x):
    return x if isinstance(x, float) else float(x)


def force_float_matrix(x):
    if not isinstance(x, np.ndarray):
        try:
            x = np.array(x)
        except Exception:
            raise TypeError("Input must be a numpy matrix or compatible object")
    if x.dtype != np.dtype("float64"):
        return x.astype("float")
    return x


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def _is_torch(x):
    return type(x).__module__.startswith("torch") and hasattr(x, "data_ptr")


def _check(ok, what):
    if not ok:
        raise ProxTVError("%s failed: %s" % (what, _lib.last_error()))


# ---- result arrays in pooled page-locked memory ----
# The reference returns a fresh ``np.zeros`` array.  For a 128 MiB image that costs more than the solve: 32768 page faults when the
# device-to-host copy first touches the pages, and a pageable copy at a fraction of the PCIe rate.  Large results are therefore
# carved out of a small pool of page-locked blocks (cudaHostAlloc through the library); a block returns to the pool when the last
# array that refers to it -- the result or any view of it -- is garbage-collected.  ``set_pinned_results(False)`` switches it off.
class _PinnedPool:
    MIN_BYTES = 1 << 20          # smaller results: plain numpy memory
    MAX_IDLE = 1 << 30           # idle blocks kept for reuse (bytes)

    def __init__(self):
        self.enabled = True
        self.free = []           # (capacity, address)

    def empty(self, shape, dtype, order):
        import weakref
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
        if not self.enabled or nbytes < self.MIN_BYTES:
            return np.zeros(shape, dtype=dtype, order=order)
        lib = load()
        fit = [b for b in self.free if nbytes <= b[0] <= 2 * nbytes]
        if fit:
            blk = min(fit); self.free.remove(blk)
        else:
            addr = lib.proxtv_host_alloc(nbytes)
            if not addr:
                return np.zeros(shape, dtype=dtype, order=order)
            blk = (nbytes, addr)
        buf = (C.c_char * nbytes).from_address(blk[1])
        weakref.finalize(buf, self._give, blk)
        return np.frombuffer(buf, dtype=dtype).reshape(shape, order=order)

    def _give(self, blk):
        try:
            if self.enabled and sum(b[0] for b in self.free) + blk[0] <= self.MAX_IDLE:
                self.free.append(blk)
            else:
                load().proxtv_host_free(C.c_void_p(blk[1]))
        except Exception:        # interpreter shutdown
            pass

    def clear(self):
        lib = load()
        for b in self.free:
            lib.proxtv_host_free(C.c_void_p(b[1]))
        self.free = []


_pool = _PinnedPool()


def set_pinned_results(on):
    """Results of at least 1 MiB come from a pool of page-locked host blocks (default: on); returns the previous setting."""
    prev = _pool.enabled
    _pool.enabled = bool(on)
    if not on:
        _pool.clear()
    return prev


# ======================================================================================================================
# 1D
# ======================================================================================================================
_TV1_METHODS = ("classictautstring", "linearizedtautstring", "hybridtautstring", "pn", "condat", "dp",
                "condattautstring", "kolmogorov")      # prox_tv/__init__.py:163-172


def tv1_1d(x, w, method="hybridtautstring", sigma=0.05, maxbacktracks=None):
    r"""1D TV-L1 prox: argmin_y 0.5||x-y||^2 + w sum_i |y_i - y_{i+1}|   (prox_tv/__init__.py:124-178).

    Every ``method`` of the reference computes the same unique minimiser; here they all run the exact linearized
    taut-string scan on the GPU (bit-identical to the reference's 'linearizedtautstring' and, whenever its backtracking
    budget is not exhausted, to its default 'hybridtautstring').  ``sigma`` / ``maxbacktracks`` are accepted and ignored.
    Returns a flat float64 array of ``np.size(x)`` elements, like the reference.
    """
    assert method in _TV1_METHODS
    assert w >= 0
    w = force_float_scalar(w)
    x = force_float_matrix(x)
    y = np.zeros(np.size(x))
    if x.size:
        lib = require_device()
        xin = x if x.flags.c_contiguous or x.flags.f_contiguous else np.ascontiguousarray(x)
        _check(lib.proxtv_prox_fibers_f64(_ptr(xin), _ptr(y), 1, int(np.size(x)), 1, w, None), "tv1_1d")
    return y


def tv1w_1d(x, w, method="tautstring", sigma=0.05):
    r"""Weighted 1D TV-L1 prox: argmin_y 0.5||x-y||^2 + sum_i w_i |y_i - y_{i+1}|   (prox_tv/__init__.py:218-254).

    Both reference methods ('tautstring', 'pn') compute the same minimiser; the GPU path is the weighted taut-string
    scan, bit-identical to the reference's 'tautstring'.
    """
    assert np.all(w >= 0)
    assert np.size(x) - 1 == np.size(w)
    w = force_float_matrix(w)
    x = force_float_matrix(x)
    y = np.zeros(np.size(x))
    n = int(np.size(x))
    if n == 1:
        y[0] = x.ravel()[0]
    elif n > 1:
        lib = require_device()
        _check(lib.proxtv_prox_fibers_f64(_ptr(np.ascontiguousarray(x)), _ptr(y), 1, n, 1, 0.0,
                                          _ptr(np.ascontiguousarray(w))), "tv1w_1d")
    return y


def _batched_1d(x, w, weights):
    """x: (B, L) numpy array or torch CUDA tensor, row-contiguous signals."""
    if _is_torch(x):
        import torch
        assert x.is_cuda and x.dim() == 2
        xt = x.contiguous()
        f32 = xt.dtype == torch.float32
        if not f32 and xt.dtype != torch.float64:
            xt = xt.double()
        out = torch.empty_like(xt)
        B, L = xt.shape
        wt = None
        if weights is not None:
            wt = weights.to(dtype=xt.dtype, device=xt.device).contiguous()
            assert tuple(wt.shape) == (B, L - 1)
        lib = require_device()
        st = C.c_void_p(torch.cuda.current_stream(xt.device).cuda_stream)
        fn = lib.proxtv_prox_fibers_dev_f32 if f32 else lib.proxtv_prox_fibers_dev_f64
        with torch.cuda.device(xt.device):
            _check(fn(C.c_void_p(xt.data_ptr()), C.c_void_p(out.data_ptr()), B, L, 1, float(w),
                      C.c_void_p(wt.data_ptr()) if wt is not None else None, st), "batched 1D prox")
        return out
    x = np.asarray(x)
    assert x.ndim == 2
    f32 = x.dtype == np.float32
    x = np.ascontiguousarray(x, dtype=np.float32 if f32 else np.float64)
    B, L = x.shape
    out = np.empty_like(x)
    wv = None
    if weights is not None:
        wv = np.ascontiguousarray(weights, dtype=x.dtype)
        assert wv.shape == (B, L - 1)
        assert np.all(wv >= 0)
    if x.size:
        lib = require_device()
        fn = lib.proxtv_prox_fibers_f32 if f32 else lib.proxtv_prox_fibers_f64
        _check(fn(_ptr(x), _ptr(out), B, L, 1, float(w), _ptr(wv) if wv is not None else None), "batched 1D prox")
    return out


def tv1_1d_batched(x, w):
    """``tv1_1d`` on every row of a (B, L) array (numpy float64/float32, or a torch CUDA tensor).

    With at least 1024 rows of at least 64 samples (and, under engine 'auto', a penalty the lane engine's guard accepts) the
    rows run on the lane engine: the result is then the slope-form taut-string scan, within ~4e-15 of ``tv1_1d`` but not
    bit-identical to it.  ``set_engine('chunked')`` restores bit-identity with ``tv1_1d``.
    """
    assert w >= 0
    return _batched_1d(x, float(w), None)


def tv1w_1d_batched(x, w):
    """``tv1w_1d`` on every row of x (B, L) with per-edge weights w (B, L-1)  -- BASELINE config 3."""
    return _batched_1d(x, 0.0, w)


# ======================================================================================================================
# 2D
# ======================================================================================================================
_TV1_2D_METHODS = ("yang", "dr", "pd", "kolmogorov", "condat", "chambolle-pock", "chambolle-pock-acc")  # :391-399


def tv1_2d(x, w, n_threads=1, max_iters=0, method="dr"):
    r"""2D anisotropic TV-L1 prox (prox_tv/__init__.py:355-416).

    ``method='dr'`` (default) reproduces the reference's DR2_TV iteration exactly (35 fixed iterations unless
    ``max_iters`` > 0 -- NOT a converged solve, see SURVEY.md section 0.3); ``'pd'`` reproduces PD2_TV.  The other
    reference methods are slower CPU baselines for the same problem and are not provided.  ``n_threads`` is ignored.
    numpy input: returns a Fortran-ordered float64 array like the reference.  torch CUDA tensor input (2D, float64 or
    float32): stays on the device and returns a tensor of the same dtype/layout.
    """
    assert w >= 0
    assert method in _TV1_2D_METHODS
    if method not in ("dr", "pd"):
        raise NotImplementedError("proxtv_b200 implements the 'dr' and 'pd' 2D solvers (the GPU hot path); got %r" % method)
    if _is_torch(x):
        assert method == "dr", "torch path implements the DR solver"
        return _dr2_torch(x, float(w), max_iters, batched=False)
    x = np.asfortranarray(x, dtype="float64")
    assert x.ndim == 2
    w = force_float_scalar(w)
    lib = require_device()
    y = _pool.empty(x.shape, np.float64, "F")
    info = np.zeros(_N_INFO)
    if method == "dr":
        lib.DR2_TV(x.shape[0], x.shape[1], _ptr(x), w, w, 1.0, 1.0, _ptr(y), int(n_threads), int(max_iters), _ptr(info))
        _check(info[2] != 3, "DR2_TV")
    else:
        lam = np.array([w, w]); norms = np.array([1.0, 1.0]); dims = np.array([1.0, 2.0])
        ns = np.array(x.shape, dtype=np.int32)
        ok = lib.PD2_TV(_ptr(x), _ptr(lam), _ptr(norms), _ptr(dims), _ptr(y), _ptr(info), _ptr(ns), 2, 2,
                        int(n_threads), int(max_iters))
        _check(ok and info[2] != 3, "PD2_TV")
    return y


def tv1w_2d(x, w_col, w_row, max_iters=0, n_threads=1):
    r"""2D weighted anisotropic TV-L1 prox by Douglas-Rachford splitting (prox_tv/__init__.py:445-481 -> DR2L1W_TV).

    ``w_col``: (M-1, N) weights of the differences along columns, ``w_row``: (M, N-1) along rows.  Same fixed-iteration
    scheme as ``tv1_2d(method='dr')`` (35 iterations unless ``max_iters`` > 0).  ``n_threads`` is ignored.
    numpy input: Fortran-ordered float64 result like the reference.  torch CUDA tensors (float64 / float32, all three on
    the same device): computed on the device, returns a tensor shaped and typed like ``x``.
    """
    if _is_torch(x):
        return _drw_torch(x, w_col, w_row, max_iters)
    assert np.all(np.asarray(w_col) >= 0)
    assert np.all(np.asarray(w_row) >= 0)
    M, N = np.shape(x)
    assert np.shape(w_col) == (M - 1, N)
    assert np.shape(w_row) == (M, N - 1)
    x = np.asfortranarray(x, dtype="float64")
    y = _pool.empty(x.shape, np.float64, "F")
    w_col = np.asfortranarray(w_col, dtype="float64")
    w_row = np.asfortranarray(w_row, dtype="float64")
    info = np.zeros(_N_INFO)
    lib = require_device()
    lib.DR2L1W_TV(M, N, _ptr(x), _ptr(w_col), _ptr(w_row), _ptr(y), int(n_threads), int(max_iters), _ptr(info))
    _check(info[2] != 3, "DR2L1W_TV")
    return y


def _drw_torch(x, w_col, w_row, max_iters):
    import torch
    assert x.is_cuda and x.dtype in (torch.float64, torch.float32) and x.dim() == 2
    M, N = int(x.shape[0]), int(x.shape[1])
    assert tuple(w_col.shape) == (M - 1, N) and tuple(w_row.shape) == (M, N - 1)
    # the solver works on column-major arrays == the row-major storage of the transposes
    xt = x.t().contiguous()
    w1 = w_col.to(device=x.device, dtype=x.dtype).t().contiguous()
    w2 = w_row.to(device=x.device, dtype=x.dtype).t().contiguous()
    out = torch.empty_like(xt)
    info = np.zeros(_N_INFO)
    lib = require_device()
    st = C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
    fn = lib.proxtv_DR2L1W_TV_dev_f32 if x.dtype == torch.float32 else lib.proxtv_DR2L1W_TV_dev_f64
    with torch.cuda.device(x.device):
        fn(M, N, C.c_void_p(xt.data_ptr()), C.c_void_p(w1.data_ptr()), C.c_void_p(w2.data_ptr()), C.c_void_p(out.data_ptr()),
           int(max_iters), _ptr(info), st)
    _check(info[2] != 3, "DR2L1W_TV (device)")
    return out.t()


def _dr2_torch(x, w, max_iters, batched):
    import torch
    assert x.is_cuda and x.dtype in (torch.float64, torch.float32)
    assert x.dim() == (3 if batched else 2)
    M, N = int(x.shape[-2]), int(x.shape[-1])
    batch = int(x.shape[0]) if batched else 1
    # accept either memory order of the trailing two dims without copying
    if x.stride(-1) == 1 and x.stride(-2) == N and (not batched or x.stride(0) == M * N):
        row_major, xin = 1, x
    elif x.stride(-2) == 1 and x.stride(-1) == M and (not batched or x.stride(0) == M * N):
        row_major, xin = 0, x
    else:
        row_major, xin = 1, x.contiguous()
    out = torch.empty_strided(xin.shape, xin.stride(), dtype=xin.dtype, device=xin.device)
    info = np.zeros(_N_INFO)
    lib = require_device()
    st = C.c_void_p(torch.cuda.current_stream(xin.device).cuda_stream)
    fn = lib.proxtv_DR2_TV_dev_f32 if xin.dtype == torch.float32 else lib.proxtv_DR2_TV_dev_f64
    with torch.cuda.device(xin.device):
        fn(M, N, batch, row_major, C.c_void_p(xin.data_ptr()), w, w, C.c_void_p(out.data_ptr()), int(max_iters),
           _ptr(info), st)
    _check(info[2] != 3, "DR2_TV (device)")
    return out


def tv1_2d_batched(x, w, max_iters=0):
    """``tv1_2d(method='dr')`` on every image of x (B, H, W)  -- BASELINE config 5.

    numpy: float64 or float32, C-ordered (B, H, W); torch: CUDA tensor (B, H, W).  Each image is solved independently with
    exactly the single-image iteration (its own 2*mean initialisation).
    """
    assert w >= 0
    if _is_torch(x):
        return _dr2_torch(x, float(w), max_iters, batched=True)
    x = np.asarray(x)
    assert x.ndim == 3
    f32 = x.dtype == np.float32
    B, H, W = x.shape
    # device layout: column-major images back to back == C-ordered (B, W, H) array of transposed images
    xt = np.ascontiguousarray(np.transpose(x, (0, 2, 1)), dtype=np.float32 if f32 else np.float64)
    out = _pool.empty(xt.shape, xt.dtype, "C")
    info = np.zeros(_N_INFO)
    lib = require_device()
    fn = lib.proxtv_DR2_TV_batched_f32 if f32 else lib.proxtv_DR2_TV_batched_f64
    fn(H, W, B, _ptr(xt), float(w), float(w), _ptr(out), int(max_iters), _ptr(info))
    _check(info[2] != 3, "DR2_TV (batched)")
    return np.transpose(out, (0, 2, 1))


# ======================================================================================================================
# ND
# ======================================================================================================================
def tvgen(x, ws, ds, ps, n_threads=1, max_iters=0):
    r"""General ND TV prox with one 1D TV-L1 term per entry of (ws, ds, ps)   (prox_tv/__init__.py:533-600).

    Dispatch follows the reference, including its quirks: the DR2_TV branch of the reference is dead code
    (``len(ds) == 2 & ds[0] == 1 & ds[1] == 2`` is always False, :585), so two terms go to PD2_TV and anything else to
    PD_TV.  PD_TV scales the caller's ``ws`` by ``len(ws)`` IN PLACE when ``ws`` is a float64 ndarray (:576 does not
    copy in that case; src/TVNDopt.cpp:100-101).  Only p = 1 norms are implemented on the GPU path.
    Extension: a float32 ``x`` is solved in float32 (the reference would upcast) when ``len(ws) != 2``.
    """
    assert len(ws) == len(ds)
    assert len(ws) == len(ps)
    assert n_threads >= 1
    assert max_iters >= 0
    info = np.zeros(_N_INFO)
    f32 = isinstance(x, np.ndarray) and x.dtype == np.float32 and len(ws) != 2
    x = np.asfortranarray(x, dtype="float32" if f32 else "float64")
    ws = force_float_matrix(ws)
    ps = force_float_matrix(ps)
    y = _pool.empty(np.shape(x), x.dtype, "F")
    if np.any(ps != 1):
        raise NotImplementedError("proxtv_b200 implements TV-L1 (p = 1) penalty terms only")
    lib = require_device()
    dsa = np.array(ds, dtype=np.float64)
    ns = np.array(x.shape, dtype=np.int32)
    if len(ws) == 2:
        ok = lib.PD2_TV(_ptr(x), _ptr(ws), _ptr(ps), _ptr(dsa), _ptr(y), _ptr(info), _ptr(ns), x.ndim, 2,
                        int(n_threads), int(max_iters))
    elif f32:
        ok = lib.proxtv_PD_TV_f32(_ptr(x), _ptr(ws), _ptr(dsa), _ptr(y), _ptr(info), _ptr(ns), x.ndim, len(ws),
                                  int(max_iters))
    else:
        ok = lib.PD_TV(_ptr(x), _ptr(ws), _ptr(ps), _ptr(dsa), _ptr(y), _ptr(info), _ptr(ns), x.ndim, len(ws),
                       int(n_threads), int(max_iters))
    _check(ok and info[2] != 3, "tvgen")
    tvgen.last_info = info
    return y


tvgen.last_info = None


def tvgen_pdr(x, ws, ds, ps, n_threads=1, max_iters=0):
    r"""The same generalized TV prox as ``tvgen`` solved with the reference's Parallel Douglas-Rachford splitting, ``PDR_TV``
    (src/TVNDopt.cpp:280-500; reached from MATLAB only in the reference, matlab/solveTVND_PDR.cpp:89 -- SURVEY.md 8f N4).

    Runs exactly ``max_iters`` iterations (0: 35; the reference's loop has no stop test) and, like PD_TV, scales a float64
    ndarray ``ws`` by ``len(ws)`` IN PLACE.  float64 only from numpy (use the C ABI's ``proxtv_PDR_TV_dev_f32`` for float32
    device arrays); p = 1 norms only.  ``tvgen_pdr.last_info`` = [iterations, mean|x - x_last|, RC].
    """
    assert len(ws) == len(ds)
    assert len(ws) == len(ps)
    assert n_threads >= 1
    assert max_iters >= 0
    info = np.zeros(_N_INFO)
    x = np.asfortranarray(x, dtype="float64")
    ws = force_float_matrix(ws)
    ps = force_float_matrix(ps)
    if np.any(ps != 1):
        raise NotImplementedError("proxtv_b200 implements TV-L1 (p = 1) penalty terms only")
    y = _pool.empty(np.shape(x), x.dtype, "F")
    lib = require_device()
    dsa = np.array(ds, dtype=np.float64)
    ns = np.array(x.shape, dtype=np.int32)
    ok = lib.PDR_TV(_ptr(x), _ptr(ws), _ptr(ps), _ptr(dsa), _ptr(y), _ptr(info), _ptr(ns), x.ndim, len(ws), int(n_threads), int(max_iters))
    _check(ok and info[2] != 3, "tvgen_pdr")
    tvgen_pdr.last_info = info
    return y


tvgen_pdr.last_info = None
