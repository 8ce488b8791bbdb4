// emu_lane.cu -- TEST INFRASTRUCTURE: runs proxtv_b200/csrc/lane_core.cuh (the code the lane-per-fiber CUDA kernel executes:
// scan steps, window management, sweep, chunk records, verification and repair) on the CPU, one warp task at a time, the 32
// lanes of a warp in a plain loop (lanes only interact through the warp collectives, which the host Env computes over the
// loop).  Feed and Drain are the host stand-ins of the kernel's TMA feeder / row drain: same window contents, same calls.
// Not part of the product; built by tests/emu/Makefile with g++ (host code only; the CUDA headers only supply the __host__
// __device__ macros), from __graft_entry__.build() or on first use by the tests (tests/emu/lane_emu.py).
#include "../../proxtv_b200/csrc/lane_core.cuh"
#include <vector>
#include <string.h>
#include <stdio.h>

using namespace ptvl;

template <typename T> struct HostEnv {
    Lane<T> L[LANES];
    template <class F> void each(F f) { for (int l = 0; l < LANES; l++) f(L[l], l); }
    template <class F> int rmin(F f) { int m = f(L[0], 0); for (int l = 1; l < LANES; l++) { int v = f(L[l], l); if (v < m) m = v; } return m; }
    template <class F> int rmax(F f) { int m = f(L[0], 0); for (int l = 1; l < LANES; l++) { int v = f(L[l], l); if (v > m) m = v; } return m; }
    template <class F> bool any(F f) { for (int l = 0; l < LANES; l++) if (f(L[l], l)) return true; return false; }
    void sync() {}
    template <int W> void scan(Lane<T>& L, const Window<T, W>& w, int lane, const TaskGeom& g, const acc_t* rcp, acc_t lam2, bool ph1, int niter) {
        if (ph1) L.template run<true, W>(w, lane, g, rcp, lam2, niter); else L.template run<false, W>(w, lane, g, rcp, lam2, niter);
    }
};

// fused input / output arithmetic of a pass (kernels_lane.cu: PassOp has the same forms)
//   0  plain              in = A                          out = x
//   1  DR second half     in = A - (2 (C - B) - C)        out = (C - B) + x        A = Y, B = x_cols, C = t   (src/TV2Dopt.cpp:411-422)
//   2  DR final           in = A - (C - B)                out = x                                             (:427-430)
//   3  DR first half (T)  in = A     d = C - x ; out = B - (2 d - C) -> X (transposed), d -> X2 (transposed)   B = Y, C = t
//   4  DR final (T)       in = A     out = B - (C - x) -> X (transposed)
//   5  DR second half (T) in = A     out = B + x -> X (transposed)                                             B = d
//   6  plain (T)          in = A     out = x -> X (transposed)
template <typename T> struct Op {
    int kind; const T* A; const T* B; const T* C; T* X; T* X2;
    T in(long long g) const {
        if (kind == 0 || kind >= 3) return A[g];
        const T d = C[g] - B[g];
        if (kind == 1) return A[g] - (T(2) * d - C[g]);
        return A[g] - d;
    }
    // g: position in the pass's own layout; tg: position in the fiber-major (transposed) result arrays
    void out(long long g, long long tg, T x) const {
        if (kind == 3) { const T d = C[g] - x; X2[tg] = d; X[tg] = B[g] - (T(2) * d - C[g]); }
        else if (kind == 4) X[tg] = B[g] - (C[g] - x);
        else if (kind == 5) X[tg] = B[g] + x;
        else if (kind == 6) X[tg] = x;
        else X[g] = (kind == 1) ? (C[g] - B[g]) + x : x;
    }
};

template <typename T> struct Fibers {          // 32 adjacent fibers of a group
    long long base[LANES]; long long tbase[LANES]; long long stride; bool valid[LANES];      // tbase: fiber index * len
};

template <typename T, int W, int RT> struct HostFeed {
    static constexpr int R = RT;
    static constexpr int MAXQ = 2;
    const Window<T, W>* w; const Op<T>* op; const Fibers<T>* fb; int n; long long* rows_fed;
    template <class Env> void request(Env&, int row0) {
        for (int r = row0; r < row0 + R && r < n; r++)
            for (int l = 0; l < LANES; l++) w->st(r, l, fb->valid[l] ? op->in(fb->base[l] + (long long)r * fb->stride) : T(0));
        *rows_fed += R;
    }
    template <class Env> bool landed(Env&, int, bool) { return true; }
};

// direct drain: every swept row goes straight out (the strided pass of the kernel)
template <typename T, int W> struct HostDrainDirect {
    const Op<T>* op; const Fibers<T>* fb;
    void rows8(const Window<T, W>&, int r0, int cnt, int lane, const T* xs, bool valid) {
        if (valid) for (int u = 0; u < cnt; u++) op->out(fb->base[lane] + (long long)(r0 + u) * fb->stride, fb->tbase[lane] + r0 + u, xs[u]);
    }
    void prefetch(int, int, bool) {}
    template <class Env> void flush(Env&, const Window<T, W>&, int, bool) {}
    int hold(int, int) const { return 0x3fffffff; }
};
// boxed drain: rows are written back into the window and leave in aligned boxes of BOX rows (the contiguous pass of the kernel,
// which transposes a box through a staging tile and stores it with TMA); the window may not slide past an unstored box
template <typename T, int W, int BOX> struct HostDrainBoxed {
    const Op<T>* op; const Fibers<T>* fb; int stored; int ce;
    void rows8(const Window<T, W>& w, int r0, int cnt, int lane, const T* xs, bool) { for (int u = 0; u < cnt; u++) w.st(r0 + u, lane, xs[u]); }
    void prefetch(int, int, bool) {}
    template <class Env> void flush(Env&, const Window<T, W>& w, int upto, bool final) {
        while (stored + BOX <= upto || (final && stored < upto)) {
            const int b1 = stored + BOX < upto ? stored + BOX : upto;
            for (int r = stored; r < b1; r++)
                for (int l = 0; l < LANES; l++) if (fb->valid[l]) op->out(fb->base[l] + (long long)r * fb->stride, fb->tbase[l] + r, w.ld(r, l));
            stored = b1;
        }
    }
    int hold(int, int) const { return stored; }
};

struct EmuStats { long long tasks, epochs, retired_events, tails, rows_fed, repairs, retired_lanes, steps_max; };

template <typename T, int W, int TITER, int RT>
static int run_all(int opkind, const T* A, const T* B, const T* C, T* X, T* X2, long long nf, int len, long long inc, T lam, int clen, int halo,
                   int boxed, EmuStats* es) {
    if (nf <= 0 || len <= 0) return 0;
    Op<T> op{opkind, A, B, C, X, X2};
    // the kernel's plan: chunk boundaries on the feed's tile rows, balanced owned rows + halo (ChunkPlan); clen only sets how many
    ChunkPlan pl; pl.n = len; pl.gran = boxed ? 16 : 8; pl.halo = (halo + pl.gran - 1) / pl.gran * pl.gran;
    pl.nchunks = (clen <= 0 || clen >= len) ? 1 : ChunkPlan::fit(len, (len + clen - 1) / clen, pl.halo, pl.gran);
    std::vector<T> win((size_t)W * LANES); std::vector<acc_t> rcp(W + 2);
    std::vector<unsigned long long> flg8((Window<T, W>::flag_bytes() + 7) / 8 + 1);
    uint8_t* flgp = reinterpret_cast<uint8_t*>(flg8.data());
    for (int k = 1; k < W + 2; k++) rcp[k] = 1.0 / (acc_t)k;
    const long long slabs = inc > 1 ? nf / inc : 1, per_slab = inc > 1 ? inc : nf;
    const long long gps = (per_slab + LANES - 1) / LANES;
    std::vector<int> rin((size_t)pl.nchunks * LANES), rout((size_t)pl.nchunks * LANES), rovf((size_t)pl.nchunks * LANES);
    std::vector<int> rin2((size_t)pl.nchunks * LANES), rin3((size_t)pl.nchunks * LANES);
    for (long long s = 0; s < slabs; s++)
        for (long long gidx = 0; gidx < gps; gidx++) {
            Fibers<T> fb;
            for (int l = 0; l < LANES; l++) {
                const long long jj = gidx * LANES + l;
                fb.valid[l] = jj < per_slab;
                if (inc > 1) { fb.base[l] = s * inc * len + jj; fb.stride = inc; fb.tbase[l] = (s * inc + jj) * len; }
                else { fb.base[l] = jj * (long long)len; fb.stride = 1; fb.tbase[l] = jj * (long long)len; }
            }
            for (int c = 0; c < pl.nchunks; c++) {
                const TaskGeom g = pl.geom(c);
                Window<T, W> w{win.data(), flgp};
                memset(flgp, 0, Window<T, W>::flag_bytes());
                HostEnv<T> env;
                for (int l = 0; l < LANES; l++) env.L[l].init(w, l, g, lam, fb.valid[l]);
                long long fed = 0;
                HostFeed<T, W, RT> feed{&w, &op, &fb, len, &fed};
                TaskStats ts{0, 0, 0, 0};
                if (boxed) {
                    HostDrainBoxed<T, W, 16> drain{&op, &fb, g.cs, g.ce};
                    warp_task<T, W, TITER>(env, feed, drain, w, rcp.data(), g, lam, TITER + RT, &ts);
                } else {
                    HostDrainDirect<T, W> drain{&op, &fb};
                    warp_task<T, W, TITER>(env, feed, drain, w, rcp.data(), g, lam, TITER + RT, &ts);
                }
                for (int l = 0; l < LANES; l++) {
                    rin[(size_t)c * LANES + l] = env.L[l].in_rec; rout[(size_t)c * LANES + l] = env.L[l].out_rec;
                    rovf[(size_t)c * LANES + l] = env.L[l].retired ? env.L[l].ovf_rec : REC_NONE;
                    rin2[(size_t)c * LANES + l] = env.L[l].in_rec2; rin3[(size_t)c * LANES + l] = env.L[l].in_rec3;
                    if (env.L[l].retired) es->retired_lanes++;
                }
                es->tasks++; es->steps_max += ts.iters; es->epochs += ts.epochs; es->retired_events += ts.retired; es->tails += ts.tail; es->rows_fed += fed;
            }
            for (int l = 0; l < LANES; l++) {
                if (!fb.valid[l]) continue;
                const long long base = fb.base[l], st = fb.stride, tb = fb.tbase[l];
                es->repairs += verify_repair_fiber<T>(pl, lam,
                    [&](int c) { return rin[(size_t)c * LANES + l]; }, [&](int c) { return rin2[(size_t)c * LANES + l]; },
                    [&](int c) { return rin3[(size_t)c * LANES + l]; }, [&](int c) { return rout[(size_t)c * LANES + l]; },
                    [&](int c) { return rovf[(size_t)c * LANES + l]; }, [](int) {},
                    [&](int r) { return op.in(base + (long long)r * st); }, [&](int r, T v) { op.out(base + (long long)r * st, tb + r, v); });
            }
        }
    return 0;
}

extern "C" {
// config: 0 -> W=64,TITER=16,R=8 ; 1 -> W=32,TITER=8,R=8 ; 2 -> W=128,TITER=16,R=16 (float) ...
int emu_lane_f64(int opkind, const double* A, const double* B, const double* C, double* X, double* X2, long long nf, int len, long long inc,
                 double lam, int clen, int halo, int boxed, int config, long long* stats) {
    EmuStats es; memset(&es, 0, sizeof(es));
    int rc;
    if (config == 0) rc = run_all<double, 64, 16, 8>(opkind, A, B, C, X, X2, nf, len, inc, lam, clen, halo, boxed, &es);
    else if (config == 1) rc = run_all<double, 32, 8, 8>(opkind, A, B, C, X, X2, nf, len, inc, lam, clen, halo, boxed, &es);
    else rc = run_all<double, 128, 16, 16>(opkind, A, B, C, X, X2, nf, len, inc, lam, clen, halo, boxed, &es);
    if (stats) memcpy(stats, &es, sizeof(es));
    return rc;
}
int emu_lane_f32(int opkind, const float* A, const float* B, const float* C, float* X, float* X2, long long nf, int len, long long inc,
                 float lam, int clen, int halo, int boxed, int config, long long* stats) {
    EmuStats es; memset(&es, 0, sizeof(es));
    int rc;
    if (config == 0) rc = run_all<float, 128, 16, 8>(opkind, A, B, C, X, X2, nf, len, inc, lam, clen, halo, boxed, &es);
    else rc = run_all<float, 32, 8, 8>(opkind, A, B, C, X, X2, nf, len, inc, lam, clen, halo, boxed, &es);
    if (stats) memcpy(stats, &es, sizeof(es));
    return rc;
}
// the chunk plan: chunk count after fit(), boundaries cs(0..nchunks) and cold-start rows p0(0..nchunks-1)
int emu_plan(int n, int want, int halo, int gran, int* cs_out, int* p0_out) {
    ChunkPlan pl; pl.n = n; pl.halo = halo; pl.gran = gran; pl.nchunks = ChunkPlan::fit(n, want, halo, gran);
    for (int c = 0; c <= pl.nchunks; c++) cs_out[c] = pl.cs(c);
    for (int c = 0; c < pl.nchunks; c++) { const TaskGeom g = pl.geom(c); p0_out[c] = g.p0; if (g.cs != pl.cs(c) || g.ce != pl.cs(c + 1)) return -1; }
    return pl.nchunks;
}
// the task plan: every task index maps to a distinct (group, chunk) with chunk < chunks_of(group); returns the task count or -1
long long emu_taskplan(int nmax, long long gfull, long long groups) {
    TaskPlan tp; tp.n = 4096; tp.halo = 32; tp.gran = 8; tp.nmax = nmax; tp.gfull = gfull;
    const long long nt = tp.ntasks(groups);
    std::vector<char> seen((size_t)groups * nmax, 0);
    for (long long t = 0; t < nt; t++) {
        long long g; int c, nc;
        tp.locate(t, &g, &c, &nc);
        if (g < 0 || g >= groups || c < 0 || c >= nc || nc != tp.chunks_of(g) || seen[(size_t)g * nmax + c]) return -1;
        seen[(size_t)g * nmax + c] = 1;
    }
    long long cnt = 0; for (char v : seen) cnt += v;
    return cnt == nt ? nt : -1;
}
// plain sequential slope-form scan of one fiber (the arithmetic the lanes use, without any window / chunk machinery)
void emu_slope_seq_f64(const double* y, int n, double lam, double* x, long long* steps) {
    long long st = 0;
    slope_seq<double>(n, lam, 0, LK_BEGIN, [&](int i) { st++; return y[i]; },
                      [&](int f, int e, double v, int) { for (int r = f; r <= e; r++) x[r] = v; return false; });
    if (steps) *steps = st;
}
// the same, one fiber after the other over nf fibers stored back to back (the reference of the GPU tests, tests/test_gpu_lane.py)
void emu_slope_seq_rows_f64(const double* y, long long nf, int n, double lam, double* x) {
    for (long long j = 0; j < nf; j++) emu_slope_seq_f64(y + j * n, n, lam, x + j * n, nullptr);
}
}
