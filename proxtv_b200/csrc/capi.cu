// capi.cu -- the extern "C" boundary of libproxtv_b200.so (declared in include/proxtv_b200.h).
//
// Host-pointer entry points stage their arrays through a cached device arena (grow-only; one per process, guarded by a
// mutex), run the device-resident solver and copy the result back.  There is no CPU fallback: if no CUDA device is usable
// every entry point fails loudly.  Error behaviour follows the reference: "<fn>: <msg>" on stdout, info[RC] = RC_ERROR,
// return 0 (src/TV2Dopt.cpp:78-82,368-372).
#include "../../include/proxtv_b200.h"
#include "ptv_internal.h"
#include <mutex>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

using namespace ptv;

namespace {

thread_local std::string g_err;
std::recursive_mutex g_mu;
int g_engine = ENGINE_AUTO;

struct Arena {
    void* p = nullptr; size_t cap = 0;
    void* get(size_t bytes) {
        if (bytes <= cap) return p;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + (bytes >> 3);
        if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); p = nullptr;
            if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); p = nullptr; cap = 0; return nullptr; }
            cap = bytes; return p; }
        cap = want; return p;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
// solver workspace ; staging of host arrays -- one pair per device, so that a process that works on several devices in turn
// (torch tensors on cuda:0 and cuda:1) never hands one device's memory to kernels running on another
constexpr int MAX_DEV = 64;
Arena g_ws_d[MAX_DEV], g_io_d[MAX_DEV];
// slot of the current device; devices beyond MAX_DEV share the last slot's workspace tables only after have_device() refused them
int cur_dev() { int d = 0; if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); d = 0; } return (d < 0 || d >= MAX_DEV) ? MAX_DEV - 1 : d; }
#define g_ws (g_ws_d[cur_dev()])
#define g_io (g_io_d[cur_dev()])

// The workspaces, pipeline streams and captured graphs are one set per device, shared by every call: calls are serialised on the
// host by g_mu, and ON THE DEVICE by a per-device event -- a call's stream first waits for the previous call's work (which may
// have been enqueued on another stream), and records the event when its own work is enqueued.  Held for the whole call.
struct WsGuard {
    std::lock_guard<std::recursive_mutex> lk;
    cudaStream_t st; int dev;
    static cudaEvent_t& ev(int d) { static cudaEvent_t e[MAX_DEV] = {}; return e[d]; }
    explicit WsGuard(cudaStream_t s) : lk(g_mu), st(s), dev(-1) {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= MAX_DEV) { cudaGetLastError(); return; }
        dev = d;
        if (!ev(d)) { if (cudaEventCreateWithFlags(&ev(d), cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); ev(d) = nullptr; dev = -1; return; } }
        else cudaStreamWaitEvent(st, ev(d), 0);
    }
    ~WsGuard() { if (dev >= 0 && ev(dev)) cudaEventRecord(ev(dev), st); }
};

bool fail(const char* fn, const char* msg, double* info) {
    g_err = std::string(fn) + ": " + msg;
    printf("%s: %s\n", fn, msg); fflush(stdout);
    if (info) info[INFO_RC] = RC_ERROR;
    return false;
}
bool cuda_ok(const char* fn, cudaError_t e, double* info) {
    if (e == cudaSuccess) return true;
    cudaGetLastError();
    return fail(fn, (std::string("CUDA error: ") + cudaGetErrorString(e)).c_str(), info);
}
bool have_device(const char* fn, double* info) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) { cudaGetLastError();
        return fail(fn, "no usable CUDA device (libproxtv_b200 has no CPU fallback)", info); }
    int d = -1;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= MAX_DEV - 1) { cudaGetLastError();
        return fail(fn, "current CUDA device index out of the supported range (0..62)", info); }
    return true;
}
inline size_t al(size_t b) { return (b + 255) & ~(size_t)255; }

// Generic host-pointer batched 1D prox.  weights: nullptr or host array with nf*(len-1) entries.
template <typename T>
int host_prox_fibers(const char* fn, const T* in, T* out, long long nf, int len, long long inc, T lam, const T* lamv) {
    if (nf <= 0 || len <= 0) return 1;
    if (!have_device(fn, nullptr)) return 0;
    WsGuard guard(0);
    const size_t n = (size_t)nf * len, nw = lamv ? (size_t)nf * (len - 1) : 0;
    char* d = (char*)g_io.get(2 * al(n * sizeof(T)) + al(nw * sizeof(T) + 8));
    // scratch: staging of strided fibers (2n), or the overlapping tiles of contiguous fibers longer than shared memory
    T* scr = (inc != 1) ? (T*)g_ws.get(al((size_t)strided_scratch_elems(nf, len) * sizeof(T)))
                        : (len > 16384 && !lamv ? (T*)g_ws.get(al((size_t)lf_scratch_elems(nf, len) * sizeof(T)) + 256) : nullptr);
    if (!d) return fail(fn, "out of device memory", nullptr) ? 1 : 0;
    T* din = (T*)d; T* dout = (T*)(d + al(n * sizeof(T))); T* dw = (T*)(d + 2 * al(n * sizeof(T)));
    cudaStream_t st = 0;
    if (!cuda_ok(fn, cudaMemcpyAsync(din, in, n * sizeof(T), cudaMemcpyHostToDevice, st), nullptr)) return 0;
    if (nw && !cuda_ok(fn, cudaMemcpyAsync(dw, lamv, nw * sizeof(T), cudaMemcpyHostToDevice, st), nullptr)) return 0;
    FiberGeom g{nf, len, inc};
    const Engine eng = (!lamv && nf >= 1024 && len >= 64) ? lane_guard<T>((Engine)g_engine, din, (long long)n, (double)lam, st) : (Engine)g_engine;
    if (!cuda_ok(fn, prox_fibers<T>(din, nullptr, IN_A, dout, 0, g, lam, lamv ? dw : nullptr, eng, scr, st,
                                     (inc == 1 && scr) ? lf_scratch_elems(nf, len) : (inc != 1 ? strided_scratch_elems(nf, len) : 0)), nullptr)) return 0;
    if (!cuda_ok(fn, cudaMemcpyAsync(out, dout, n * sizeof(T), cudaMemcpyDeviceToHost, st), nullptr)) return 0;
    if (!cuda_ok(fn, cudaStreamSynchronize(st), nullptr)) return 0;
    return 1;
}

template <typename T>
int host_dr2(const char* fn, size_t M, size_t N, int batch, const T* Y, T W1, T W2, T* out, int maxit, double* info) {
    if (!have_device(fn, info)) return 0;
    WsGuard guard(0);
    const size_t n = M * N * (size_t)batch;
    if (n == 0) { if (info) { info[INFO_ITERS] = maxit <= 0 ? MAX_ITERS_DR : maxit; info[INFO_RC] = RC_OK; } return 0; }
    char* d = (char*)g_io.get(2 * al(n * sizeof(T)));
    void* ws = g_ws.get(ws_bytes_dr2<T>(M, N, batch));
    if (!d || !ws) { fail(fn, "out of memory", info); return 0; }                       // TV2Dopt.cpp:383-384
    T* dY = (T*)d; T* dout = (T*)(d + al(n * sizeof(T)));
    cudaStream_t st = 0;
    if (!cuda_ok(fn, cudaMemcpyAsync(dY, Y, n * sizeof(T), cudaMemcpyHostToDevice, st), info)) return 0;
    double linfo[3] = {0, 0, RC_OK};                   // a NULL info must not hide a failed solve (nothing is copied back then)
    double* pinfo = info ? info : linfo;
    dr2_device<T>(M, N, batch, 0, dY, W1, W2, dout, maxit, pinfo, ws, (Engine)g_engine, st);
    if (pinfo[INFO_RC] == RC_ERROR) { fail(fn, "device solver failed", info); return 0; }
    if (!cuda_ok(fn, cudaMemcpyAsync(out, dout, n * sizeof(T), cudaMemcpyDeviceToHost, st), info)) return 0;
    if (!cuda_ok(fn, cudaStreamSynchronize(st), info)) return 0;
    return 0;
}

// DR2L1W_TV with host (host_io) or device arrays.  W1: (M-1) x N, W2: M x (N-1), column-major like Y.
template <typename T>
int run_drw(const char* fn, bool host_io, size_t M, size_t N, const T* Y, const T* W1, const T* W2, T* out, int maxit, double* info,
            cudaStream_t st) {
    if (!have_device(fn, info)) return 0;
    WsGuard guard(st);
    const size_t n = M * N, n1 = M ? (M - 1) * N : 0, n2 = N ? M * (N - 1) : 0;
    if (n == 0) { if (info) { info[INFO_ITERS] = maxit <= 0 ? MAX_ITERS_DR : maxit; info[INFO_RC] = RC_OK; } return 0; }
    void* ws = g_ws.get(ws_bytes_dr2<T>(M, N, 1));
    if (!ws) { fail(fn, "out of memory", info); return 0; }                             // TV2DWopt.cpp:78-79
    if (!host_io) return drw_device<T>(M, N, Y, W1, W2, out, maxit, info, ws, (Engine)g_engine, st);
    char* d = (char*)g_io.get(2 * al(n * sizeof(T)) + al(n1 * sizeof(T) + 8) + al(n2 * sizeof(T) + 8));
    if (!d) { fail(fn, "out of memory", info); return 0; }
    T* dY = (T*)d; T* dout = (T*)(d + al(n * sizeof(T))); T* d1 = (T*)(d + 2 * al(n * sizeof(T))); T* d2 = (T*)((char*)d1 + al(n1 * sizeof(T) + 8));
    if (!cuda_ok(fn, cudaMemcpyAsync(dY, Y, n * sizeof(T), cudaMemcpyHostToDevice, st), info)) return 0;
    if (n1 && !cuda_ok(fn, cudaMemcpyAsync(d1, W1, n1 * sizeof(T), cudaMemcpyHostToDevice, st), info)) return 0;
    if (n2 && !cuda_ok(fn, cudaMemcpyAsync(d2, W2, n2 * sizeof(T), cudaMemcpyHostToDevice, st), info)) return 0;
    double linfo[3] = {0, 0, RC_OK};
    double* pinfo = info ? info : linfo;
    drw_device<T>(M, N, dY, d1, d2, dout, maxit, pinfo, ws, (Engine)g_engine, st);
    if (pinfo[INFO_RC] == RC_ERROR) { fail(fn, "device solver failed", info); return 0; }
    if (!cuda_ok(fn, cudaMemcpyAsync(out, dout, n * sizeof(T), cudaMemcpyDeviceToHost, st), info)) return 0;
    if (!cuda_ok(fn, cudaStreamSynchronize(st), info)) return 0;
    return 0;
}

// mode 0: PD2_TV, 1: PD_TV, 2: PDR_TV.  y/x host (host_io) or device pointers.
template <typename T>
int run_pd(const char* fn, int mode, bool host_io, const T* y, double* lambdas, double* norms, double* dims, T* x, double* info,
           int* ns, int nds, int npen, int maxIters, cudaStream_t st) {
    if (!have_device(fn, info)) return 0;
    if (norms) for (int i = 0; i < npen; i++) if (norms[i] != 1.0) {
        fail(fn, "only p = 1 (TV-L1) penalty terms are implemented on the GPU path", info); return 0; }
    if (nds <= 0 || !ns) { fail(fn, "invalid dimensions", info); return 0; }
    long long n = 1; for (int i = 0; i < nds; i++) n *= ns[i];
    WsGuard guard(st);
    if (mode >= 1) for (int i = 0; i < npen; i++) lambdas[i] *= npen;                   // TVNDopt.cpp:100-101, :339-340 (in place)
    void* ws = g_ws.get(ws_bytes_pd<T>(n, npen > 2 ? npen : 2));
    if (!ws) { fail(fn, "out of memory", info); return 0; }
    const T* dy = y; T* dx = x;
    if (host_io && n > 0) {
        char* d = (char*)g_io.get(2 * al((size_t)n * sizeof(T)));
        if (!d) { fail(fn, "out of memory", info); return 0; }
        dy = (T*)d; dx = (T*)(d + al((size_t)n * sizeof(T)));
        if (!cuda_ok(fn, cudaMemcpyAsync((void*)dy, y, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, st), info)) return 0;
    }
    int rc = mode == 0 ? pd2_device<T>(dy, lambdas, dims, dx, info, ns, nds, npen, maxIters, ws, (Engine)g_engine, st)
           : mode == 1 ? pd_device<T>(dy, lambdas, dims, dx, info, ns, nds, npen, maxIters, ws, (Engine)g_engine, st)
                       : pdr_device<T>(dy, lambdas, dims, dx, info, ns, nds, npen, maxIters, ws, (Engine)g_engine, st);
    if (!rc) return 0;
    if (host_io && n > 0) {
        if (!cuda_ok(fn, cudaMemcpyAsync(x, dx, (size_t)n * sizeof(T), cudaMemcpyDeviceToHost, st), info)) return 0;
        if (!cuda_ok(fn, cudaStreamSynchronize(st), info)) return 0;
    }
    return 1;
}

template <typename T> static T* dev_scratch(long long nf, int len, long long inc) {
    if (nf <= 0 || len <= 0 || (inc == 1 && len <= 16384)) return nullptr;
    std::lock_guard<std::recursive_mutex> lk(g_mu);
    if (inc == 1) return (T*)g_ws.get(al((size_t)lf_scratch_elems(nf, len) * sizeof(T)) + 256);
    return (T*)g_ws.get(al((size_t)strided_scratch_elems(nf, len) * sizeof(T)));
}

template <typename T>
static int dev_dr2(const char* fn, size_t M, size_t N, int batch, int row_major, const T* Y, T W1, T W2, T* out, int maxit, double* info, void* stream) {
    if (!have_device(fn, info)) return 0;
    WsGuard guard((cudaStream_t)stream);
    void* ws = g_ws.get(ws_bytes_dr2<T>(M, N, batch));
    if (!ws) { fail(fn, "out of memory", info); return 0; }
    return dr2_device<T>(M, N, batch, row_major, Y, W1, W2, out, maxit, info, ws, (Engine)g_engine, (cudaStream_t)stream);
}

}  // namespace

extern "C" {

int proxtv_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; } return n; }
const char* proxtv_last_error(void) { return g_err.c_str(); }
const char* proxtv_version(void) { return "proxtv_b200 0.1 (sm_100a)"; }
int proxtv_set_engine(int e) { int o = g_engine; if (e >= 0 && e <= 8) g_engine = e; return o; }
void* proxtv_host_alloc(size_t bytes) { void* p = nullptr; if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; } return p; }
void proxtv_host_free(void* p) { if (p) cudaFreeHost(p); }
void proxtv_profile_enable(int on) { profile_enable(on); }
void proxtv_profile_reset(void) { profile_reset(); }
void proxtv_profile_read(double* ms, long long* launches, long long* spans) { profile_read(ms, launches, spans); }
void proxtv_release_workspace(void) { std::lock_guard<std::recursive_mutex> lk(g_mu); for (int d = 0; d < MAX_DEV; d++) { g_ws_d[d].release(); g_io_d[d].release(); } }

// ---- experimental: the lane-per-fiber streaming engine (kernels_lane.cu), device pointers ----
int proxtv_lane_prox_dev_f64(int op, const double* A, const double* B, const double* C, double* X, long long nf, int len, long long inc,
                             double lam, void* stream) {
    WsGuard guard((cudaStream_t)stream);
    void* scr = ptvl::lane_scratch(nf, len);
    if (!scr) return 0;
    cudaError_t e = ptvl::lane_prox<double>(op, A, B, C, X, nf, len, inc, lam, scr, (cudaStream_t)stream);
    if (e != cudaSuccess) { cudaGetLastError(); g_err = std::string("proxtv_lane_prox_dev_f64: ") + cudaGetErrorString(e); return 0; }
    return 1;
}
int proxtv_lane_prox2_dev_f64(int op, const double* A, const double* B, const double* C, double* X, double* X2, long long nf, int len, long long inc,
                              double lam, void* stream) {
    WsGuard guard((cudaStream_t)stream);
    void* scr = ptvl::lane_scratch(nf, len);
    if (!scr) return 0;
    cudaError_t e = ptvl::lane_prox<double>(op, A, B, C, X, nf, len, inc, lam, scr, (cudaStream_t)stream, X2);
    if (e != cudaSuccess) { cudaGetLastError(); g_err = std::string("proxtv_lane_prox2_dev_f64: ") + cudaGetErrorString(e); return 0; }
    return 1;
}
int proxtv_lane_prox_dev_f32(int op, const float* A, const float* B, const float* C, float* X, long long nf, int len, long long inc,
                             float lam, void* stream) {
    WsGuard guard((cudaStream_t)stream);
    void* scr = ptvl::lane_scratch(nf, len);
    if (!scr) return 0;
    cudaError_t e = ptvl::lane_prox<float>(op, A, B, C, X, nf, len, inc, lam, scr, (cudaStream_t)stream);
    if (e != cudaSuccess) { cudaGetLastError(); g_err = std::string("proxtv_lane_prox_dev_f32: ") + cudaGetErrorString(e); return 0; }
    return 1;
}
int proxtv_lane_prox2_dev_f32(int op, const float* A, const float* B, const float* C, float* X, float* X2, long long nf, int len, long long inc,
                              float lam, void* stream) {
    WsGuard guard((cudaStream_t)stream);
    void* scr = ptvl::lane_scratch(nf, len);
    if (!scr) return 0;
    cudaError_t e = ptvl::lane_prox<float>(op, A, B, C, X, nf, len, inc, lam, scr, (cudaStream_t)stream, X2);
    if (e != cudaSuccess) { cudaGetLastError(); g_err = std::string("proxtv_lane_prox2_dev_f32: ") + cudaGetErrorString(e); return 0; }
    return 1;
}
void proxtv_lane_tuning(int clen, int halo, int variant) { ptvl::lane_set_tuning(clen, halo, variant); }
void proxtv_lane_tasklog(unsigned long long* dev, long long cap_tasks) { ptvl::lane_set_tasklog(dev, cap_tasks); }
int proxtv_lane_guard_last(void) { return lane_guard_last(); }
unsigned long long proxtv_lane_stats(int reset) { return ptvl::lane_read_stats(reset); }

// ---- Part 1: drop-in symbols ----
void hybridTautString_TV1(double* y, int n, double lambda, double* x) {
    host_prox_fibers<double>("hybridTautString_TV1", y, x, 1, n, 1, lambda, nullptr);
}
void hybridTautString_TV1_custom(double* y, int n, double lambda, double* x, double) {
    host_prox_fibers<double>("hybridTautString_TV1_custom", y, x, 1, n, 1, lambda, nullptr);
}
int classicTautString_TV1(double* signal, int n, double lam, double* prox) {
    if (n <= 0) return 1;
    if (lam <= 0 || n == 1) { memmove(prox, signal, (size_t)n * sizeof(double)); return 1; }   // TVL1opt_tautstring.cpp:258-263
    host_prox_fibers<double>("classicTautString_TV1", signal, prox, 1, n, 1, lam, nullptr);
    return 1;
}
int linearizedTautString_TV1(double* y, double lambda, double* x, int n) {
    host_prox_fibers<double>("linearizedTautString_TV1", y, x, 1, n, 1, lambda, nullptr);
    return 1;
}
void TV1D_denoise(double* input, double* output, const int width, const double lambda) {
    if (width > 0 && lambda >= 0) host_prox_fibers<double>("TV1D_denoise", input, output, 1, width, 1, lambda, nullptr);
}
int tautString_TV1_Weighted(double* y, double* lambda, double* x, int n) {
    if (n == 1) { x[0] = y[0]; return 1; }
    host_prox_fibers<double>("tautString_TV1_Weighted", y, x, 1, n, 1, 0.0, lambda);
    return 1;
}
// The reference's alternative 1D TV-L1 solvers compute the same unique minimiser (<= 4e-14 apart on random data, 9e-7 for Condat's
// float-truncating taut-string variant -- measured with the compiled reference): they all map onto the exact kernel.
static void ok_info(double* info) { if (info) { info[INFO_ITERS] = 0; info[INFO_GAP] = 0; info[INFO_RC] = RC_OK; } }
int PN_TV1(double* y, double lambda, double* x, double* info, int n, double, void*) {
    if (!host_prox_fibers<double>("PN_TV1", y, x, 1, n, 1, lambda, nullptr)) { if (info) info[INFO_RC] = RC_ERROR; return 0; }
    ok_info(info); return 1;
}
int PN_TV1_Weighted(double* Y, double* W, double* X, double* info, int n, double, void*) {
    if (n == 1) { X[0] = Y[0]; ok_info(info); return 1; }
    if (!host_prox_fibers<double>("PN_TV1_Weighted", Y, X, 1, n, 1, 0.0, W)) { if (info) info[INFO_RC] = RC_ERROR; return 0; }
    ok_info(info); return 1;
}
void TV1D_denoise_tautstring(double* input, double* output, int width, const double lambda) {
    if (width > 0 && lambda >= 0) host_prox_fibers<double>("TV1D_denoise_tautstring", input, output, 1, width, 1, lambda, nullptr);
}
void SolveTVConvexQuadratic_a1_nw(int n, double* b, double w, double* solution) {
    host_prox_fibers<double>("SolveTVConvexQuadratic_a1_nw", b, solution, 1, n, 1, w, nullptr);
}
void SolveTVConvexQuadratic_a1(int n, double* b, double* w, double* solution) {
    if (n == 1) { solution[0] = b[0]; return; }
    host_prox_fibers<double>("SolveTVConvexQuadratic_a1", b, solution, 1, n, 1, 0.0, w);
}
void dp(int n, double* y, double lam, double* beta) {
    host_prox_fibers<double>("dp", y, beta, 1, n, 1, lam, nullptr);
}
int TV(double* y, double lambda, double* x, double* info, int n, double p, void*) {
    if (p < 1) { fail("TVopt", "TV only works for norms p >= 1", info); return 0; }                // TVgenopt.cpp:37-38
    if (p != 1) { fail("TVopt", "only p = 1 (TV-L1) is implemented on the GPU path", info); return 0; }
    if (!host_prox_fibers<double>("TVopt", y, x, 1, n, 1, lambda, nullptr)) { if (info) info[INFO_RC] = RC_ERROR; return 0; }
    if (info) { info[INFO_RC] = RC_OK; info[INFO_ITERS] = 0; info[INFO_GAP] = 0; }                 // :43-47
    return 1;
}
int DR2_TV(size_t M, size_t N, double* unary, double W1, double W2, double norm1, double norm2, double* s, int, int maxit,
           double* info) {
    if (norm1 != 1.0 || norm2 != 1.0) { fail("DR2_TV", "only p = 1 (TV-L1) penalties are implemented on the GPU path", info); return 0; }
    return host_dr2<double>("DR2_TV", M, N, 1, unary, W1, W2, s, maxit, info);
}
int DR2L1W_TV(size_t M, size_t N, double* unary, double* W1, double* W2, double* s, int, int maxit, double* info) {
    return run_drw<double>("DR2L1W_TV", true, M, N, unary, W1, W2, s, maxit, info, 0);
}
int PD2_TV(double* y, double* lambdas, double* norms, double* dims, double* x, double* info, int* ns, int nds, int npen, int,
           int maxIters) {
    return run_pd<double>("PD2_TV", 0, true, y, lambdas, norms, dims, x, info, ns, nds, npen, maxIters, 0);
}
int PD_TV(double* y, double* lambdas, double* norms, double* dims, double* x, double* info, int* ns, int nds, int npen, int,
          int maxIters) {
    return run_pd<double>("PD_TV", 1, true, y, lambdas, norms, dims, x, info, ns, nds, npen, maxIters, 0);
}
int PDR_TV(double* y, double* lambdas, double* norms, double* dims, double* x, double* info, int* ns, int nds, int npen, int,
           int maxIters) {
    return run_pd<double>("PDR_TV", 2, true, y, lambdas, norms, dims, x, info, ns, nds, npen, maxIters, 0);
}

// ---- Part 2: extensions ----
int proxtv_prox_fibers_dev_f64(const double* in, double* out, long long nf, int len, long long inc, double lam, const double* lamv, void* stream) {
    if (!have_device("proxtv_prox_fibers_dev_f64", nullptr)) return 0;
    WsGuard guard((cudaStream_t)stream);
    const Engine eng = (!lamv && nf >= 1024 && len >= 64) ? lane_guard<double>((Engine)g_engine, in, nf * (long long)len, lam, (cudaStream_t)stream) : (Engine)g_engine;
    return cuda_ok("proxtv_prox_fibers_dev_f64", prox_fibers<double>(in, nullptr, IN_A, out, 0, FiberGeom{nf, len, inc}, lam, lamv, eng, dev_scratch<double>(nf, len, inc), (cudaStream_t)stream,
                                                                 (inc == 1 && len > 16384) ? lf_scratch_elems(nf, len) : (inc != 1 ? strided_scratch_elems(nf, len) : 0)), nullptr);
}
int proxtv_prox_fibers_dev_f32(const float* in, float* out, long long nf, int len, long long inc, float lam, const float* lamv, void* stream) {
    if (!have_device("proxtv_prox_fibers_dev_f32", nullptr)) return 0;
    WsGuard guard((cudaStream_t)stream);
    const Engine eng = (!lamv && nf >= 1024 && len >= 64) ? lane_guard<float>((Engine)g_engine, in, nf * (long long)len, (double)lam, (cudaStream_t)stream) : (Engine)g_engine;
    return cuda_ok("proxtv_prox_fibers_dev_f32", prox_fibers<float>(in, nullptr, IN_A, out, 0, FiberGeom{nf, len, inc}, lam, lamv, eng, dev_scratch<float>(nf, len, inc), (cudaStream_t)stream,
                                                                 (inc == 1 && len > 16384) ? lf_scratch_elems(nf, len) : (inc != 1 ? strided_scratch_elems(nf, len) : 0)), nullptr);
}
int proxtv_prox_fibers_f64(const double* in, double* out, long long nf, int len, long long inc, double lam, const double* lamv) {
    return host_prox_fibers<double>("proxtv_prox_fibers_f64", in, out, nf, len, inc, lam, lamv);
}
int proxtv_prox_fibers_f32(const float* in, float* out, long long nf, int len, long long inc, float lam, const float* lamv) {
    return host_prox_fibers<float>("proxtv_prox_fibers_f32", in, out, nf, len, inc, lam, lamv);
}

int proxtv_DR2_TV_dev_f64(size_t M, size_t N, int batch, int row_major, const double* Y, double W1, double W2, double* out, int maxit, double* info, void* stream) {
    return dev_dr2<double>("proxtv_DR2_TV_dev_f64", M, N, batch, row_major, Y, W1, W2, out, maxit, info, stream); }
int proxtv_DR2_TV_dev_f32(size_t M, size_t N, int batch, int row_major, const float* Y, float W1, float W2, float* out, int maxit, double* info, void* stream) {
    return dev_dr2<float>("proxtv_DR2_TV_dev_f32", M, N, batch, row_major, Y, W1, W2, out, maxit, info, stream); }
int proxtv_DR2_TV_batched_f64(size_t M, size_t N, int batch, const double* Y, double W1, double W2, double* out, int maxit, double* info) {
    return host_dr2<double>("proxtv_DR2_TV_batched_f64", M, N, batch, Y, W1, W2, out, maxit, info); }
int proxtv_DR2_TV_batched_f32(size_t M, size_t N, int batch, const float* Y, float W1, float W2, float* out, int maxit, double* info) {
    return host_dr2<float>("proxtv_DR2_TV_batched_f32", M, N, batch, Y, W1, W2, out, maxit, info); }

int proxtv_DR2L1W_TV_dev_f64(size_t M, size_t N, const double* Y, const double* W1, const double* W2, double* out, int maxit, double* info, void* stream) {
    return run_drw<double>("proxtv_DR2L1W_TV_dev_f64", false, M, N, Y, W1, W2, out, maxit, info, (cudaStream_t)stream); }
int proxtv_DR2L1W_TV_dev_f32(size_t M, size_t N, const float* Y, const float* W1, const float* W2, float* out, int maxit, double* info, void* stream) {
    return run_drw<float>("proxtv_DR2L1W_TV_dev_f32", false, M, N, Y, W1, W2, out, maxit, info, (cudaStream_t)stream); }

int proxtv_PD2_TV_dev_f64(const double* y, double* lambdas, double* dims, double* x, double* info, int* ns, int nds, int npen, int maxIters, void* stream) {
    return run_pd<double>("proxtv_PD2_TV_dev_f64", 0, false, y, lambdas, nullptr, dims, x, info, ns, nds, npen, maxIters, (cudaStream_t)stream); }
int proxtv_PD2_TV_dev_f32(const float* y, double* lambdas, double* dims, float* x, double* info, int* ns, int nds, int npen, int maxIters, void* stream) {
    return run_pd<float>("proxtv_PD2_TV_dev_f32", 0, false, y, lambdas, nullptr, dims, x, info, ns, nds, npen, maxIters, (cudaStream_t)stream); }
int proxtv_PD_TV_dev_f64(const double* y, double* lambdas, double* dims, double* x, double* info, int* ns, int nds, int npen, int maxIters, void* stream) {
    return run_pd<double>("proxtv_PD_TV_dev_f64", 1, false, y, lambdas, nullptr, dims, x, info, ns, nds, npen, maxIters, (cudaStream_t)stream); }
int proxtv_PD_TV_dev_f32(const float* y, double* lambdas, double* dims, float* x, double* info, int* ns, int nds, int npen, int maxIters, void* stream) {
    return run_pd<float>("proxtv_PD_TV_dev_f32", 1, false, y, lambdas, nullptr, dims, x, info, ns, nds, npen, maxIters, (cudaStream_t)stream); }
int proxtv_PDR_TV_dev_f64(const double* y, double* lambdas, double* dims, double* x, double* info, int* ns, int nds, int npen, int maxIters, void* stream) {
    return run_pd<double>("proxtv_PDR_TV_dev_f64", 2, false, y, lambdas, nullptr, dims, x, info, ns, nds, npen, maxIters, (cudaStream_t)stream); }
int proxtv_PDR_TV_dev_f32(const float* y, double* lambdas, double* dims, float* x, double* info, int* ns, int nds, int npen, int maxIters, void* stream) {
    return run_pd<float>("proxtv_PDR_TV_dev_f32", 2, false, y, lambdas, nullptr, dims, x, info, ns, nds, npen, maxIters, (cudaStream_t)stream); }
int proxtv_PD_TV_f32(const float* y, double* lambdas, double* dims, float* x, double* info, int* ns, int nds, int npen, int maxIters) {
    return run_pd<float>("proxtv_PD_TV_f32", 1, true, y, lambdas, nullptr, dims, x, info, ns, nds, npen, maxIters, 0); }

}  // extern "C"
