/*
 * proxtv_b200.h -- C ABI of libproxtv_b200.so, the B200-native TV-L1 proximity operators.
 *
 * Part 1 re-exports, with identical names, prototypes, argument meaning, return values and info[] contents, the hot-path
 * subset of the reference's C interface (src/TVopt.h:88-141 == the cffi cdef in prox_tv/prox_tv_build.py:8-77), so the
 * reference's Python wrapper (prox_tv/__init__.py) or MATLAB mex glue can bind this library instead of its own object
 * code (see INTEGRATION.md).  All pointers in Part 1 are HOST pointers, arrays are float64, 2D/ND arrays column-major;
 * the caller owns every buffer; nothing is retained after return.  The computation runs on the current CUDA device
 * (cuda:0 unless cudaSetDevice was called by the host process); there is no CPU fallback: without a usable device
 * the calls print an error, set info[2] = RC_ERROR (3) where an info array exists and leave the output untouched.
 *
 * Part 2 adds what the BASELINE configurations need and the reference lacks: device-pointer variants (no PCIe traffic),
 * a leading batch dimension, float32 instantiations and pinned-host helpers.
 *
 * Plain C: no C++/torch types cross this boundary.
 */
#ifndef PROXTV_B200_H
#define PROXTV_B200_H
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* info[] slots and return codes -- reference: src/general.h:58-73 */
#define PROXTV_INFO_ITERS 0
#define PROXTV_INFO_GAP 1
#define PROXTV_INFO_RC 2
#define PROXTV_RC_OK 0
#define PROXTV_RC_ITERS 1
#define PROXTV_RC_STUCK 2
#define PROXTV_RC_ERROR 3

/* ------------------------------------------------------------------------------------------------------------------
 * Part 1 -- drop-in symbols (host pointers, float64)
 * ------------------------------------------------------------------------------------------------------------------ */

/* replaces src/TVL1opt_hybridtautstring.cpp:237 (prototype src/TVopt.h:96).  x = argmin 0.5|x-y|^2 + lambda*sum|x_i-x_{i+1}|.
 * Computed with the linearized taut-string scan; the reference's switch to the classic method after n^1.05 steps is an
 * execution-time heuristic that changes results by <= 5e-11 abs and is not reproduced. */
void hybridTautString_TV1(double *y, int n, double lambda, double *x);
/* replaces src/TVL1opt_hybridtautstring.cpp:56 (src/TVopt.h:97); backtracksexp is accepted and ignored (see above). */
void hybridTautString_TV1_custom(double *y, int n, double lambda, double *x, double backtracksexp);
/* replaces src/TVL1opt_tautstring.cpp:355 (src/TVopt.h:95).  Returns 1.  lam <= 0 or n == 1: x = signal (:258-263). */
int classicTautString_TV1(double *signal, int n, double lam, double *prox);
/* replaces src/TVL1opt.cpp:359 (src/TVopt.h:94).  Returns 1.  Bit-identical to the reference. */
int linearizedTautString_TV1(double *y, double lambda, double *x, int n);
/* replaces src/condat_fast_tv.cpp:78 (src/condat_fast_tv.h).  In-place (output == input) allowed; width <= 0 or
 * lambda < 0: nothing is done (:79). */
void TV1D_denoise(double *input, double *output, const int width, const double lambda);
/* replaces src/TVL1Wopt.cpp:364 (src/TVopt.h:103).  lambda has n-1 entries.  Returns 1.  Bit-identical to the reference. */
int tautString_TV1_Weighted(double *y, double *lambda, double *x, int n);
/* The reference's other 1D TV-L1 solvers: projected Newton (src/TVL1opt.cpp:44, src/TVL1Wopt.cpp:36), Condat's taut-string
 * variant (src/condat_fast_tv.cpp:133), Kolmogorov's (src/TVL1opt_kolmogorov.cpp) and Johnson's dynamic programming
 * (src/johnsonRyanTV.cpp).  Same unique minimiser as the functions above (<= 4e-14 apart on random data with the compiled
 * reference; 9e-7 for TV1D_denoise_tautstring, which truncates a slope to float), so they are served by the same exact kernel.
 * info = {0, 0, RC_OK}; sigma and ws are ignored; weighted forms take n-1 weights. */
int PN_TV1(double *y, double lambda, double *x, double *info, int n, double sigma, void *ws);
int PN_TV1_Weighted(double *Y, double *W, double *X, double *info, int n, double sigma, void *ws);
void TV1D_denoise_tautstring(double *input, double *output, int width, const double lambda);
void SolveTVConvexQuadratic_a1_nw(int n, double *b, double w, double *solution);
void SolveTVConvexQuadratic_a1(int n, double *b, double *w, double *solution);
void dp(int n, double *y, double lam, double *beta);
/* replaces src/TVgenopt.cpp:30 (src/TVopt.h:91) for p == 1 only (other norms: prints an error, RC_ERROR, returns 0).
 * ws is ignored (the reference's Python wrapper always passes NULL). */
int TV(double *y, double lambda, double *x, double *info, int n, double p, void *ws);
/* replaces src/TV2Dopt.cpp:352 (src/TVopt.h:128).  M x N column-major; fixed maxit iterations (<= 0: 35) + final
 * projection; info = {maxit, untouched, RC_OK}; returns 0 on success AND on error, like the reference (:440, :372).
 * norm1, norm2 must be 1; nThreads is ignored. */
int DR2_TV(size_t M, size_t N, double *unary, double W1, double W2, double norm1, double norm2, double *s, int nThreads,
           int maxit, double *info);
/* replaces src/TV2DWopt.cpp:46 (src/TVopt.h:116): DR2_TV's iteration with per-edge weights.  unary, s: M x N column-major;
 * W1: (M-1) x N column-major (weights of the edges along columns), W2: M x (N-1) column-major (edges along rows).
 * info = {maxit, untouched, RC_OK}; returns 0 on success AND on error, like the reference (:135, :64-68).  nThreads is
 * ignored.  Fibers of length 1 (M == 1 or N == 1) are left unchanged (the reference reads past an empty weight line). */
int DR2L1W_TV(size_t M, size_t N, double *unary, double *W1, double *W2, double *s, int nThreads, int maxit, double *info);
/* replaces src/TV2Dopt.cpp:59 (src/TVopt.h:126).  npen <= 2, norms must be 1, dims are 1-based; info = {iters, stop, RC};
 * RC_ITERS is set when iters >= 35 regardless of maxIters (:289); returns 1 ok / 0 error. */
int PD2_TV(double *y, double *lambdas, double *norms, double *dims, double *x, double *info, int *ns, int nds, int npen,
           int ncores, int maxIters);
/* replaces src/TVNDopt.cpp:48 (src/TVopt.h:137).  Like the reference it multiplies lambdas[] by npen IN PLACE (:100-101). */
int PD_TV(double *y, double *lambdas, double *norms, double *dims, double *x, double *info, int *ns, int nds, int npen,
          int ncores, int maxIters);
/* replaces src/TVNDopt.cpp:280 (src/TVopt.h:138; reached from MATLAB only in the reference, matlab/solveTVND_PDR.cpp:89): parallel
 * Douglas-Rachford over npen one-dimensional TV-L1 terms.  Runs exactly maxIters iterations (<= 0: 35; the reference's loop has no
 * stop test); multiplies lambdas[] by npen IN PLACE (:339-340); info = {iters, mean|x - x_last| of the last iteration, RC_ITERS when
 * iters >= 35 else RC_OK}; returns 1 ok / 0 error.  norms must be 1 (the reference's p = 2 / general-p terms are out of scope). */
int PDR_TV(double *y, double *lambdas, double *norms, double *dims, double *x, double *info, int *ns, int nds, int npen,
           int ncores, int maxIters);

/* ------------------------------------------------------------------------------------------------------------------
 * Part 2 -- extensions.  *_dev functions take DEVICE pointers and a cudaStream_t passed as void* (NULL = default
 * stream); they run on the CURRENT device (cudaSetDevice), which must own the pointers and the stream -- workspaces, streams and
 * captured graphs are kept per device; they enqueue work and return without synchronising unless stated.  Return value: 1 ok / 0 error, except the
 * DR2 family which follows DR2_TV (always 0; check info[2]).
 * ------------------------------------------------------------------------------------------------------------------ */

int proxtv_device_count(void);                 /* usable CUDA devices (0 => every entry point fails loudly) */
const char *proxtv_last_error(void);           /* last error text of the calling thread ("" if none) */
const char *proxtv_version(void);

/* kernel family / Douglas-Rachford schedule (for measurements and tests).  0 auto: the lane-per-fiber streaming engine in slope
 * form (7) wherever the shape suits TMA tiling (16-byte aligned bases, row pitch a multiple of 16 bytes, positive weights, enough
 * fibers), else the chunked family; 1 sequential lane-per-fiber; 2 chunked speculative scan with the plain serial schedule;
 * 3 chunked with direct strided staging; 4 pipelined gather/scatter schedule; 5 transposeless schedule (scan kernels write both
 * layouts); 6 plain transposes around a fused row kernel; 7 the lane engine (kernels_lane.cu; DR2_TV: column pass over contiguous
 * fibers, row pass with the three operands combined at landing); 8 the lane engine with the transposed DR2_TV schedule (both passes
 * strided, arithmetic in the drains, results written transposed; what row-major images always use).  Engines 2, 4, 5, 6 are
 * bit-identical to each other (the reference's own arithmetic); 7 and 8 are bit-identical to each other and agree with the others to
 * ~1e-13 (same decisions, slope-form arithmetic).  The 1D entry points of Part 1 always use the bit-faithful chunked kernels.
 * Returns the previous value. */
int proxtv_set_engine(int engine);

/* Batched 1D prox over the fibers of a column-major array: nf fibers of len samples, fiber j starting at
 * (j / inc) * inc * len + (j % inc) with element stride inc (the reference's slicing rule, src/TVNDopt.cpp:184-188;
 * inc == 1: nf contiguous signals back to back).  lamv == NULL: uniform weight lam, else per-edge weights laid out the
 * same way with len-1 samples per fiber (batched tautString_TV1_Weighted).  Unweighted calls with at least 1024 fibers of at least
 * 64 samples whose shape suits TMA tiling run on the lane engine under engines 0 (auto, while the data passes its guard), 7 and 8:
 * the result is then the slope-form scan, within ~4e-15 of the reference's linearized taut string but not bit-identical to it.
 * Engine 2 (chunked) keeps these calls bit-identical to the reference. */
int proxtv_prox_fibers_dev_f64(const double *in, double *out, long long nf, int len, long long inc, double lam,
                               const double *lamv, void *stream);
int proxtv_prox_fibers_dev_f32(const float *in, float *out, long long nf, int len, long long inc, float lam,
                               const float *lamv, void *stream);
/* host-pointer form of the above (pageable or pinned memory); synchronous. */
int proxtv_prox_fibers_f64(const double *in, double *out, long long nf, int len, long long inc, double lam,
                           const double *lamv);
int proxtv_prox_fibers_f32(const float *in, float *out, long long nf, int len, long long inc, float lam,
                           const float *lamv);

/* DR2_TV on `batch` independent M x N images stored back to back.  info (host, 3 doubles, may be NULL).
 * row_major = 0: column-major images (the reference's layout); 1: row-major (C order) images -- the pass order
 * (axis 0 first, then axis 1) is the same, only the kernels' stride roles swap, so no transpose is ever made. */
int proxtv_DR2_TV_dev_f64(size_t M, size_t N, int batch, int row_major, const double *Y, double W1, double W2, double *out, int maxit,
                          double *info, void *stream);
int proxtv_DR2_TV_dev_f32(size_t M, size_t N, int batch, int row_major, const float *Y, float W1, float W2, float *out, int maxit,
                          double *info, void *stream);
int proxtv_DR2_TV_batched_f64(size_t M, size_t N, int batch, const double *Y, double W1, double W2, double *out, int maxit,
                              double *info);
int proxtv_DR2_TV_batched_f32(size_t M, size_t N, int batch, const float *Y, float W1, float W2, float *out, int maxit,
                              double *info);

/* DR2L1W_TV with device arrays (layouts as above; f32 is an extension the reference lacks). */
int proxtv_DR2L1W_TV_dev_f64(size_t M, size_t N, const double *Y, const double *W1, const double *W2, double *out, int maxit,
                             double *info, void *stream);
int proxtv_DR2L1W_TV_dev_f32(size_t M, size_t N, const float *Y, const float *W1, const float *W2, float *out, int maxit,
                             double *info, void *stream);

/* PD2_TV / PD_TV with device arrays y, x (lambdas, dims, ns, info stay on the host).  Synchronous (the stop test needs
 * one 8-byte read-back per iteration).  proxtv_PD_TV_* scale lambdas in place like PD_TV. */
int proxtv_PD2_TV_dev_f64(const double *y, double *lambdas, double *dims, double *x, double *info, int *ns, int nds,
                          int npen, int maxIters, void *stream);
int proxtv_PD2_TV_dev_f32(const float *y, double *lambdas, double *dims, float *x, double *info, int *ns, int nds, int npen,
                          int maxIters, void *stream);
int proxtv_PD_TV_dev_f64(const double *y, double *lambdas, double *dims, double *x, double *info, int *ns, int nds, int npen,
                         int maxIters, void *stream);
int proxtv_PD_TV_dev_f32(const float *y, double *lambdas, double *dims, float *x, double *info, int *ns, int nds, int npen,
                         int maxIters, void *stream);
int proxtv_PDR_TV_dev_f64(const double *y, double *lambdas, double *dims, double *x, double *info, int *ns, int nds, int npen,
                          int maxIters, void *stream);
int proxtv_PDR_TV_dev_f32(const float *y, double *lambdas, double *dims, float *x, double *info, int *ns, int nds, int npen,
                          int maxIters, void *stream);
int proxtv_PD_TV_f32(const float *y, double *lambdas, double *dims, float *x, double *info, int *ns, int nds, int npen,
                     int maxIters);                                          /* host pointers, float32 */

/* Launch accounting and optional CUDA-event timing per kernel class (0: prox over contiguous fibers, 1: prox over strided
 * fibers, 2: elementwise/reduction helpers).  Launch counters always run; event timing only while enabled.  read():
 * arrays of 3; ms = summed event time, launches = kernels launched, spans = timed brackets; synchronises the events. */
void proxtv_profile_enable(int on);
void proxtv_profile_reset(void);
void proxtv_profile_read(double *ms, long long *launches, long long *spans);

/* pinned host memory for the end-to-end path (cudaHostAlloc / cudaFreeHost) */
void *proxtv_host_alloc(size_t bytes);
void proxtv_host_free(void *p);
/* release the cached device workspace */
void proxtv_release_workspace(void);

/* Lane engine, one batched prox pass with the fused arithmetic `op` over the fibers (nf, len, inc) as above (inc == 1 only with op 0);
 * used by the multi-GPU driver (proxtv_b200/distributed.py) and by the measurement tools.  With x = prox(scan input):
 *   0 plain                 X = prox(A)
 *   1 DR second half        X = (C - B) + prox(A - (2 (C - B) - C))                 (operands combined when their tiles land)
 *   2 DR final projection   X = prox(A - (C - B))
 *   3 DR first half, T      x = prox(A); d = C - x; X^T = B - (2 d - C); X2^T = d   (operands read in the drain; ^T: results written
 *   4 DR final, T           X^T = B - (C - prox(A))                                  fiber-major, element (fiber f, row r) at f * len + r)
 *   5 DR second half, T     X^T = B + prox(A)
 *   6 plain, T              X^T = prox(A)
 * Returns 0 when the shape does not suit the engine (bases and row pitch multiples of 16 bytes).  tuning: chunk length (0 = automatic),
 * halo rows, kernel variant (-1 = default per storage type); stats: fibers that went through the repair path since the last reset. */
int proxtv_lane_prox_dev_f64(int op, const double *A, const double *B, const double *C, double *X, long long nf, int len,
                             long long inc, double lam, void *stream);
int proxtv_lane_prox_dev_f32(int op, const float *A, const float *B, const float *C, float *X, long long nf, int len,
                             long long inc, float lam, void *stream);
/* same with a second result array (the ops that write two results: 3 = first half of a Douglas-Rachford iteration, transposed) */
int proxtv_lane_prox2_dev_f64(int op, const double *A, const double *B, const double *C, double *X, double *X2, long long nf, int len,
                              long long inc, double lam, void *stream);
int proxtv_lane_prox2_dev_f32(int op, const float *A, const float *B, const float *C, float *X, float *X2, long long nf, int len,
                              long long inc, float lam, void *stream);
void proxtv_lane_tuning(int clen, int halo, int variant);
unsigned long long proxtv_lane_stats(int reset);
/* Under engine 0 (auto) the solvers use the lane engine only while the data keeps segments short -- penalty not larger than about the
 * mean step |y[i+1] - y[i]| of (a sample of) the input, measured with one small kernel and one stream synchronisation per call --
 * and the chunked engine otherwise.  Last decision on the current device: 1 lane, 0 chunked, -1 none taken. */
int proxtv_lane_guard_last(void);
/* tools: device buffer of 4 x cap_tasks uint64 that receives, per warp task of the next launches, {start ns, scan end ns, end ns, SM id}
 * (globaltimer); NULL switches the log off. */
void proxtv_lane_tasklog(unsigned long long *dev, long long cap_tasks);

#ifdef __cplusplus
}
#endif
#endif /* PROXTV_B200_H */
