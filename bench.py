#!/usr/bin/env python
"""bench.py -- headline benchmark of proxtv_b200:  tv1_2d (DR2_TV) Mpixels/s on 4096 x 4096 float64 images, lambda = 0.2.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--size M] [--engine auto|lane|lane-t|chunked|seq]
                    [--workload cfg2|cfg3|cfg4|cfg5|split] [--batch B] [--pieces P] [--dump-outputs DIR]

One "step" = one complete solve (35 Douglas-Rachford iterations + the final projection pair, 72 fiber passes) of one
4096 x 4096 image per GPU (BASELINE.json configs[1]; synthetic piecewise-constant + Gaussian-noise input, SURVEY.md 8d).
N > 1 (launched by torchrun, one rank per GPU): every rank solves its own independent image -- the path has no data-path
collective (SURVEY.md 8e: "replicas only" for a single array), so scaling is weak and `value` aggregates all ranks.

Rank 0 prints ONE JSON line.  Keys beyond the base contract:
  roofline      dominant kernel class (by summed CUDA-event time inside the timed steps): algorithmic bytes per launch /
                average launch duration, against MEASURED_PEAKS.json's hbm_gbs (fallback 6650 GB/s, flagged).
  roofline_solve  the north-star figure: whole-solve algorithmic bytes (1728 B/pixel, SURVEY.md 8d) / solve time.
  e2e           same metric through the reference-facing C ABI call DR2_TV() with pinned HOST buffers (H2D + D2H inside).
  cpu_baseline  the reference's own OpenMP DR2_TV (oracle/_ref, compiled from the unmodified sources) on this box's host
                cores (thread count from a short sweep), N = 1 only, one solve of the FULL image.
--impl reference times only that CPU implementation (rank 0 alone), same metric/config.
--workload cfg3 | cfg4 | cfg5: the other BASELINE.json configurations (cfg5 over N GPUs: NCCL scatter / gather of image slabs,
pipelined); --workload split: ONE image over all N ranks (strong scaling; two all-to-alls per iteration).
--dump-outputs DIR (cfg2): after the timed steps, rank 0 writes what its last timed step returned, DIR/x.npy (the solved image, or
                a fixed seeded sample of its rows when it is larger than 32 MiB) and DIR/info.npy (DR2_TV's info[]), float64.  The
                inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_PIXEL_SOLVE = lambda b, maxit=35: b * (1 + 6 * maxit + 5)      # noqa: E731  SURVEY.md 8d: M*N*b*(1 + 6*maxit + 5)
LAM = 0.2
DUMP_BYTES = 32 << 20


def dump_outputs(d, image, info):
    """--dump-outputs: the image whole if it fits DUMP_BYTES, else the rows of a fixed seeded sample (sorted), float64."""
    M, N = image.shape
    if image.nbytes > DUMP_BYTES:
        image = image[np.sort(np.random.default_rng(0).choice(M, DUMP_BYTES // (8 * N), replace=False))]
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "x.npy"), np.ascontiguousarray(image, dtype=np.float64))
    np.save(os.path.join(d, "info.npy"), np.asarray(info, dtype=np.float64))


def ncu_traffic(cls=-1, lane_t=False):
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel from the committed ncu --set full capture.
    cls 0 / 1: the lane engine's column / row pass (profiles/r2_lane_staged_ncu_full.csv, or r2_lane_t_ncu_full.csv for the transposed
    schedule; columns launch0 = row pass, launch1 = column pass); -1: round 1's chunked scan (mean of its two captured launches)."""
    try:
        path = "r1_contig_kernel_ncu_full.csv" if cls < 0 else ("r2_lane_t_ncu_full.csv" if lane_t else "r2_lane_staged_ncu_full.csv")
        r = w = None
        for line in open(os.path.join(ROOT, "profiles", path)):
            p = line.strip().split(",")
            if p[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                scale = 1e6 if p[1] == "Mbyte" else 1e9 if p[1] == "Gbyte" else 1e3 if p[1] == "Kbyte" else 1.0
                vals = [float(x) for x in p[2:]]
                v = (sum(vals) / len(vals) if cls < 0 else vals[1 - cls]) * scale      # r2 file: launch0 = row pass (class 1), launch1 = column pass (class 0)
                if p[0] == "dram__bytes_read.sum": r = v
                else: w = v
        return r + w if r is not None and w is not None else None
    except Exception:  # noqa: BLE001
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index; self.proc = None; self.path = "/tmp/proxtv_clocks_%d_%d.csv" % (os.getpid(), index)

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            p = [q.strip() for q in line.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def host_threads():
    """Threads this process may use: scheduler affinity, capped by the cgroup CPU quota when there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:  # noqa: BLE001
        pass
    return max(1, n)


def best_threads(R, Y, lam):
    """The reference's OpenMP DR2_TV is not fastest with every hardware thread (oversubscription, NUMA): time one solve of a
    4096 x 512 strip (full-length first-pass fibers) per candidate thread count and keep the best."""
    nmax = host_threads()
    cands = sorted({c for c in (8, 16, 32, 64, nmax) if c <= nmax} | {nmax})
    S = np.asfortranarray(Y[:, :max(Y.shape[1] // 8, 8)])
    best, sweep = None, {}
    for c in cands:
        t0 = time.perf_counter(); R.dr2_tv(S, lam, n_threads=c); dt = time.perf_counter() - t0
        sweep[c] = S.size / dt / 1e6
        if best is None or sweep[c] > sweep[best]:
            best = c
    return best, sweep


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation (OpenMP DR2_TV), all host cores, rank 0 only."""
    if rank != 0:
        return
    from oracle import oracle as O
    try:
        R = O.Ref(); kind = "reference"
    except Exception:  # noqa: BLE001
        R = O.Port(); kind = "port"
    M = args.size
    Y = O.gen_cfg2(M, M, seed=0)
    # the FULL image, every step; thread count chosen once from a short sweep (stated in cpu_baseline)
    cores, sweep = best_threads(R, Y, LAM)
    S = Y
    for _ in range(args.warmup):
        R.dr2_tv(S, LAM, n_threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        R.dr2_tv(S, LAM, n_threads=cores)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    v = S.size / dt / 1e6
    sample = "full %dx%d image per step; %d OpenMP threads (best of sweep %s on a %dx%d strip; %d threads available)" % (
        M, M, cores, {k: round(x, 2) for k, x in sweep.items()}, M, max(M // 8, 8), host_threads())
    print(json.dumps({
        "impl": "reference", "metric": "tv1_2d Mpixels/s", "value": v, "unit": "Mpixels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "tv1_2d DR2_TV %dx%d f64 lambda=%.1f, 35 iterations + final projection" % (M, M, LAM)},
        "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def run_other_workload(args, rank, world, local):
    """--workload cfg3 | cfg4 | cfg5: the other BASELINE.json configurations, same JSON contract (value = whole-job throughput,
    device-resident; roofline = the workload's algorithmic bytes, SURVEY.md 8d, over the measured step time)."""
    import torch
    import torch.distributed as dist
    import proxtv_b200 as ptv
    import synth_inputs as S

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = ptv.require_device()
    peak, peak_src = peaks()
    wl = args.workload
    vp = C.c_void_p

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    extra = {}
    if wl == "cfg3":                    # tv1w_1d on 65536 signals x 4096, per-element weights, f64 (new batched API)
        B, L = args.batch or 65536, 4096
        g = torch.Generator(device="cuda"); g.manual_seed(rank)
        X = (torch.randn((B, L // 64), device="cuda", dtype=torch.float64, generator=g) * 2).repeat_interleave(64, dim=1) \
            + torch.randn((B, L), device="cuda", dtype=torch.float64, generator=g) * 0.5
        Wt = torch.rand((B, L - 1), device="cuda", dtype=torch.float64, generator=g) * 0.9 + 0.1
        out = torch.empty_like(X)
        st = vp(torch.cuda.current_stream().cuda_stream)
        step = lambda: lib.proxtv_prox_fibers_dev_f64(vp(X.data_ptr()), vp(out.data_ptr()), B, L, 1, 0.0, vp(Wt.data_ptr()), st)  # noqa: E731
        units, unit, metric = B * L, "Msamples/s", "tv1w_1d Msamples/s"
        alg_bytes = B * (L * 16 + (L - 1) * 8)
        workload = "tv1w_1d batch %d x %d f64, per-element weights U(0.1,1)" % (B, L); dtype = "f64"
        h2d, d2h = B * (2 * L - 1) * 8, B * L * 8
    elif wl == "cfg4":                  # tvgen 3D anisotropic TV (PD_TV), 512 x 512 x 256 f32
        shp = (512, 512, 256)
        V = S.gen_cfg4(shp, seed=rank)
        Vd = torch.from_numpy(np.ascontiguousarray(V.astype(np.float32).transpose(2, 1, 0))).cuda(); outd = torch.empty_like(Vd)
        ns = np.array(shp, dtype=np.int32); dims = np.array([1.0, 2.0, 3.0]); inf = np.zeros(3)

        def step():
            lam = np.array([0.2, 0.2, 0.2])
            lib.proxtv_PD_TV_dev_f32(vp(Vd.data_ptr()), vp(lam.ctypes.data), vp(dims.ctypes.data), vp(outd.data_ptr()), vp(inf.ctypes.data),
                                     vp(ns.ctypes.data), 3, 3, 0, None)
        units, unit, metric = int(np.prod(shp)), "Mvoxels/s", "tvgen PD_TV Mvoxels/s"
        k = 3
        alg_bytes = None                 # needs the iteration count: filled in after the run
        workload = "tvgen PD_TV %dx%dx%d f32, ws=(.2,.2,.2), ds=(1,2,3)" % shp; dtype = "f32 storage, f64 scan arithmetic"
        h2d = d2h = units * 4
    elif wl == "split":                 # ONE image split over all ranks (SURVEY 8f N3): column / row slabs, two all-to-alls per iteration
        from proxtv_b200.distributed import tv1_2d_single_sharded
        H = args.size
        x = None
        if rank == 0:
            g = torch.Generator(device="cuda"); g.manual_seed(0)
            lv = torch.randn((H // 64, H // 64), device="cuda", dtype=torch.float64, generator=g).repeat_interleave(64, dim=0).repeat_interleave(64, dim=1)
            x = (lv + torch.randn((H, H), device="cuda", dtype=torch.float64, generator=g) * 0.3).t()      # column-major view, like the reference's arrays
        tm = {}
        step = (lambda: tv1_2d_single_sharded(x, LAM)) if world > 1 else (lambda: ptv.tv1_2d(x, LAM))  # noqa: E731
        units, unit, metric = H * H, "Mpixels/s", "tv1_2d single image Mpixels/s"
        alg_bytes = units * B_PER_PIXEL_SOLVE(8)
        workload = "tv1_2d DR2_TV ONE %dx%d f64 image over %d GPU(s), lambda=%.1f; %s" % (
            H, H, world, LAM, "column / row slabs, 2 NCCL all-to-alls per iteration, scatter + gather from/to rank 0 inside the timed region" if world > 1 else "single GPU")
        dtype = "f64"
        h2d = d2h = 0
    else:                               # cfg5: tv1_2d on a batch of 2048 x 2048 f32 images, 128 per GPU, NCCL scatter / gather of images
        from proxtv_b200.distributed import tv1_2d_batched_sharded
        per_gpu = args.batch or 128; H = 2048; B = per_gpu * world
        x = None
        if rank == 0:
            g = torch.Generator(device="cuda"); g.manual_seed(0)
            x = torch.empty((B, H, H), device="cuda", dtype=torch.float32)
            for b0 in range(0, B, 32):
                nb = min(32, B - b0)
                lv = torch.randn((nb, H // 64, H // 64), device="cuda", generator=g).repeat_interleave(64, dim=1).repeat_interleave(64, dim=2)
                x[b0:b0 + nb] = lv + torch.randn((nb, H, H), device="cuda", generator=g) * 0.3
        tm = {}
        step = (lambda: tv1_2d_batched_sharded(x, LAM, pieces=args.pieces, timings=tm)) if world > 1 else (lambda: ptv.tv1_2d_batched(x, LAM))  # noqa: E731
        units, unit, metric = B * H * H, "Mpixels/s", "tv1_2d batched Mpixels/s"
        alg_bytes = units * B_PER_PIXEL_SOLVE(4)
        workload = "tv1_2d DR2_TV batch %d x %dx%d f32 (%d images per GPU), lambda=%.1f; %s" % (
            B, H, H, per_gpu, LAM, ("NCCL scatter + gather of image slabs from/to rank 0, %d pipelined pieces" % args.pieces) if world > 1 else "single GPU, no collective")
        dtype = "f32 storage, f64 scan arithmetic"
        h2d = d2h = 0
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    clocks = ClockSampler(local); clocks.start()
    lib.proxtv_profile_reset()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    stt = torch.cuda.current_stream()
    barrier(); e0.record(stt)
    for _ in range(args.steps):
        step()
    e1.record(stt); barrier()
    ms = e0.elapsed_time(e1)
    kms = (C.c_double * 3)(); kl = (C.c_longlong * 3)(); ks = (C.c_longlong * 3)()
    lib.proxtv_profile_read(kms, kl, ks)
    clk = clocks.stop()
    tmax = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_step = float(tmax.item()) / args.steps
    total_units = units if wl in ("cfg5", "split") else units * world
    if wl == "cfg4":
        iters = int(inf[0]); extra["iterations"] = iters; extra["stop"] = float(inf[1])
        alg_bytes = units * 4 * ((k + 1) + iters * (5 * k + 2))
    if rank == 0:
        ach = alg_bytes * (1 if wl in ("cfg5", "split") else world) / (ms_step * 1e-3) / 1e9 / world
        line = {"metric": metric, "value": total_units / (ms_step * 1e-3) / 1e6, "unit": unit, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if wl == "split" else "weak", "vs_baseline": None,
                "dtype": dtype, "data": "synthetic", "config": dict({"workload": workload}, **extra),
                "roofline": {"bound": "hbm", "kernel": "whole step (all kernels of the workload)", "achieved": ach, "peak": peak, "unit": "GB/s per GPU",
                             "frac": ach / peak, "algorithmic_bytes_per_step_per_gpu": alg_bytes / (world if wl in ("cfg5", "split") else 1), "peak_source": peak_src, "traffic": None},
                "gpu_launches": (args.steps * 71 if (wl == "split" and world > 1) else int(sum(kl[i] for i in range(3))))   # split: 35 column + 36 row lane passes per solve on every rank, issued through proxtv_lane_prox_dev_*
                                , "clocks": clk,
                "e2e": {"value": None, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "note": "device-resident workload (inputs generated on the GPU); the headline e2e number is config 2's"}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--engine", default="auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5", "split"])
    ap.add_argument("--batch", type=int, default=0, help="cfg3: signals; cfg5: images per GPU (0 = BASELINE.json's)")
    ap.add_argument("--pieces", type=int, default=4, help="cfg5: pipelined transfer pieces per GPU slab")
    ap.add_argument("--dump-outputs", metavar="DIR", help="cfg2: write the last timed step's result to DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps: at least one timed step")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "cfg2"):
        ap.error("--dump-outputs: the cfg2 workload of --impl ours only")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload != "cfg2":
        run_other_workload(args, rank, world, local)
        return

    import torch
    import torch.distributed as dist
    import proxtv_b200 as ptv
    import synth_inputs as S               # seeded input generators (SURVEY 8d); oracle/ is imported by the cpu_baseline leg only

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = ptv.require_device()
    ptv.set_engine(args.engine)
    M = args.size
    Yh = S.gen_cfg2(M, M, seed=rank)                                     # F-ordered float64, one image per rank
    Yd = torch.from_numpy(np.ascontiguousarray(Yh.T)).cuda()             # device copy, column-major image
    out = torch.empty_like(Yd)
    info = np.zeros(3)
    st = torch.cuda.current_stream()
    stp = C.c_void_p(st.cuda_stream)

    def solve():
        lib.proxtv_DR2_TV_dev_f64(M, M, 1, 0, C.c_void_p(Yd.data_ptr()), LAM, LAM, C.c_void_p(out.data_ptr()), 0,
                                  C.c_void_p(info.ctypes.data), stp)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        solve()
    barrier()
    assert info[2] == 0, "DR2_TV reported an error: " + ptv._lib.last_error()
    # ---- timed region: exactly K steps, device-resident, CUDA events on the launching stream (launch counters only) ----
    lib.proxtv_profile_reset()
    clocks = ClockSampler(local); clocks.start()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(args.steps):
        solve()
    e1.record(st)
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out.cpu().numpy().T, info)        # out holds the column-major image
    kms = (C.c_double * 3)(); kl = (C.c_longlong * 3)(); ks = (C.c_longlong * 3)()
    lib.proxtv_profile_read(kms, kl, ks)
    launches_timed_region = int(sum(kl[i] for i in range(3)))
    # ---- per-kernel timing for the roofline: K more steps with CUDA events around EVERY launch, on the serial schedule
    #      (engine 'chunked': same kernels, no stream overlap) so that a launch's duration is the kernel's own ----
    ptv.set_engine("lane" if args.engine == "auto" else args.engine)
    lib.proxtv_profile_reset(); lib.proxtv_profile_enable(1)
    for _ in range(args.steps):
        solve()
    barrier()
    lib.proxtv_profile_enable(0)
    lib.proxtv_profile_read(kms, kl, ks)
    ptv.set_engine(args.engine)
    tmax = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_step = float(tmax.item()) / args.steps
    value = world * M * M / (ms_step * 1e-3) / 1e6

    # ---- end to end through the reference-facing C ABI (host buffers, pinned; H2D + D2H inside the timed region) ----
    nbytes = M * M * 8
    hin = lib.proxtv_host_alloc(nbytes); hout = lib.proxtv_host_alloc(nbytes)
    C.memmove(hin, Yh.ctypes.data, nbytes)
    einfo = np.zeros(3)

    def solve_host():
        lib.DR2_TV(M, M, C.c_void_p(hin), LAM, LAM, 1.0, 1.0, C.c_void_p(hout), 1, 0, C.c_void_p(einfo.ctypes.data))

    solve_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        solve_host()                       # synchronous: returns after the D2H copy completed
    torch.cuda.synchronize()
    et = torch.tensor([(time.perf_counter() - t0) * 1e3], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
    e2e_value = world * M * M / (float(et.item()) / args.steps * 1e-3) / 1e6
    # the numpy drop-in: prox_tv.tv1_2d's surface on a pageable F-ordered ndarray (what a prox_tv user calls)
    ptv.tv1_2d(Yh, LAM)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res_np = ptv.tv1_2d(Yh, LAM)
    np_t = torch.tensor([(time.perf_counter() - t0) * 1e3], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(np_t, op=dist.ReduceOp.MAX)
    e2e_numpy = world * M * M / (float(np_t.item()) / args.steps * 1e-3) / 1e6
    clk = clocks.stop()
    res = np.ctypeslib.as_array(C.cast(hout, C.POINTER(C.c_double)), shape=(M * M,))
    same = bool(np.array_equal(res, out.cpu().numpy().ravel()))
    lib.proxtv_host_free(hin); lib.proxtv_host_free(hout)

    if rank == 0:
        peak, peak_src = peaks()
        names = ["prox_contiguous_fibers", "prox_strided_fibers", "elementwise"]
        lane_t = args.engine == "lane-t"
        lane = args.engine in ("auto", "lane") or lane_t
        # algorithmic bytes per launch of each kernel class for this workload (DESIGN.md "Kernels"), in f64 sweeps of the image.
        # lane engine: class 0 = k_lane CONTIG (column pass: 1R + 1W), class 1 = k_lane STRIDED with the fused Douglas-Rachford
        # arithmetic (row pass: reads Y, t, x_cols, writes t': 3R + 1W; the final projection pass has the same traffic).
        # chunked engines: both prox classes are the chunked scan (1R + 1W); gather (2R+1W) / scatter+combine (4R+1W) average 4.
        # engine lane-t: class 0 = k_lane STRIDED LOP_DRA over the row-major copies (reads t, Y; writes u, d transposed: 2R + 2W),
        # class 1 = k_lane STRIDED LOP_DRB (reads u, d; writes t' transposed: 2R + 1W).
        sweeps = {0: 4.0 if lane_t else 2.0, 1: (3.0 if lane_t else 4.0) if lane else 2.0, 2: 4.0}
        kname = {0: ("k_lane<STRIDED, LOP_DRA> (column pass over row-major copies, results transposed)" if lane_t else
                     "k_lane<CONTIG, plain> (column pass)") if lane else "k_prox_chunked_contig",
                 1: ("k_lane<STRIDED, LOP_DRB> (row pass, result transposed)" if lane_t else
                     "k_lane<STRIDED, fused Douglas-Rachford> (row pass)") if lane else "k_prox_chunked_contig (on gathered rows)", 2: "elementwise"}
        if lane:
            dom = max(range(3), key=lambda i: kms[i])
            avg_ms = kms[dom] / max(ks[dom], 1)
        else:
            scan_ms, scan_n = kms[0] + kms[1], ks[0] + ks[1]
            dom = 0 if scan_ms >= kms[2] else 2
            avg_ms = (scan_ms / max(scan_n, 1)) if dom == 0 else kms[2] / max(ks[2], 1)
        ach = sweeps[dom] * M * M * 8 / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
        per_class = {names[i]: {"kernel": kname[i], "ms_per_step": kms[i] / args.steps, "launches_per_step": ks[i] / args.steps,
                                "avg_launch_ms": kms[i] / max(ks[i], 1),
                                "achieved_GBs": (sweeps[i] * M * M * 8 / (kms[i] / max(ks[i], 1) * 1e-3) / 1e9) if kms[i] > 0 else 0.0,
                                "frac": (sweeps[i] * M * M * 8 / (kms[i] / max(ks[i], 1) * 1e-3) / 1e9 / peak) if kms[i] > 0 else 0.0}
                     for i in range(3)}
        solve_bytes = B_PER_PIXEL_SOLVE(8) * M * M
        line = {
            "metric": "tv1_2d Mpixels/s", "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "tv1_2d DR2_TV %dx%d f64 lambda=%.1f, 35 iterations + final projection, one image per GPU"
                                   % (M, M, LAM), "engine": args.engine + (" (lane-per-fiber slope-form engine, kernels_lane.cu)" if lane else ""),
                       "l2": "working set 4 x %d MiB > 126 MB L2 (inputs larger than L2, no flush)" % (nbytes >> 20)},
            "roofline": {"bound": "hbm", "kernel": kname[dom], "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "traffic": ncu_traffic(dom if lane else -1, lane_t) if M == 4096 else None,
                         "traffic_source": ("profiles/r2_lane_t_ncu_full.csv" if lane_t else "profiles/r2_lane_staged_ncu_full.csv") + " (ncu --set full, same kernels and shape)" if lane else "profiles/r1_contig_kernel_ncu_full.csv",
                         "algorithmic_bytes_per_launch": sweeps[dom] * M * M * 8, "peak_source": peak_src,
                         "avg_launch_ms": avg_ms, "launches_timed": int(ks[dom]),
                         "timing_region": "%d additional steps right after the timed region, same kernels launched one by one (no graph replay), CUDA events around every launch" % args.steps,
                         "classes": per_class},
            "roofline_solve": {"algorithmic_bytes": solve_bytes, "achieved": solve_bytes / (ms_step * 1e-3) / 1e9,
                               "peak": peak, "unit": "GB/s", "frac": solve_bytes / (ms_step * 1e-3) / 1e9 / peak},
            "e2e": {"value": e2e_value, "unit": "Mpixels/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                    "api": "DR2_TV() C ABI, pinned host buffers", "matches_device_path": same,
                    "numpy_dropin_value": e2e_numpy, "numpy_dropin_api": "proxtv_b200.tv1_2d(ndarray): pageable memory, allocates its result"},
            "gpu_launches": launches_timed_region,
            "clocks": clk,
        }
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as O          # the cpu_baseline leg: the one place the measured arm's process touches oracle/
            try:
                R = O.Ref(); kind = "reference"
            except Exception:  # noqa: BLE001
                R = O.Port(); kind = "port"
            cores, sweep = best_threads(R, Yh, LAM)
            t0 = time.perf_counter(); R.dr2_tv(Yh, LAM, n_threads=cores); dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": Yh.size / dt / 1e6, "unit": "Mpixels/s", "cores": cores, "kind": kind,
                                    "sample": "one DR2_TV solve of the full %dx%d image, %d OpenMP threads (best of sweep %s Mpixels/s on a %dx%d strip; %d threads available)"
                                              % (M, M, cores, {k: round(x, 2) for k, x in sweep.items()}, M, max(M // 8, 8), host_threads())}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
