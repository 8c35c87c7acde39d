#!/usr/bin/env python
"""bench.py -- headline benchmark: BA residual+Jacobian evaluations per second (BASELINE.json `metric`).

    python bench.py --gpus 1 --steps 20 --warmup 3                 # ours, 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference --steps 5 --warmup 1          # the reference's CPU path (oracle port; Ceres itself is not installable)

Workload (config.workload): BASELINE.json configs[2] -- ONE synthetic problem of 100 cameras / 200k points / 1.6M observations.
`--gpus N` is STRONG scaling, as BASELINE.json states it ("1/2/4/8 x B200 NCCL-reduced camera system"): the 200k points are
sharded over the N ranks, the 100 cameras are replicated, the reduced camera system is summed over ranks once per LM iteration.
(Weak scaling -- 200k points per rank -- is measured too and reported under the key "weak".)  `--workload cfg2` selects
configs[1] (20 / 10k / 80k).
A step = ONE Levenberg-Marquardt iteration: residual+Jacobian evaluation of every observation fused with the per-point
Schur elimination (K3a/K3b), the rank sum, the dense Cholesky solve (K4), back-substitution and evaluation of the candidate.
Every iteration evaluates all observations, so evals/s = observations * iterations / time.
`--dump-outputs DIR` writes what the timed pass returned after its last iteration (cameras.npy [nc,6], points.npy [np,3],
focal.npy [1], all float64) so that two builds can be compared output for output; the inputs are seeded, identical from run to run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "BA residual+Jacobian evals/sec"
UNIT = "evals/s"
PREHEAT_ITERS = 120
L2_FLUSH_MB = 192


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(nc, npts, nobs):
    """SURVEY.md section 8(d): per observation 16 B (float2 xy + int32 cam + int32 CSR share); per point 24 B read + 24 B
    write + 4 B offset; cameras 48 B r/w; S + rhs written once.  cfg3: ~38.9 MB per residual+Jacobian+Schur pass."""
    n = 6 * nc + 1
    return 16 * nobs + 52 * npts + 96 * nc + n * (n + 1) * 8


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  The region is ~20 ms, so NVML is polled from a thread every
    few milliseconds (the ctypes call that runs the solver releases the GIL); `nvidia-smi -lms` is the fallback without pynvml."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        import threading
        self.sm, self.mx, self.reasons, self.source = [], [], set(), None
        self.p = self.f = self.thread = None
        self._stop = False
        # NVML queries take the driver lock: polled every millisecond they delayed this rank's kernel launches enough to
        # stall a 2-GPU step from 1.3 to 10 ms (every rank spins on its peers' flags).  4 ms keeps >= 4 samples in the region.
        period = float(os.environ.get("SFMB200_BENCH_CLOCK_PERIOD_MS", "2")) * 1e-3
        if os.environ.get("SFMB200_BENCH_CLOCKS", "nvml") == "off":
            return
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(gpu_index)
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self._stop:
                    try:
                        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))); self.mx.append(mx)
                        r = int(get_reasons(h))
                        for k, bit in names.items():
                            if r & bit:
                                self.reasons.add(k)
                    except Exception:
                        pass
                    time.sleep(period)
            self.thread = threading.Thread(target=loop, daemon=True); self.thread.start(); self.source = f"nvml thread, {period * 1e3:g} ms period"
        except Exception:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            try:
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                          stdout=self.f, stderr=subprocess.DEVNULL); self.source = "nvidia-smi -lms 20"
            except Exception:
                self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": self.source}
        if self.thread is not None:
            self._stop = True; self.thread.join(timeout=2)
        elif self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
            self.f.flush(); self.f.seek(0)
            for line in self.f.read().splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    self.sm.append(float(c[1])); self.mx.append(float(c[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            try:
                os.unlink(self.f.name)
            except OSError:
                pass
        if self.sm:
            out.update(sm_mhz=float(np.median(self.sm)), sm_max_mhz=float(np.max(self.mx)), reasons=sorted(self.reasons), samples=len(self.sm))
        return out


def make_shard(workload, rank):
    """Weak-scaling shard: every rank its own points (rank 0 = THE problem of the strong-scaling run), shared cameras."""
    from sfm_toy_library_b200 import synth
    cfg = synth.BA_CONFIGS[workload]
    return synth.make_ba_problem(seed=0, point_seed=1000 + rank if rank else 0, **cfg)


def fixed_iteration_options(capi_or_oracle, iters, **kw):
    """Exactly `iters` LM iterations: the three tolerance tests are disabled, the time cap lifted."""
    return capi_or_oracle.ba_default_options(max_num_iterations=iters, max_solver_time_in_seconds=0.0, function_tolerance=-1.0,
                                             parameter_tolerance=-1.0, gradient_tolerance=-1.0, **kw)


SOLVE_ITERS = 20     # LM iterations per solve inside a pass: with the tolerances off a converged solve keeps rejecting steps and
                     # Ceres' "minimum trust region radius" test ends it after ~55 iterations on cfg 3, so long passes restart from x0


def run_steps(prob, capi, k, **kw):
    """Exactly k LM iterations as solves of at most SOLVE_ITERS (reset to x0 in between); summed summary fields."""
    tot = None
    done = 0
    while done < k:
        n = min(SOLVE_ITERS if k > SOLVE_ITERS + 4 else k, k - done)
        if done:
            prob.reset()
        s = prob.run(fixed_iteration_options(capi, n, **kw))
        if s["num_iterations"] != n:
            raise RuntimeError(f"solve stopped after {s['num_iterations']} of {n} iterations: {s['message']}")
        if tot is None:
            tot = dict(s)
        else:
            for key in ("num_iterations", "num_successful_steps", "num_unsuccessful_steps", "num_jacobian_passes", "num_linear_solves", "schur_ms_total",
                        "schur_launches", "pair_ms_total", "pair_launches", "camera_ms_total", "solve_ms_total", "flush_ms_total", "kernel_launches"):
                tot[key] += s[key]
        done += n
    return tot


def dump_outputs(out_dir, cams, pts, focal):
    """The BA result a caller of the timed path receives, as DIR/<name>.npy (float64; cfg3: 4.8 MB in all)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, x in (("cameras", cams), ("points", pts), ("focal", [focal])):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(x, np.float64))


# ----------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path.  The C++ reference cannot be built (no OpenCV/Ceres/Boost in
    the image), so this is the oracle port: Ceres-equivalent LM + DENSE_SCHUR with dual-number (autodiff) Jacobians --
    what adjustBundle does (SfMBundleAdjustmentUtils.cpp:91-94, :171-179) -- on all host threads (the reference itself
    leaves Ceres at 1 thread)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle
    cores = os.cpu_count() or 1
    p = make_shard(args.workload, 0)
    a = (p["cams"], p["pts"], p["focal"], p["obs_xy"], p["obs_cam"], p["pt_off"])
    sample = f"{args.workload} full problem ({p['nc']} cams / {p['np']} pts / {p['nobs']} obs), one LM iteration per step"
    # bound the run: probe one iteration; if a step is too slow for (warmup+steps) to finish in ~4 min, subsample points
    # "all the host threads it can use": the port stops scaling well before 100+ threads, so pick the fastest count
    probe, best = None, cores
    for cand in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16)}, reverse=True):
        t0 = time.perf_counter()
        oracle.ba_solve(*a, fixed_iteration_options(oracle, 1, jacobian_mode=0, num_threads=cand))
        dt1 = (time.perf_counter() - t0) / 2.0        # a 1-iteration solve evaluates the Jacobian twice
        if probe is None or dt1 < probe:
            probe, best = dt1, cand
    cores = best
    budget = 240.0 / max(1, args.steps + args.warmup + 2)
    if probe > budget:
        frac = max(0.02, budget / probe)
        npts = max(1000, int(p["np"] * frac))
        nobs = int(p["pt_off"][npts])
        a = (p["cams"], p["pts"][:npts], p["focal"], p["obs_xy"][:nobs], p["obs_cam"][:nobs], p["pt_off"][:npts + 1])
        sample = f"{args.workload} first {npts} points / {nobs} obs (bounded sample), one LM iteration per step"
    else:
        nobs = p["nobs"]
    if args.warmup:
        oracle.ba_solve(*a, fixed_iteration_options(oracle, args.warmup, jacobian_mode=0, num_threads=cores))
    t0 = time.perf_counter()
    cams, pts, focal, s = oracle.ba_solve(*a, fixed_iteration_options(oracle, args.steps, jacobian_mode=0, num_threads=cores))
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cams, pts, focal)
    value = nobs * s["num_iterations"] / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, s["num_iterations"]), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"BASELINE.json configs[{2 if args.workload == 'cfg3' else 1}] ({args.workload})", "cams": p["nc"],
                       "points": p["np"], "observations": p["nobs"], "solver": "LM + DENSE_SCHUR, autodiff (dual numbers), Ceres defaults"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from sfm_toy_library_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = capi.Context(local)
    if world > 1:
        uid = [capi.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()

    from sfm_toy_library_b200 import dist as sdist
    p_full = make_shard(args.workload, 0)                 # THE problem (every rank generates the same one)
    p = sdist.shard_ba_problem(p_full, rank, world) if world > 1 else p_full      # strong scaling: this rank's points
    a = (p["cams"], p["pts"], p["focal"], p["obs_xy"], p["obs_cam"], p["pt_off"])
    prob = ctx.ba_problem(*a)
    exchange = "none"
    if world > 1:
        exchange = "nccl"
        if os.environ.get("SFMB200_EXCHANGE", "peer") == "peer":
            try:
                if sdist.attach_peers(prob, dist):
                    exchange = "peer-memory kernels (CUDA IPC, NVLink loads)"
            except Exception as e:                      # e.g. no peer access between the devices: NCCL still works
                sys.stderr.write(f"peer attach failed ({e}); using NCCL\n")
    flush = torch.empty(L2_FLUSH_MB << 20, dtype=torch.uint8, device="cuda")

    # ---- value: inputs resident in HBM; W warm-up iterations, then exactly K timed LM iterations -------------------
    # The GPU idles for seconds while the host builds the synthetic problem; its clocks need ~100 ms of load to settle
    # (first solves after an idle period measured up to 1.8x slower).  Pre-heat with untimed LM iterations, then the W warm-up steps.
    # Both untimed phases run with the timed pass's options: its first use creates the profiling events and the flush scratch.
    run_steps(prob, capi, PREHEAT_ITERS, profile=1, l2_flush_mb=L2_FLUSH_MB); prob.reset()
    if args.warmup:
        run_steps(prob, capi, args.warmup, profile=1, l2_flush_mb=L2_FLUSH_MB)
    prob.reset()
    with torch.cuda.stream(stream):
        flush.zero_()                                   # L2 flush before the timed region (inputs < L2 on one GPU)
    barrier()
    launches0 = ctx.kernel_launches
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t0 = time.perf_counter()
    s = run_steps(prob, capi, args.steps, profile=1, l2_flush_mb=L2_FLUSH_MB)
    e1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    dev_ms_raw = e0.elapsed_time(e1)
    # the L2 flush writes sit between the iterations on the same stream; they are benchmark hygiene, not part of the step,
    # so their own CUDA-event time (summary.flush_ms_total) is taken out of the bracket
    flush_ms = float(s["flush_ms_total"])
    dev_ms = dev_ms_raw - flush_ms
    launches = ctx.kernel_launches - launches0
    if args.dump_outputs:                               # outside the bracket; before the reset below discards the result
        cams_out, pts_out, focal_out = prob.download()
        if world > 1:                                   # every rank holds all cameras and its contiguous range of points
            shards = [None] * world
            dist.all_gather_object(shards, pts_out)
            pts_out = np.concatenate(shards)
        if rank == 0:
            dump_outputs(args.dump_outputs, cams_out, pts_out, focal_out)
    # Clocks and throttle reasons: NVML / nvidia-smi queries hold the driver lock for 1-40 ms on these hosts and stall the
    # kernel launches of the process they observe (measured: the 0.83 ms step became 1.2-2.2 ms, a 2-GPU step 10 ms), so the
    # sampler does not run inside the reported pass.  It runs during an IDENTICAL second pass of the same K iterations right
    # after it (same problem, same flush, at least 60 iterations), whose time is reported as clocks.sampled_pass_ms_per_step for comparison.
    prob.reset()
    with torch.cuda.stream(stream):
        flush.zero_()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    t2 = time.perf_counter()
    s2 = run_steps(prob, capi, max(args.steps, 60), profile=1, l2_flush_mb=L2_FLUSH_MB)   # long enough for several (slow) NVML queries
    barrier()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["sampled_pass_ms_per_step"] = (time.perf_counter() - t2) * 1e3 / max(1, s2["num_iterations"])
        clocks["note"] = "sampled during an identical second pass; sampling inside the reported pass stalls its kernel launches (driver lock)"
    iters = s["num_iterations"]
    assert iters == args.steps, s
    t = torch.tensor([dev_ms, wall * 1e3, dev_ms_raw], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(p["nobs"]), float(launches), float(p["np"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    dev_ms, wall_ms, dev_ms_raw = t.tolist(); nobs_total, launches_total, np_total = tot.tolist()
    value = nobs_total * iters / (dev_ms * 1e-3)

    # ---- N-rank answer == 1-rank answer (checked here because the driver's GPU test box has one GPU): 10 LM iterations of
    # the sharded problem on all ranks, the same 10 iterations of the whole problem on rank 0 alone (a second context without
    # communicator), cameras + focal + cost compared; every rank must hold bit-identical cameras.
    equivalence = None
    if world > 1:
        prob.reset()
        s_eq = prob.run(fixed_iteration_options(capi, 10))
        cams_n, _, f_n = prob.download()
        blob = torch.from_numpy(np.concatenate([cams_n.ravel(), [f_n, s_eq["final_cost"]]])).cuda()
        gathered = [torch.empty_like(blob) for _ in range(world)]
        dist.all_gather(gathered, blob)
        identical = all(bool(torch.equal(g, gathered[0])) for g in gathered)
        if rank == 0:
            ctx1 = capi.Context(local)
            p1 = ctx1.ba_problem(p_full["cams"], p_full["pts"], p_full["focal"], p_full["obs_xy"], p_full["obs_cam"], p_full["pt_off"])
            s1 = p1.run(fixed_iteration_options(capi, 10)); cams_1, _, f_1 = p1.download()
            p1.close(); ctx1.close()
            equivalence = {"iterations": 10, "final_cost_rel_diff": abs(s_eq["final_cost"] - s1["final_cost"]) / s1["final_cost"],
                           "max_camera_abs_diff": float(np.abs(cams_n - cams_1).max()), "focal_rel_diff": abs(f_n - f_1) / f_1,
                           "ranks_bit_identical": identical}
            assert equivalence["final_cost_rel_diff"] < 1e-9 and equivalence["max_camera_abs_diff"] < 1e-7 and identical, equivalence
        barrier()
    prob.close()
    # ---- weak scaling (secondary): every rank its own 200k points, same K iterations, same hygiene
    weak = None
    if world > 1:
        pw = make_shard(args.workload, rank)
        probw = ctx.ba_problem(pw["cams"], pw["pts"], pw["focal"], pw["obs_xy"], pw["obs_cam"], pw["pt_off"])
        if exchange.startswith("peer"):
            sdist.attach_peers(probw, dist)
        run_steps(probw, capi, 40, profile=1, l2_flush_mb=L2_FLUSH_MB); probw.reset()
        barrier()
        w0 = torch.cuda.Event(enable_timing=True); w1 = torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        sw = run_steps(probw, capi, args.steps, profile=1, l2_flush_mb=L2_FLUSH_MB)
        w1.record(stream)
        barrier()
        tw = torch.tensor([w0.elapsed_time(w1) - float(sw["flush_ms_total"])], dtype=torch.float64, device="cuda")
        nw = torch.tensor([float(pw["nobs"])], dtype=torch.float64, device="cuda")
        dist.all_reduce(tw, op=dist.ReduceOp.MAX); dist.all_reduce(nw, op=dist.ReduceOp.SUM)
        weak = {"value": nw.item() * sw["num_iterations"] / (tw.item() * 1e-3), "unit": UNIT, "ms_per_step": tw.item() / sw["num_iterations"],
                "points_per_gpu": pw["np"], "observations_total": int(nw.item())}
        probw.close()
    # the resident problem gave its workspace back to the context's cache: the one-shot solves below borrow it instead of
    # paying cudaMalloc / cudaFree of ~600 MB per call (which cost 1 ms on a quiet host and 100+ ms on a busy one)
    # ---- e2e: the same K iterations through the one-shot C-ABI call with pinned HOST buffers ------------------------
    def pinned(x):
        return torch.from_numpy(np.ascontiguousarray(x)).pin_memory().numpy()
    h = [pinned(p["cams"]), pinned(p["pts"]), p["focal"], pinned(p["obs_xy"]), pinned(p["obs_cam"]), pinned(p["pt_off"])]
    cams0, pts0 = np.array(h[0]), np.array(h[1])                       # pristine start; h[0], h[1] are overwritten with the result
    h2d = sum(x.nbytes for x in h if isinstance(x, np.ndarray)) + 8
    d2h = h[0].nbytes + h[1].nbytes + 8
    reps = 3
    e2e_steps = args.steps if args.steps <= SOLVE_ITERS + 4 else SOLVE_ITERS     # iterations of one solve call
    for _ in range(3):                  # untimed warm-up solves: allocator, first touch of every code path, clocks (pinning idled the GPU)
        h[0][...] = cams0; h[1][...] = pts0
        ctx.ba_solve(*h, fixed_iteration_options(capi, e2e_steps), inplace=True)
    e2e_iters = 0
    rep_ms = []
    for _ in range(reps):
        h[0][...] = cams0; h[1][...] = pts0                            # untimed: restore the inputs in the pinned buffers
        barrier()
        t1 = time.perf_counter()
        e2e_iters += ctx.ba_solve(*h, fixed_iteration_options(capi, e2e_steps), inplace=True)[3]["num_iterations"]
        rep_ms.append(round((time.perf_counter() - t1) * 1e3, 3))
    barrier()
    e2e_wall = sum(rep_ms) * 1e-3
    te = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = nobs_total * e2e_iters / te.item()

    # ---- roofline of K3 = residual+Jacobian evaluation fused with the Schur reduction (SURVEY.md 8d's unit): three kernels,
    # timed live with CUDA events on the library stream inside the timed region (summary.*_ms_total)
    peak, peak_src = load_peaks()
    nl = max(1, s["schur_launches"])
    k_point, k_pair, k_cam = s["schur_ms_total"] / nl, s["pair_ms_total"] / nl, s["camera_ms_total"] / nl
    k3_ms = k_point + k_pair + k_cam
    abytes = algorithmic_bytes(p["nc"], p["np"], p["nobs"])
    achieved = abytes / (k3_ms * 1e-3) / 1e9 if k3_ms > 0 else 0.0
    # DRAM bytes of the K3 kernels from the committed ncu --set full capture -- only if it was taken on THESE sources
    # (profiles/traffic.json carries a hash of csrc/, tools/update_traffic.py); a stale figure is reported as null
    traffic, traffic_note = None, None
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import update_traffic
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("source_id") == update_traffic.source_id():
            traffic = tj.get(args.workload)
        else:
            traffic_note = "profiles/traffic.json was captured on other sources (source_id mismatch): not reported"
    except Exception:
        pass
    kernels = {"ba_point_kernel": k_point, "ba_pair_kernel": k_pair, "ba_camera_kernel+ba_combine_kernel": k_cam}
    # fp64 side of the roofline (SURVEY.md 8d asks for it next to the HBM fraction): useful flops of one LM iteration, counted from the
    # algorithm -- three closed-form Jacobian evaluations per observation (point pass, camera pass, step evaluation; ~300 flop each),
    # the per-observation Schur terms (~760 flop) and 2*6*6*3 flop per (observation pair of a point) for the off-diagonal blocks --
    # against the fp64 peak measured on this GPU pool (profiles/fp64_peak.json, tools/fp64_peak.cu)
    kk = np.diff(p["pt_off"]).astype(np.int64)
    pair_entries = int((kk * (kk - 1) // 2).sum())
    flops_iter = float(p["nobs"]) * (3 * 300 + 760) + 216.0 * pair_entries
    try:
        fp64_peak = float(json.load(open(os.path.join(ROOT, "profiles", "fp64_peak.json")))["dmma_m8n8k4_tflops"]); fp64_src = "measured (profiles/fp64_peak.json, mma.sync m8n8k4 f64)"
    except Exception:
        fp64_peak, fp64_src = 40.0, "nominal B200 fp64"
    fp64 = {"flops_per_step": flops_iter, "pair_entries": pair_entries, "peak_tflops": fp64_peak, "peak_source": fp64_src}
    dominant = max(kernels, key=kernels.get)

    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_ms / iters, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": f"BASELINE.json configs[{2 if args.workload == 'cfg3' else 1}] ({args.workload})",
                           "cams": p_full["nc"], "points": p_full["np"], "observations": p_full["nobs"],
                           "points_per_gpu": p["np"], "observations_per_gpu": p["nobs"],
                           "points_total": int(np_total), "observations_total": int(nobs_total),
                           "step": "one LM iteration: residual+Jacobian+Schur pass, rank sum, dense Cholesky, back-substitution, candidate evaluation"
                                   + (f"; the {args.steps} timed iterations are solves of {SOLVE_ITERS} restarted from x0" if args.steps > SOLVE_ITERS + 4 else ""),
                           "parallelism": f"the problem's points sharded over {world} GPU(s) (strong scaling), cameras replicated, reduced camera system "
                                          f"summed over ranks ({exchange}); every rank factors the 601x601 reduced system redundantly",
                           "l2": f"flushed: a {L2_FLUSH_MB} MB scratch buffer is written before every timed LM iteration (per-GPU working set ~90 MB < L2); "
                                 "the flush writes run inside the event bracket and their own event time is subtracted (ms_per_step_incl_flush keeps the raw bracket)"},
                "wall_ms_per_step": wall_ms / iters, "ms_per_step_incl_flush": dev_ms_raw / iters,
                "dense_solve_ms": s["solve_ms_total"] / max(1, s["num_linear_solves"]),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "note": f"one sfmb200_ba_solve call (create+upload from pinned host, {e2e_steps} LM iterations, download) = one step; mean of {reps}", "rep_ms": rep_ms},
                "gpu_launches": int(launches_total),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                             "kernel": "K3 = ba_point_kernel + ba_pair_kernel + ba_camera_kernel + ba_combine_kernel (one residual+Jacobian+Schur pass)",
                             "kernel_ms": k3_ms, "kernels_ms": kernels, "dominant": dominant, "algorithmic_bytes": int(abytes), "peak_source": peak_src,
                             "traffic_note": traffic_note,
                             "note": "not HBM-bound: fp64 arithmetic and L1/L2 request rate of the per-camera-pair accumulation dominate (DESIGN.md section 4)"},
                "clocks": clocks}
        if weak is not None:
            line["weak"] = weak
        if equivalence is not None:
            line["equivalence"] = equivalence
        step_s = dev_ms / iters * 1e-3
        fp64["step_tflops"] = flops_iter / step_s / 1e12; fp64["step_frac"] = fp64["step_tflops"] / fp64_peak
        if k_pair > 0:
            fp64["pair_kernel_tflops"] = 216.0 * pair_entries / (k_pair * 1e-3) / 1e12; fp64["pair_kernel_frac"] = fp64["pair_kernel_tflops"] / fp64_peak
        line["fp64"] = fp64
    # ---- CPU baseline on the host cores (rank 0, 1 GPU only) ---------------------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        it = 2 if args.workload == "cfg3" else 20
        t0 = time.perf_counter()
        so = oracle.ba_solve(*a, fixed_iteration_options(oracle, it, jacobian_mode=0, num_threads=1))[3]
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": p["nobs"] * so["num_iterations"] / dt, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": f"{args.workload} full problem, {it} LM iterations of the oracle (Ceres-equivalent LM+DENSE_SCHUR, dual-number Jacobians, 1 thread as the reference leaves Ceres), {dt:.1f} s"}
    # ---- BASELINE configs[0] (crazyhorse, the only real-data configuration): stage times of the runSfM replay, GPU stages
    # through the drop-in call shape beside the reference's own OpenCV calls / the oracle's Ceres restatement on the host cores
    if rank == 0 and world == 1 and not args.no_stages:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools")); sys.path.insert(0, os.path.join(ROOT, "tests"))
            import bench_cfg1
            c1 = bench_cfg1.measure(reps=2)
            keep = ("wall_s", "hot_path_s", "seconds", "calls", "cloud")
            line["cfg1"] = {"workload": c1["workload"], "gpu": {k: c1["gpu_batched"][k] for k in keep},
                            "gpu_per_call_match_s": c1["gpu_per_call"]["seconds"]["match"],
                            "gpu_per_call_match_nocache_s": c1["gpu_per_call_nocache"]["seconds"]["match"],
                            "cpu_all_threads": {k: c1["cpu_cv2_all_threads"][k] for k in keep}, "cpu_threads": c1["cpu_threads"],
                            "speedup_hot_path": c1["speedup_hot_path"], "speedup_per_stage": c1["speedup_per_stage"],
                            "note": "seconds per stage summed over the replay's calls; RANSAC stages are cv2 in both arms (SURVEY.md 8 f-2)"}
        except Exception as e:                                  # never lose the headline line to a secondary measurement
            line["cfg1"] = {"error": repr(e)}
        # BASELINE configs[3] (all-pairs matching, 50 x 5000: reference-faithful ORB/Hamming and the SIFT-128/L2 wording) and
        # configs[4] (1 M point triangulation): device-timed value, host-buffer e2e incl. descriptor upload, roofline, cv2 CPU baseline
        try:
            import bench_stages
            for st in bench_stages.measure_all(reps=3, ctx=ctx):
                key = {"match_hamming": "cfg4_hamming", "match_l2": "cfg4_sift_l2", "triangulate": "cfg5"}[st["stage"]]
                line[key] = st
        except Exception as e:
            line["cfg4_cfg5"] = {"error": repr(e)}
        # SURVEY.md 8 row f-3, the step before matching: ORB(5000) extraction of the 7 images of cfg 1 (1024 x 768, B,G,R) from HOST buffers,
        # beside cv2's detectAndCompute on the host cores
        try:
            import bench_orb
            line["f3_orb"] = bench_orb.run(n_images=7, reps=3, cpu=not args.no_cpu_baseline, ctx=ctx)
        except Exception as e:
            line["f3_orb"] = {"error": repr(e)}
    # ---- BASELINE configs[1] (cfg 2: 20 cameras / 10 k points / 80 k observations), N = 1: the same step, resident and one-shot
    if rank == 0 and world == 1 and not args.no_stages and args.workload != "cfg2":
        try:
            from sfm_toy_library_b200 import synth
            p2 = synth.make_ba_problem(seed=0, **synth.BA_CONFIGS["cfg2"])
            a2 = (p2["cams"], p2["pts"], p2["focal"], p2["obs_xy"], p2["obs_cam"], p2["pt_off"])
            pr2 = ctx.ba_problem(*a2)
            run_steps(pr2, capi, 40); pr2.reset()
            g0 = torch.cuda.Event(enable_timing=True); g1 = torch.cuda.Event(enable_timing=True)
            ctx.synchronize(); g0.record(stream); s2 = run_steps(pr2, capi, 20); g1.record(stream); ctx.synchronize(); torch.cuda.synchronize()
            ms2 = g0.elapsed_time(g1) / s2["num_iterations"]
            pr2.close()
            ctx.ba_solve(*a2, fixed_iteration_options(capi, 20))
            t1 = time.perf_counter(); ctx.ba_solve(*a2, fixed_iteration_options(capi, 20)); e2 = time.perf_counter() - t1
            line["cfg2"] = {"workload": "BASELINE.json configs[1]: 20 cams / 10000 points / 80000 observations", "ms_per_step": ms2,
                            "value": p2["nobs"] / (ms2 * 1e-3), "unit": UNIT, "e2e": {"value": p2["nobs"] * 20 / e2, "unit": UNIT, "seconds_per_20_iteration_solve": e2},
                            "note": "no L2 flush between iterations (working set 5 MB); launch-latency regime"}
        except Exception as e:
            line["cfg2"] = {"error": repr(e)}
    # ---- all-pairs matching sharded over the ranks (SURVEY.md 8e: image pairs are independent, no collective): every rank holds all
    # descriptors and matches its round-robin share of the 1225 pairs of cfg 4 (H); device time, max over ranks
    if world > 1 and not args.no_stages:
        try:
            from sfm_toy_library_b200 import synth
            descs = synth.make_descriptor_set(50, n=5000)
            allp = [(i, j) for i in range(50) for j in range(i + 1, 50)]
            mine = sdist.shard_pairs(allp, rank, world)
            dsm = ctx.descriptor_set(descs)
            rows = 5000 * len(mine)
            dq = torch.empty(rows, dtype=torch.int32, device="cuda"); dt_ = torch.empty(rows, dtype=torch.int32, device="cuda")
            dd = torch.empty(rows, dtype=torch.float32, device="cuda"); dst = torch.empty(len(mine) + 1, dtype=torch.int32, device="cuda")
            dtot = torch.empty(1, dtype=torch.int64, device="cuda")
            for _ in range(2):
                dsm.match_pairs_device(mine, dq.data_ptr(), dt_.data_ptr(), dd.data_ptr(), dst.data_ptr(), dtot.data_ptr())
            barrier()
            m0 = torch.cuda.Event(enable_timing=True); m1 = torch.cuda.Event(enable_timing=True)
            m0.record(stream)
            for _ in range(3):
                dsm.match_pairs_device(mine, dq.data_ptr(), dt_.data_ptr(), dd.data_ptr(), dst.data_ptr(), dtot.data_ptr())
            m1.record(stream)
            barrier()
            tm = torch.tensor([m0.elapsed_time(m1) / 3.0], dtype=torch.float64, device="cuda")
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dsm.close()
            if rank == 0:
                line["cfg4_hamming_sharded"] = {"pairs": len(allp), "ranks": world, "ms_per_step": tm.item(), "value": len(allp) / (tm.item() * 1e-3), "unit": "pairs/s",
                                                "note": "pairs dealt round-robin to the ranks, descriptors replicated, no collective; max over ranks of the device time"}
        except Exception as e:
            if rank == 0:
                line["cfg4_hamming_sharded"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg2"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stages", action="store_true", help="skip the secondary stage measurements (cfg1 replay)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the cameras, points and focal length of the last timed iteration as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
