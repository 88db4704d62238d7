#!/usr/bin/env python
"""Headline benchmark: leg-frames/s of the 4-stage sequential leg IK (+FK) on synthetic pose data.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--trials T] [--frames F] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (stages 1-4 + 9-row FK) over T trials x 6 legs x F frames per GPU
(default T = 1000, F = 1000: BASELINE.json config "synthetic 1k trials x 1000 frames x 6 legs on 1 B200").
Under torchrun every rank owns its own T trials (weak scaling; no collective on the data path).

Prints ONE JSON line (rank 0).  `value` times the kernel with the pose already resident in HBM; `e2e` times
the public batched call with HOST pinned buffers (H2D of the pose, solve, D2H of angles + FK in the timed
region).  `roofline` describes the solver kernel; `cpu_baseline` is the CPU oracle (the reference's
algorithm: restated ikpy glue + scipy TRF) timed on this box's host cores on a bounded sample.
The same line carries
  config4      BASELINE.json config 4: the FIXED 10 000-trial x 1000-frame x 6-leg workload, trials sharded over the
               N ranks (10000 / N per rank; all 60 000 chains on one GPU at N = 1) -- kernel and end-to-end figures, so
               that dividing config4 at N = 8 by config4 at N = 1 is the strong-scaling factor of north_star;
  secondary    driver-timed records of config 5 (fused long sequence), the HBM-bound stream kernels, config 1 (bundled
               locomotion recording) and config 2 (bundled grooming trial) through the dict API with their parity figures
               against the oracle / the reference's shipped angles (rank 0).

--impl reference times that CPU implementation alone, with every host core, on bounded samples of the same
workload (see DESIGN.md: the reference's own per-frame chain rebuild needs ikpy/sympy, which is not
installable offline; the oracle is its arithmetic without that overhead, i.e. a faster stand-in).

--dump-outputs DIR writes what the last timed step returned (rank 0: the angles and FK of `value`'s solve_device call)
as DIR/angles.npy (chains, frames, 7) and DIR/fk.npy (chains, frames, 9, 3), float32.  The synthetic pose is seeded, so
the same arguments give the same inputs and two builds can be compared output for output.  Outputs above DUMP_BYTES are
sampled with a fixed seed: whole chains while one fits, else a subset of frames as well (sorted indices).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
os.environ.setdefault("OMP_NUM_THREADS", "1")

import numpy as np  # noqa: E402

METRIC = "leg-frames/sec, 4-stage seq IK"
UNIT = "leg-frames/s"
ALG_BYTES_PER_LEG_FRAME = 60 + 28 + 108          # pose in + angles out + FK out, fp32 (SURVEY.md 8d / DESIGN.md)
ALG_FLOP_PER_LEG_FRAME = 14.5e3                   # nominal full-chain model of SURVEY.md 8d (DESIGN.md)
DUMP_BYTES = 60_000_000                           # --dump-outputs: array bytes in all (64 MB less room for the .npy headers)


# --------------------------------------------------------------------------------------------- CPU oracle legs
def _oracle_job(job):
    """One (trial, leg) chain through the CPU oracle over frames [f0, f0 + n); returns leg-frames solved.  f0 > 0: the
    warm start of frame f0 is the synthetic ground truth of frame f0 - 1 (steady-state frames: no cold first solve)."""
    from oracle import seqik_oracle as O
    from seqikpy_b200 import synthetic as S
    from seqikpy_b200.kinematic_chain import DOF_ORDER, STAGE_ACTIVE_DOFS, STAGE_ACTIVE_SLOTS
    trial, li, f0, n_frame = job
    size, bounds, init = S.chain_constants()
    leg = S.LEGS[li]
    pose, truth = S.make_trial(trial, 1000, return_truth=True)
    seeds = {k: np.array(v, dtype=float) for k, v in init[leg].items()}
    if f0 > 0:
        for stage in (1, 2, 3, 4):
            for slot, dof in zip(STAGE_ACTIVE_SLOTS[stage], STAGE_ACTIVE_DOFS[stage]):
                seeds[f"stage_{stage}"][slot] = truth[f0 - 1, li, DOF_ORDER.index(dof)]
    O.run_ik_and_fk({f"{leg}_leg": pose[f0:f0 + n_frame, li]}, size, bounds, {leg: seeds})
    return n_frame


def oracle_throughput(n_trial, n_frame, procs, repeats=1):
    """leg-frames/s of the CPU oracle over n_trial x 6 chains with `procs` worker processes
    (process-level parallelism over legs like examples/example_leg_inv_kinematics_parallel.py:186-189)."""
    from multiprocessing import get_context
    jobs = [(tr, li, 0, n_frame) for tr in range(n_trial) for li in range(6)]
    ctx = get_context("fork")
    with ctx.Pool(procs) as pool:
        pool.map(_oracle_job, [(0, 0, 0, 2)] * procs)       # import + first-call costs out of the timed region
        times = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            done = sum(pool.map(_oracle_job, jobs, chunksize=1))
            times.append(time.perf_counter() - t0)
    return done, times


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    procs = max(1, min(cores, 64))
    n_trial = max(1, (procs + 5) // 6)                      # enough chains to occupy every worker
    n_frame = args.ref_frames
    per_step = n_trial * 6 * n_frame
    from multiprocessing import get_context
    f0 = 100                                                # steady-state frames: warm-started, no cold first solve
    jobs = [(tr, li, f0, n_frame) for tr in range(n_trial) for li in range(6)]
    with get_context("fork").Pool(procs) as pool:
        pool.map(_oracle_job, [(0, 0, 0, 2)] * procs)
        for _ in range(args.warmup):
            pool.map(_oracle_job, jobs, chunksize=1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_oracle_job, jobs, chunksize=1)
        dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = (f"{n_trial} trial(s) x 6 legs x frames {f0}..{f0 + n_frame} (steady state, warm-started) per step, "
              f"{procs} worker processes (one chain each)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, note="CPU oracle on a bounded sample of this workload"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- helpers
def workload_config(args, note=None):
    cfg = {
        "workload": f"synthetic {args.trials} trials x {args.frames} frames x 6 legs per GPU, 4-stage seq IK + FK "
                    f"(BASELINE config 'synthetic 1k trials x 1000 frames x 6 legs on 1 B200' at the defaults)",
        "trials_per_gpu": args.trials, "frames": args.frames, "legs": 6,
        "chains_per_gpu": args.trials * 6, "parallelism": f"trial shards x{args.gpus}, no collective",
        "l2": "inputs+outputs per step (1.18 GB at the defaults) exceed the 126 MB L2; no explicit flush",
    }
    if note:
        cfg["note"] = note
    return cfg


def sample_outputs(angles, fk):
    """Device copies of a fixed, seeded sample of (angles, fk) of at most DUMP_BYTES, enqueued behind the step that wrote
    them, so that later calls into the same session buffers do not change what is dumped."""
    import torch
    n_chain, n_frame = angles.shape[:2]
    lf_budget = DUMP_BYTES // (angles[0, 0].nbytes + fk[0, 0].nbytes)
    n_c = max(1, min(n_chain, lf_budget // n_frame))
    n_f = min(n_frame, lf_budget // n_c)
    rng = np.random.default_rng(0)
    chains = torch.from_numpy(np.sort(rng.choice(n_chain, n_c, replace=False))).to(angles.device)
    frames = torch.from_numpy(np.sort(rng.choice(n_frame, n_f, replace=False))).to(angles.device)
    return {name: t.index_select(0, chains).index_select(1, frames) for name, t in (("angles", angles), ("fk", fk))}


def write_outputs(out_dir, outputs):
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, t in outputs.items():
        np.save(out / f"{name}.npy", t.cpu().numpy())
    print(f"bench.py: wrote {', '.join(f'{n}.npy {tuple(t.shape)}' for n, t in outputs.items())} to {out}", file=sys.stderr)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML every ~10 ms; falls back to
    polling nvidia-smi when the NVML binding is unavailable)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self._stop_evt = index, threading.Event()
        self.sm, self.max_sm, self.reasons, self.how = [], None, set(), "nvml"

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.max_sm = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        names = {"hw_slowdown": "nvmlClocksThrottleReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksThrottleReasonHwThermalSlowdown",
                 "sw_thermal_slowdown": "nvmlClocksThrottleReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksThrottleReasonSwPowerCap"}
        bits = {k: getattr(nv, v) for k, v in names.items() if hasattr(nv, v)}
        while not self._stop_evt.is_set():
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.reasons.update(k for k, b in bits.items() if mask & b)
            self._stop_evt.wait(0.01)

    def _run_smi(self):
        self.how = "nvidia-smi"
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                r = [c.strip() for c in out.split(",")]
                self.sm.append(float(r[0])); self.max_sm = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.05)

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "how": self.how}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        ids = [v for v in vis.split(",") if v.strip()]
        if local_rank < len(ids) and ids[local_rank].strip().isdigit():
            return int(ids[local_rank])
    return local_rank


# --------------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from seqikpy_b200 import _native, synthetic as S
    from seqikpy_b200.batch import BatchedLegIK
    from seqikpy_b200.kinematic_chain import KinematicChainSeq

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # Only the JSON line may reach stdout (NCCL and friends print banners there): park fd 1 on stderr until the end.
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    # CPU baseline first (rank 0, fresh interpreter, before this process touches CUDA or NCCL)
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        procs = max(1, min(6, host_cores()))
        n_fr = args.cpu_frames
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")
               and not k.startswith("TORCHELASTIC")}
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--cpu-baseline-only", "--cpu-frames", str(n_fr),
                              "--cpu-procs", str(procs)], capture_output=True, text=True, env=env)
        try:
            res = json.loads(out.stdout.strip().splitlines()[-1])
            cpu = {"value": res["leg_frames"] / res["seconds"], "unit": UNIT, "cores": procs, "kind": "port",
                   "one_core_value": res["one_core_leg_frames"] / res["one_core_seconds"],
                   "sample": f"trial 0 x 6 legs x first {n_fr} frames of this workload, CPU oracle (restated ikpy glue + scipy TRF), "
                             f"{procs} processes over legs like the reference's Pool(6) example"}
        except Exception as exc:                      # keep the GPU measurement even if the CPU leg fails
            print(f"bench.py: cpu baseline failed: {exc!r}\n{out.stderr[-2000:]}", file=sys.stderr)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: a CUDA device is required (there is no CPU fallback for the product path)")
    _native.load_library()
    from seqikpy_b200.batch import bind_to_gpu_numa
    numa_cpus = bind_to_gpu_numa(physical_gpu_index(local_rank)) if not args.no_numa_bind else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)

    T, F = args.trials, args.frames
    size, bounds, init = S.chain_constants()
    chain = KinematicChainSeq(bounds, list(S.LEGS), size)
    sess = BatchedLegIK(chain, init, S.LEGS, T, F, device=dev, schedule=args.schedule, chains_per_warp=args.cpw)

    # synthetic pose of this rank's trials, chain-major, in pinned host memory
    t_gen = time.perf_counter()
    host_pose = torch.empty((T, 6, F, 5, 3), dtype=torch.float32, pin_memory=True)
    hp = host_pose.numpy()
    for i in range(T):
        hp[i] = S.make_trial(rank * T + i, F).astype(np.float32).transpose(1, 0, 2, 3)
    t_gen = time.perf_counter() - t_gen
    sess.d_pose.copy_(host_pose.reshape(sess.n_chain, F, 5, 3))
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps bracketed by barrier + synchronize; CUDA events on the launching stream; max over ranks (ms)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    # ---- kernel-only (inputs resident in HBM)
    for _ in range(max(args.warmup, 3)):
        sess.solve_device()
    sampler = ClockSampler(physical_gpu_index(local_rank)) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_total = timed(lambda: sess.solve_device(want_stats=False), args.steps)
    ms_step = ms_total / args.steps
    dumped = sample_outputs(sess.d_angles, sess.d_fk) if args.dump_outputs and rank == 0 else None
    # ---- end to end through the public batched call with host buffers
    for _ in range(2):
        sess.solve_host(host_pose, n_chunks=args.chunks)
    ms_e2e = timed(lambda: sess.solve_host(host_pose, synchronize=False, n_chunks=args.chunks), args.steps) / args.steps
    e2e_launches = sess.launches_per_call + 1                     # one solve per frame chunk + the first-frame kernel of chunk 0
    clocks = sampler.stop() if sampler else None
    # ---- the same call with the joints-only FK layout (rows 5..8: the rows that carry information); a secondary figure,
    #      the headline `e2e` above keeps the reference's 9-row layout
    ms_e2e_joints = ms_e2e_wire = expand_threads = None
    if not args.no_joints_e2e:
        sess_j = BatchedLegIK(chain, init, S.LEGS, T, F, device=dev, schedule=args.schedule, chains_per_warp=args.cpw, fk_layout="joints")
        for _ in range(2):
            sess_j.solve_host(host_pose, n_chunks=args.chunks)
        ms_e2e_joints = timed(lambda: sess_j.solve_host(host_pose, synchronize=False, n_chunks=args.chunks), args.steps) / args.steps
        del sess_j
        # ... and as a WIRE format only: joints-only over the host link, the reference's 9-row layout rebuilt in host memory
        sess_w = BatchedLegIK(chain, init, S.LEGS, T, F, device=dev, schedule=args.schedule, chains_per_warp=args.cpw, wire="joints")
        for _ in range(2):
            sess_w.solve_host(host_pose, n_chunks=args.chunks)
        ms_e2e_wire = timed(lambda: sess_w.solve_host(host_pose, synchronize=False, n_chunks=args.chunks), args.steps) / args.steps
        expand_threads = sess_w.expand_threads
        del sess_w

    # ---- the same kernel family walking the reference's own iterates (SEQIK_FLAG_REFERENCE_ITERATES: no Newton steps, no
    #      closed-form warm step; runs on the stage-pipeline schedule): a secondary figure that shows what the default flags save
    ms_ref_it, nfev_ref_it = None, torch.zeros(4, dtype=torch.float64, device=dev)
    if not args.no_ref_iterates:
        sess.flags = _native.FLAG_REFERENCE_ITERATES
        for _ in range(3):
            sess.solve_device()
        ms_ref_it = timed(lambda: sess.solve_device(want_stats=False), max(3, args.steps // 2)) / max(3, args.steps // 2)
        sess.solve_device()
        torch.cuda.synchronize()
        nfev_ref_it = sess.nfev.to(torch.float64).sum(0)
        sess.flags = _native.FLAG_DEFAULT

    sess.solve_device()
    torch.cuda.synchronize()
    nfev = sess.nfev.to(torch.float64).sum(0)                     # evaluations per stage, this rank
    fk_err = torch.tensor([sess.mean_fk_error()], dtype=torch.float64, device=dev)
    maxfev = (sess.status == 0).sum().to(torch.float64).reshape(1)
    if world > 1:
        dist.all_reduce(nfev); dist.all_reduce(fk_err); dist.all_reduce(maxfev); dist.all_reduce(nfev_ref_it)
    leg_frames_rank = sess.leg_frames
    leg_frames = leg_frames_rank * world
    nfev_per_lf = (nfev / leg_frames).tolist()

    # ---- BASELINE config 4: the FIXED 10 000-trial workload, trials sharded over the ranks (strong scaling).  The device
    #      pose is tiled from this rank's unique trials (the kernel's cost does not depend on the values repeating); the
    #      end-to-end leg moves every byte of the shard through the 1000-trial session's pinned buffers, sub-batch by sub-batch
    config4 = None
    if not args.no_config4:
        from seqikpy_b200.batch import shard_range
        T4_total = args.config4_trials
        lo4, hi4 = shard_range(T4_total, rank, world)
        T4 = hi4 - lo4
        sess4 = BatchedLegIK(chain, init, S.LEGS, T4, F, device=dev, schedule=args.schedule, chains_per_warp=args.cpw, host_buffers=False)
        reps4 = (T4 + T - 1) // T
        sess4.d_pose.copy_(sess.d_pose.view(T, 6, F, 5, 3).repeat(reps4, 1, 1, 1, 1)[:T4].reshape(sess4.n_chain, F, 5, 3))
        for _ in range(3):
            sess4.solve_device(want_stats=False)
        steps4 = max(3, args.steps // 2)
        ms4 = timed(lambda: sess4.solve_device(want_stats=False), steps4) / steps4
        sess4.solve_device()
        torch.cuda.synchronize()
        ok4 = (sess4.status == 1).sum().to(torch.float64).reshape(1)
        err4 = torch.tensor([sess4.mean_fk_error() * T4], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ok4); dist.all_reduce(err4)
        del sess4
        torch.cuda.empty_cache()
        # end to end: full sub-batches through `sess`, the remainder through a smaller session
        n_full, rem = divmod(T4, T)
        sess_rem = host_rem = None
        if rem:
            sess_rem = BatchedLegIK(chain, init, S.LEGS, rem, F, device=dev, schedule=args.schedule, chains_per_warp=args.cpw)
            host_rem = host_pose[:rem].contiguous().pin_memory()

        def e2e4():
            for _ in range(n_full):
                sess.solve_host(host_pose, synchronize=False, n_chunks=args.chunks)
            if sess_rem is not None:
                sess_rem.solve_host(host_rem, synchronize=False, n_chunks=args.chunks)
        e2e4(); torch.cuda.synchronize()
        steps4e = max(2, args.steps // 4)
        ms4_e2e = timed(e2e4, steps4e) / steps4e
        lf4 = T4_total * 6 * F
        config4 = {
            "workload": f"synthetic {T4_total} trials x {F} frames x 6 legs IN TOTAL (BASELINE.json config 4), trials sharded over "
                        f"{world} GPU(s) in contiguous shards, no collective; strong scaling: divide by the same object at N = 1",
            "trials_total": T4_total, "trials_this_rank": T4, "chains_this_rank": T4 * 6, "scaling": "strong",
            "value": lf4 / (ms4 * 1e-3), "unit": UNIT, "ms_per_step": ms4, "steps": steps4, "timing": "CUDA events, max over ranks, pose resident in HBM",
            "e2e": {"value": lf4 / (ms4_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms4_e2e, "steps": steps4e,
                    "h2d_bytes_per_step": T4 * 6 * F * 60, "d2h_bytes_per_step": T4 * 6 * F * 136, "bytes_are": "per GPU",
                    "how": f"{n_full} sub-batch(es) of {T} trials" + (f" + one of {rem}" if rem else "") + " through BatchedLegIK.solve_host "
                           "(pinned host pose in, pinned host angles + 9-row FK out; the sub-batches reuse the same pinned buffers)"},
            "chains_converged": int(ok4.item()), "chains": T4_total * 6, "mean_fk_error_mm": float(err4.item()) / T4_total,
            "data": f"device-tiled from each rank's {T} unique synthetic trials",
        }
        del sess_rem, host_rem

    # ---- secondary, driver-timed records (rank 0; the other ranks wait at the barrier below)
    secondary = {}
    if rank == 0 and not args.no_secondary:
        sys.path.insert(0, str(ROOT / "scripts"))
        import bench_secondary as B2
        peaks_ = {}
        try:
            peaks_ = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        for name, fn in (("config1_dict_api", B2.config1_dict_api), ("config2_dict_api", B2.config2_dict_api), ("stream_kernels", lambda: B2.stream_kernels(float(peaks_.get("hbm_gbs", 6650.0)))),
                         ("config5_fused", lambda: B2.config5_fused(args.config5_trials, args.config5_frames))):
            try:
                t_s = time.perf_counter()
                secondary[name] = fn()
                secondary[name]["record_wall_s"] = time.perf_counter() - t_s
            except Exception as exc:                                  # never lose the headline to a secondary record
                secondary[name] = {"error": repr(exc)[:300]}
            torch.cuda.empty_cache()

    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        sm_max = float(peaks.get("sm_max_mhz", 1965.0))
        fp32_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12           # TFLOP/s at max clock
        ach_gbs = leg_frames_rank * ALG_BYTES_PER_LEG_FRAME / (ms_step * 1e-3) / 1e9
        ach_tf = leg_frames_rank * ALG_FLOP_PER_LEG_FRAME / (ms_step * 1e-3) / 1e12
        # static ncu counters of the committed capture (profiles/solver_traffic.json): quoted only for the configuration they
        # were captured on and only while this run's kernel time agrees with the capture's within 5 %
        traffic = ncu_flop = ncu_issue = None
        capture = None
        try:
            prof = json.loads((ROOT / "profiles" / "solver_traffic.json").read_text())
            cap_ms = 1e3 * float(prof.get("step_duration_s_under_ncu", prof["duration_s_under_ncu"]))   # block kernel + first-frame kernel
            agrees = abs(ms_step - cap_ms) <= 0.05 * cap_ms
            capture = {"file": "profiles/solver_traffic.json", "source": prof.get("source"), "commit": prof.get("commit"),
                       "kernel": prof.get("kernel"), "duration_ms": cap_ms, "this_run_ms": ms_step, "agrees_within_5pct": bool(agrees),
                       "what": "STATIC counters of one committed ncu --set full capture (default configuration), not measured in this run"}
            if agrees and args.trials == 1000 and args.frames == 1000:
                traffic = prof.get("dram_bytes_per_launch")
                ncu_flop = prof.get("fp32_flop_per_launch", 0) / 6e6  # measured FP32 FLOP per leg-frame (ffma x2 + fmul + fadd)
                ncu_issue = prof.get("issue_active_per_smsp")
        except Exception:
            pass
        c2 = secondary.get("config2_dict_api", {})
        line = {
            "metric": METRIC, "value": leg_frames / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args),
            "e2e": {"value": leg_frames / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": leg_frames_rank * 60, "d2h_bytes_per_step": leg_frames_rank * (28 + 108),
                    "bytes_are": "per GPU", "frame_chunks": args.chunks, "gpu_launches": args.steps * e2e_launches},
            "e2e_joints_only": None if ms_e2e_joints is None else {
                "value": leg_frames / (ms_e2e_joints * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e_joints,
                "h2d_bytes_per_step": leg_frames_rank * 60, "d2h_bytes_per_step": leg_frames_rank * (28 + 48),
                "note": "fk_layout='joints': FK rows 5..8 only (rows 0-3 of the reference layout repeat the input origin, row 4 repeats row 5)"},
            "e2e_joints_wire": None if ms_e2e_wire is None else {
                "value": leg_frames / (ms_e2e_wire * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e_wire,
                "h2d_bytes_per_step": leg_frames_rank * 60, "d2h_bytes_per_step": leg_frames_rank * (28 + 48 + 12), "host_threads": expand_threads,
                "note": "BatchedLegIK(wire='joints'): the caller still receives the reference's (..., 9, 3) FK; only rows 5..8 and a compact "
                        "copy of the origin row (seqik_origin_rows_f32) cross the host link, rows 0-4 are rebuilt in host memory by host "
                        "threads with streaming stores (seqik_fk_expand_host_f32), chunk by chunk behind the copies; bit-identical to `e2e`"},
            "gpu_launches": args.steps * 2,                           # per step: leg_first_frame_kernel + leg_solve_block_kernel
            "kernels": "leg_first_frame_kernel (frame 0 of every chain, lane per chain) + leg_solve_block_kernel (schedule 3: a warp per "
                       "chain, 32 frames per pass, bulk-copy staged)",
            "config4": config4,
            "parity_extras": {k: c2[k] for k in c2 if k.startswith(("rf_", "lf_", "head_"))} or None,
            "secondary": secondary or None,
            "solver_flags": {"value": "SEQIK_FLAG_DEFAULT (0xFF): Gauss-Newton mode, escape, skip-confirm, Newton steps, closed-form warm step",
                             "reference_iterates": None if ms_ref_it is None else {
                                 "flags": "SEQIK_FLAG_REFERENCE_ITERATES (0x3F), stage-pipeline schedule", "ms_per_step": ms_ref_it,
                                 "value": leg_frames / (ms_ref_it * 1e-3), "unit": UNIT,
                                 "nfev_per_leg_frame_by_stage": (nfev_ref_it / leg_frames).tolist()}},
            "roofline": {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
                         "traffic": traffic, "kernel": "leg_solve_block_kernel (+ leg_first_frame_kernel, ~5 % of the step)",
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst)" if peaks else "fallback",
                         "algorithmic_bytes_per_leg_frame": ALG_BYTES_PER_LEG_FRAME, "ncu_capture": capture,
                         "note": "achieved = 196 B x leg-frames per step / the step's CUDA-event time (both kernels of the step); the rest "
                                 "of the gap to the copy peak is instruction issue: ~40 warp-instructions per leg-frame at ~0.7 issue slots "
                                 "per cycle per scheduler (DESIGN.md 5.1)",
                         "fp32": {"achieved": ach_tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach_tf / fp32_peak,
                                  "flop_model": "nominal 14.5 kFLOP per leg-frame = the REFERENCE's work (SURVEY.md 8d: full-chain, "
                                                "finite-difference evaluations x its iteration counts).  The kernel does not do "
                                                "that work (two-variable closed forms, one evaluation per solve), so `achieved`/"
                                                "`frac` here say how fast the reference's work is retired and can exceed 1; how busy "
                                                "the FP32 pipe is: ncu_frac",
                                  "ncu_flop_per_leg_frame": ncu_flop,
                                  "ncu_achieved": None if not ncu_flop else leg_frames_rank * ncu_flop / (ms_step * 1e-3) / 1e12,
                                  "ncu_frac": None if not ncu_flop else leg_frames_rank * ncu_flop / (ms_step * 1e-3) / 1e12 / fp32_peak,
                                  "ncu_issue_slots_per_cycle_per_smsp": ncu_issue,
                                  "peak_is": "148 SMs x 128 FMA lanes x 2 x sm_max_mhz",
                                  "nfev_per_leg_frame_by_stage": nfev_per_lf}},
            "cpu_baseline": cpu,
            "mean_fk_error_mm": float(fk_err.item()) / world, "chains_at_max_nfev": int(maxfev.item()),
            "clocks": clocks, "data_gen_s": t_gen, "schedule": args.schedule, "numa_cpus_rank0": None if numa_cpus is None else len(numa_cpus),
        }
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--trials", type=int, default=1000, help="trials per GPU")
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--schedule", type=int, default=0, help="kernel schedule (0 auto, 1 lane per chain, 2 stage pipeline)")
    ap.add_argument("--chunks", type=int, default=8, help="frame chunks of the host pipeline (e2e)")
    ap.add_argument("--cpw", type=int, default=0, help="chains per warp of schedule 2 (0 auto)")
    ap.add_argument("--cpu-frames", type=int, default=200, help="frames per leg of the cpu_baseline sample")
    ap.add_argument("--ref-frames", type=int, default=100, help="frames per chain and step of --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin each rank to its GPU's local CPUs")
    ap.add_argument("--no-joints-e2e", action="store_true", help="skip the secondary end-to-end figure with the joints-only FK layout")
    ap.add_argument("--no-ref-iterates", action="store_true", help="skip the secondary figure with SEQIK_FLAG_REFERENCE_ITERATES (stage-pipeline kernel)")
    ap.add_argument("--no-config4", action="store_true", help="skip the config-4 (fixed 10 000-trial, sharded) record")
    ap.add_argument("--config4-trials", type=int, default=10000, help="total trials of the config-4 record")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary records (config 2 dict API, stream kernels, config 5)")
    ap.add_argument("--config5-trials", type=int, default=100)
    ap.add_argument("--config5-frames", type=int, default=100000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the angles and FK of the last timed step as DIR/*.npy (seeded sample above 64 MB)")
    ap.add_argument("--cpu-baseline-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--cpu-procs", type=int, default=6, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm returns no arrays)")
    if args.cpu_baseline_only:
        done, times = oracle_throughput(1, args.cpu_frames, args.cpu_procs)
        t0 = time.perf_counter()
        one = _oracle_job((0, 0, 0, min(args.cpu_frames, 100)))       # one chain, one process: the per-core rate
        t_one = time.perf_counter() - t0
        print(json.dumps({"leg_frames": done, "seconds": times[0], "one_core_leg_frames": one, "one_core_seconds": t_one}))
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
