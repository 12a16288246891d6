#!/usr/bin/env python
"""bench.py — simulation steps/s of the rigid-body step (collide -> cache -> setup -> N sweeps -> cache -> advance).

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU implementation on the host cores
  --dump-outputs DIR                                       also write what the last timed step computed, as DIR/<name>.npy

Workload (BASELINE.json configs[1]): 65,536 random boxes dropped onto a ground plane, 8 solver iterations, measured on the
settled pile.  One "step" = one sub-step of example/main.cpp:274-328.  Prints ONE JSON line (see README / DESIGN.md §5)."""
import argparse, json, os, subprocess, sys, threading, time
os.environ.setdefault("NCCL_DEBUG", "WARN")

# stdout must carry exactly ONE JSON line, but libraries write there too (NCCL prints its version banner through C stdio).
# File descriptor 1 is pointed at stderr for the whole run and the result line goes to the saved descriptor.
_REAL_STDOUT = None


def _own_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from nudge_b200 import scenes  # noqa: E402

# BASELINE.json configs[0..4] as --config c1..c5.  c2 is the configuration the metric is quoted on (the default; N > 1 scales it weakly:
# one scene of N x 65,536 boxes).  c3/c4/c5 are fixed-size scenes: on N > 1 GPUs they are sharded (strong scaling).
CONFIGS = {
    "c1": dict(workload="reference example scene: 1024 boxes + 1024 spheres falling onto ground, 8 solver iters (BASELINE.json configs[0]), settled",
               scene=lambda a, w: scenes.demo_scene(1024, 1024, iterations=a.iterations or 8), small=lambda a, seed: scenes.demo_scene(1024, 1024, iterations=a.iterations or 8, seed=seed),
               presim=1700, scaling="weak"),   # the bodies fall from up to 300 units: ~940 steps until the last one lands
    "c2": dict(workload="64k boxes random drop onto ground plane, 8 solver iters (BASELINE.json configs[1]), settled pile",
               scene=lambda a, w: scenes.box_drop(a.boxes * w, iterations=a.iterations or 8, seed=2), small=lambda a, seed: scenes.box_drop(8191, iterations=a.iterations or 8, seed=seed),
               presim=900, scaling="weak"),
    "c3": dict(workload="256k mixed box/sphere stack (50/50), 16 solver iters (BASELINE.json configs[2]), settled",
               scene=lambda a, w: scenes.mixed_stack(262144, iterations=a.iterations or 16), small=lambda a, seed: scenes.mixed_stack(8190, iterations=a.iterations or 16, seed=seed),
               presim=500, scaling="strong"),
    "c4": dict(workload="1M boxes random drop, 8 solver iters (BASELINE.json configs[3]), settled pile",
               scene=lambda a, w: scenes.box_drop(1 << 20, iterations=a.iterations or 8, seed=2), small=lambda a, seed: scenes.box_drop(8191, iterations=a.iterations or 8, seed=seed),
               presim=900, scaling="strong"),
    "c5": dict(workload="256k-box brick wall (running bond, deep stacking), 20 solver iters (BASELINE.json configs[4])",
               scene=lambda a, w: scenes.brick_wall(262144, iterations=a.iterations or 20), small=lambda a, seed: scenes.brick_wall(8191, iterations=a.iterations or 20),
               presim=300, scaling="strong"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md recipe).  NVML in-process (a query takes
    microseconds, so a 40 ms region still gets dozens of samples); `nvidia-smi` once per 0.2 s if pynvml is unavailable."""
    REASONS = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index; self.rows = []; self.stop_flag = False; self.max_mhz = None; self.nvml = None; self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml, self.handle = pynvml, h
        except Exception:
            self.nvml = None

    def run(self):
        if self.nvml is not None:
            n, h = self.nvml, self.handle
            while not self.stop_flag:
                try:
                    mhz = int(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                    self.rows.append((mhz, mask))
                except Exception:
                    pass
                time.sleep(0.002)
            return
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6 and f[0].isdigit():
                    mask = sum(bit for k, (bit, _) in enumerate(self.REASONS) if f[2 + k].lower().startswith("active"))
                    self.rows.append((int(f[0]), mask))
                    if f[1].isdigit(): self.max_mhz = int(f[1])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"]}
        sm = sorted(r[0] for r in self.rows)
        reasons = [name for bit, name in self.REASONS if any(r[1] & bit for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def pin_body_arrays(sim):
    """Moves the caller-side body arrays of a Sim into pinned host memory (what an application that streams state in and out every
    step would use) and re-points the BodyData struct at them.  Returns the owning tensors (keep them alive)."""
    import torch
    from nudge_b200 import abi
    keep = {}
    for name in ("transforms", "properties", "momentum", "idle"):
        a = getattr(sim, name)
        t = torch.empty(max(a.nbytes, 1), dtype=torch.uint8, pin_memory=True)
        v = t.numpy()[:a.nbytes].view(a.dtype)
        v[:] = a
        keep[name] = t; setattr(sim, name, v)
    sim.bodies = abi.BodyData(abi.ptr(sim.transforms), abi.ptr(sim.properties), abi.ptr(sim.momentum), abi.ptr(sim.idle), len(sim.transforms))
    return keep


def settle_gpu(sim, steps):
    for _ in range(steps):
        sim.step()
    return sim.counts()


def run_sharded(args, rank, world, local):
    """N > 1: ONE scene sharded across the GPUs (gx x gz cells, ghost copies of the neighbours' bodies); the ghost bodies' momentum is
    exchanged after the warm start and after every solver sweep by the C++ host behind nb_shard_* (include/nudge_b200.h): one
    ncclAllGather ("nccl") or the library's own peer-memory push/pull kernels over NVLink ("peer").  The whole sharded sub-step,
    exchanges included, is one CUDA-graph replay per step (nb_shard_step)."""
    import torch
    import torch.distributed as dist
    import nudge_b200
    from nudge_b200 import shard
    if args.dump_outputs:
        raise SystemExit("--dump-outputs: not available for a scene sharded across GPUs (use --replicas, or one GPU)")
    side = torch.cuda.Stream()                     # a capturable stream: nb_shard_step records the step into a CUDA graph there
    torch.cuda.set_stream(side)
    stream = side.cuda_stream
    cfg = CONFIGS[args.config]
    g = cfg["scene"](args, world)
    strong = cfg["scaling"] == "strong"
    unit_bodies = 65536.0 if not strong else float(g.n_bodies - 1)     # `value` counts steps of a scene of this many bodies
    gloo = dist.new_group(backend="gloo")          # host-side bookkeeping (handles, re-partition) and the parity check's host transport

    def make_sim(scene, max_bodies):
        sm = nudge_b200.Sim(scene, device=local, stream=stream, max_bodies=max_bodies, max_boxes=max_bodies, max_spheres=(max_bodies if g.n_spheres else 0), contact_capacity=30 * max_bodies)
        if args.solver == "throughput":
            sm.set_solver_mode("throughput")
        return sm

    sim = shard.ShardedSim(g, rank, world, make_sim, margin=args.margin, transport=args.transport, group=gloo)
    for k in range(args.presim):
        if k and k % 25 == 0:
            sim.reshard()
        sim.step()
    torch.cuda.synchronize(); dist.barrier()
    t_rs = time.perf_counter()
    sim.reshard()                                   # host side (gather, nb_shard_partition, re-upload, new plan): reported, outside the timed region
    torch.cuda.synchronize(); dist.barrier()
    reshard_ms = (time.perf_counter() - t_rs) * 1e3
    for _ in range(2):
        sim.step()

    # ---- parity of the path that is timed: the same steps from the same state through NCCL, peer memory and the host exchange ----
    def snapshot():
        sim.sim.download_bodies(); sim.sim.download_cache()
        s_ = sim.sim
        n = s_.cache.count
        return dict(transforms=s_.transforms.copy(), momentum=s_.momentum.copy(), idle=s_.idle.copy(), n=n,
                    tags=s_.cache_tags[:n].copy(), feats=s_.cache_features[:n].copy(), data=s_.cache_data[:n].copy())

    def restore(st):
        s_ = sim.sim
        s_.transforms[:] = st["transforms"]; s_.momentum[:] = st["momentum"]; s_.idle[:] = st["idle"]
        n = st["n"]; s_.cache_tags[:n] = st["tags"]; s_.cache_features[:n] = st["feats"]; s_.cache_data[:n] = st["data"]; s_.cache.count = n
        s_.upload_bodies(); s_.upload_cache()

    parity = None
    if not args.no_parity_check and args.solver == "parity":
        s0 = snapshot()
        res = {}
        for t in ("nccl", "peer", "host"):
            if t == "peer" and not getattr(sim, "peer_ok", True):
                res[t] = None
                continue
            restore(s0)
            for _ in range(3):
                sim.step(t)
            r_ = snapshot()
            res[t] = (r_["transforms"].tobytes(), r_["momentum"].tobytes(), r_["idle"].tobytes())
        same = torch.tensor([float(res["nccl"] == res["host"]), float(res["peer"] is None or res["peer"] == res["host"])], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        parity = {"steps": 3, "nccl_equals_host_exchange": bool(same[0] > 0), "peer_equals_host_exchange": bool(same[1] > 0),
                  "what": "3 steps from the same state through each transport; transforms, momentum and idle counters of every rank compared bit for bit"}
        restore(s0)
        if not (parity["nccl_equals_host_exchange"] and parity["peer_equals_host_exchange"]):
            if rank == 0:
                print("PARITY CHECK FAILED: %r" % parity, file=sys.stderr)

    K = args.steps
    E = lambda: torch.cuda.Event(enable_timing=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(transport):
        for _ in range(max(args.warmup, 3)):
            sim.step(transport)
        ev = [(E(), E()) for _ in range(K)]
        dist.barrier(); torch.cuda.synchronize()
        l0 = sim.launch_count()
        for k in range(K):
            flush.fill_(k & 255)
            ev[k][0].record()
            sim.step(transport)
            ev[k][1].record()
        torch.cuda.synchronize()
        n_launch = sim.launch_count() - l0
        dist.barrier()
        return float(sum(a.elapsed_time(b) for a, b in ev)), n_launch

    main_transport = sim.transport                      # "nccl" if the peer inboxes could not be opened on this box
    peer_ok = getattr(sim, "peer_ok", True)
    other = "nccl" if main_transport == "peer" else "peer"
    other_ms = float("nan")
    if peer_ok or other == "nccl":
        other_ms, _ = timed(other)
    sampler = ClockSampler(local); sampler.start()
    total_ms, launches = timed(main_transport)
    sampler.stop_flag = True
    graphed = sim.sim.shard_graph_active()
    # diagnostic: the same ranks stepping their local problems WITHOUT the ghost hand-over (not a simulation of the global scene any more:
    # timed after everything that is reported, state restored from a snapshot afterwards is not needed - the run ends here)
    local_only_ms = None
    if os.environ.get("NB_BENCH_LOCAL_ONLY", "0") == "1":
        keep = snapshot() if 'snapshot' in dir() else None
        sim.sim.shard_no_exchange(True)
        local_only_ms, _ = timed(main_transport)
        sim.sim.shard_no_exchange(False)
        if keep is not None:
            restore(keep)
    cnt = sim.sim.counts()
    lc = sim.local_counts()
    # end to end: host state of the local bodies in and out every step
    h2d = sum(getattr(sim.sim, n).nbytes for n in ("transforms", "properties", "momentum", "idle"))
    d2h = sum(getattr(sim.sim, n).nbytes for n in ("transforms", "momentum", "idle"))
    pinned = pin_body_arrays(sim.sim)
    sim.sim.download_bodies()
    for _ in range(2):
        sim.sim.upload_bodies(); sim.step(); sim.sim.download_bodies()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = E(), E()
    e0.record()
    for k in range(K):
        sim.sim.upload_bodies(); sim.step(); sim.sim.download_bodies()
    e1.record(); torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1)
    t = torch.tensor([total_ms, e2e_ms, other_ms], dtype=torch.float64, device="cuda")
    tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    per_rank = torch.zeros((world, 3), dtype=torch.float64, device="cuda")        # ms per step, contacts, ghosts of every rank: shows imbalance
    per_rank[rank] = torch.tensor([(local_only_ms if local_only_ms is not None else total_ms) / K, float(cnt.contacts), float(lc["ghosts"])], dtype=torch.float64, device="cuda")
    dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
    ssum = torch.tensor([float(cnt.contacts), float(lc["owned"]), float(lc["ghosts"]), float(lc["export"]), float(h2d), float(d2h), float(cnt.overflow)], dtype=torch.float64, device="cuda")
    dist.all_reduce(ssum, op=dist.ReduceOp.SUM)
    if rank == 0:
        total_ms, e2e_ms, other_ms = float(tmax[0]), float(tmax[1]), float(tmax[2])
        rate = K / (total_ms * 1e-3)
        gx, gz = sim.part["grid"]
        exch = {"nccl": "pack -> ONE ncclAllGather (called from the C++ host) -> unpack, after the warm start and after every sweep",
                "peer": "k_shard_push / k_shard_pull: export rows stored straight into the subscribers' inboxes over NVLink peer memory (CUDA IPC), arrival flags instead of a collective, after the warm start and after every sweep"}
        line = {
            "metric": "simulation steps/s", "value": rate * (g.n_bodies - 1) / unit_bodies, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "config": args.config, "bodies_total": int(g.n_bodies), "bodies_per_gpu_owned": int(ssum[1] / world), "ghost_bodies_per_gpu": int(ssum[2] / world),
                       "exchanged_rows_per_gpu_per_sweep": int(ssum[3] / world), "solver_iterations": int(g.iterations), "contacts_incl_ghost_copies": int(ssum[0]),
                       "transport": main_transport, "exchange": exch[main_transport], "other_transport": other, "other_transport_scene_steps_per_s": (K / (other_ms * 1e-3) if other_ms == other_ms else None),
                       "peer_memory_available": bool(peer_ok),
                       "step_call": ("nb_shard_step: one CUDA-graph replay per step (kernels + exchanges)" if graphed else "nb_shard_step: plain launches"),
                       "presim_steps": args.presim, "parallelism": "one scene of %d bodies in %d x %d cells (x, z), one cell per GPU; halo = body radius + max radius + %.2f" % (g.n_bodies - 1, gx, gz, args.margin),
                       "value_definition": ("scene steps/s of the fixed-size scene" if strong else "scene steps/s x (total bodies / 65,536): 65,536-box-equivalent steps per second of the whole job"),
                       "scene_steps_per_s": rate, "l2": "flushed between timed steps (256 MiB write), flush excluded", "timing": "CUDA events per step, summed; max over ranks",
                       "overflow_flags": int(ssum[6]), "reshard_ms_host_side_untimed": reshard_ms,
                       ("per_rank_local_only_ms_per_step" if local_only_ms is not None else "per_rank_ms_per_step"): [round(float(x), 4) for x in per_rank[:, 0]], "per_rank_contacts": [int(x) for x in per_rank[:, 1]], "per_rank_ghosts": [int(x) for x in per_rank[:, 2]],
                       "solver_mode": ("throughput (mass-splitting Jacobi) inside a rank" if args.solver == "throughput" else "exact reference Gauss-Seidel order inside a rank") + ", block-Jacobi across ranks"},
            "parity_check": parity,
            "e2e": {"value": ((g.n_bodies - 1) / unit_bodies) * K / (e2e_ms * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": int(ssum[4]), "d2h_bytes_per_step": int(ssum[5]),
                    "what": "per rank: nb_upload_bodies (host) + nb_shard_step + nb_download_bodies, every step"},
            "gpu_launches": int(launches), "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "kernel": "k_solve", "achieved": None, "peak": peaks()[0], "unit": "GB/s", "frac": None, "traffic": None,
                         "note": "per-sweep launches interleaved with the ghost exchange; see the N=1 line for the solver roofline"},
        }
        emit(line)
    sim.sim.close()
    dist.destroy_process_group()


def run_ours(args):
    import torch
    import torch.distributed as dist
    import nudge_b200
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        if not args.replicas:
            return run_sharded(args, rank, world, local)
    # everything runs on one non-default stream: nb_step records its launches into a CUDA graph there (the legacy default
    # stream cannot be captured); torch.cuda.Event and the L2 flush follow torch's current stream, i.e. the same one
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    stream = side.cuda_stream
    cfg = CONFIGS[args.config]
    if args.config == "c2":
        scene = scenes.box_drop(args.boxes, iterations=args.iterations or 8, seed=2 + rank)
    else:
        scene = cfg["scene"](args, 1)
    sim = nudge_b200.Sim(scene, device=local, stream=stream)
    if args.solver == "throughput":
        sim.set_solver_mode("throughput")
    c = settle_gpu(sim, args.presim)
    if c.overflow:
        raise RuntimeError("capacity overflow during settling: %d" % c.overflow)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def staged_step(ev=None, st=None):
        sim.collide()
        if st: st[0].record()
        sim.apply_gravity_damping(); sim.read_cached_impulses()
        if st: st[1].record()
        sim.setup_contact_constraints()
        if ev: ev[0].record()
        sim.apply_impulses(scene.iterations)
        if ev: ev[1].record()
        sim.update_cached_impulses(); sim.write_cached_impulses(); sim.advance()

    for _ in range(max(args.warmup, 3)):
        sim.step()
    K = args.steps
    E = lambda: torch.cuda.Event(enable_timing=True)
    step_ev = [(E(), E()) for _ in range(K)]
    sampler = ClockSampler(local); sampler.start()
    if world > 1: dist.barrier()
    torch.cuda.synchronize()
    launches0 = sim.launch_count()
    prof = os.environ.get("NB_CUDA_PROFILER")     # "1": the timed nb_step loop; "staged": the stage-call loop below
    if prof and prof != "staged":
        torch.cuda.profiler.start()           # ncu --profile-from-start off: capture the timed region only
    wall0 = time.perf_counter()
    for k in range(K):
        flush.fill_(k & 255)                      # L2 flush between timed iterations (not part of the step time)
        step_ev[k][0].record()
        sim.step()                                # one nb_step call = one sub-step of the hot path
        step_ev[k][1].record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    if prof and prof != "staged":
        torch.cuda.profiler.stop()
    launches = sim.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_bodies(sim, args.dump_outputs)
    if world > 1: dist.barrier()
    sampler.stop_flag = True
    step_ms = [a.elapsed_time(b) for a, b in step_ev]
    total_ms = float(sum(step_ms))

    # ---- stage breakdown and the solver's launch time: the same step through the seven stage calls (untimed for `value`) ----
    KS = min(K, 10)
    sstep_ev = [(E(), E()) for _ in range(KS)]; solve_ev = [(E(), E()) for _ in range(KS)]; stage_ev = [(E(), E()) for _ in range(KS)]
    if prof == "staged":
        torch.cuda.profiler.start()
    sim.timing_enable(True)                       # CUDA events around every launch of the dominant solver kernel, recorded by the library on its stream
    kernel_launches, kernel_ms = 0, 0.0
    for k in range(KS):
        flush.fill_(k & 255)
        sstep_ev[k][0].record()
        staged_step(solve_ev[k], stage_ev[k])
        sstep_ev[k][1].record()
        nl, ms = sim.timing(); kernel_launches += nl; kernel_ms += ms
    torch.cuda.synchronize()
    sim.timing_enable(False)
    if prof == "staged":
        torch.cuda.profiler.stop()
    solve_ms = [a.elapsed_time(b) for a, b in solve_ev]
    staged_ms = [a.elapsed_time(b) for a, b in sstep_ev]
    stage_ms = {"collide": float(np.mean([sstep_ev[k][0].elapsed_time(stage_ev[k][0]) for k in range(KS)])),
                "gravity+read_cached_impulses": float(np.mean([stage_ev[k][0].elapsed_time(stage_ev[k][1]) for k in range(KS)])),
                "setup_contact_constraints": float(np.mean([stage_ev[k][1].elapsed_time(solve_ev[k][0]) for k in range(KS)])),
                "apply_impulses": float(np.mean(solve_ms)),
                "update+write_cache+advance": float(np.mean([solve_ev[k][1].elapsed_time(sstep_ev[k][1]) for k in range(KS)])),
                "whole_step_staged": float(np.mean(staged_ms))}
    cnt = sim.counts()

    # ---- end to end through the public API with HOST buffers (pinned): upload state, step, read state back ----
    pinned = pin_body_arrays(sim)
    sim.download_bodies()
    h2d = sum(getattr(sim, n).nbytes for n in ("transforms", "properties", "momentum", "idle"))
    d2h = sum(getattr(sim, n).nbytes for n in ("transforms", "momentum", "idle"))
    for _ in range(3):
        sim.upload_bodies(); sim.step(); sim.download_bodies()
    if world > 1: dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = E(), E()
    e0.record()
    for k in range(K):
        sim.upload_bodies(); sim.step(); sim.download_bodies()   # download synchronises: the caller holds the new transforms
    e1.record(); torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1)

    # ---- the same settled scene through the throughput-mode solver (extra key; `value` stays the parity-mode number) ----
    tp_leg = None
    if world == 1 and args.solver == "parity" and not args.no_throughput_leg:
        tp_leg = throughput_leg(sim, scene, flush, K)

    t = torch.tensor([total_ms, e2e_ms, float(cnt.contacts), float(sum(solve_ms))], dtype=torch.float64, device="cuda")
    torch.cuda.set_stream(torch.cuda.default_stream())
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        total_ms, e2e_ms = float(tmax[0]), float(tmax[1]); contacts_all = float(tsum[2])
    else:
        contacts_all = float(cnt.contacts)
    if rank != 0:
        if world > 1: dist.destroy_process_group()
        return
    steps_per_s = world * K / (total_ms * 1e-3)          # every rank advances its own 64k-box scene: replicas of the workload
    e2e_steps_per_s = world * K / (e2e_ms * 1e-3)
    peak, peak_src = peaks()
    sweeps = scene.iterations
    C, A = cnt.contacts, cnt.active
    throughput = args.solver == "throughput"
    sweeps_per_launch = 1 if throughput else sweeps        # k_jacobi_sweep = one sweep per launch; k_solve = all sweeps of a step in one launch
    alg_bytes = (184.0 * C + 64.0 * A) * sweeps_per_launch  # SURVEY.md §8(d): per sweep 184 B/contact + 64 B/active body
    solve_avg_ms = kernel_ms / max(kernel_launches, 1)      # live: CUDA events around each launch of that kernel in the stage-call loop above
    achieved = alg_bytes / (solve_avg_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "solver_traffic_throughput.json" if throughput else "solver_traffic.json")
    if os.path.exists(tp):
        try: traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception: traffic = None
    line = {
        "metric": "simulation steps/s", "value": steps_per_s, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "config": args.config, "bodies_per_gpu": scene.n_bodies, "colliders_per_gpu": scene.n_colliders, "solver_iterations": sweeps,
                   "contacts": int(C), "broadphase_pairs": int(cnt.pairs), "batches": int(cnt.batches),
                   "presim_steps": args.presim,
                   "solver_mode": ("throughput: mass-splitting Jacobi over the reference's rows (not bit-comparable with the reference; see DESIGN.md)" if throughput else "exact reference Gauss-Seidel order (per-body dataflow)"),
                   "parallelism": "1 GPU" if world == 1 else "%d independent replicas of the workload, one per GPU (no cross-GPU contacts)" % world,
                   "l2": "flushed between timed steps (256 MiB write), flush excluded from step time", "timing": "CUDA events around each nb_step call, summed; max over ranks",
                   "step_call": "nb_step (CUDA graph replay of the step's launches); stage_ms is the same step through the seven stage calls"},
        "contacts_solved_per_s": contacts_all * sweeps * K / (total_ms * 1e-3),
        "wall_ms_per_step_incl_flush": wall * 1e3 / K,
        "solver_share_of_step": float(np.mean(solve_ms)) / float(np.mean(staged_ms)), "stage_ms": stage_ms,
        "roofline": {"bound": "hbm", "kernel": ("k_jacobi_sweep (one sweep per launch)" if throughput else "k_solve (%d sweeps per launch)" % sweeps), "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": solve_avg_ms, "timed_launches": kernel_launches,
                     "note": ("streams the rows once per sweep through TMA bulk copies; body velocities and accumulators stay in L2" if throughput else
                              "latency bound: the reference's Gauss-Seidel order is a dependency chain per body; rows stay L2 resident")},
        "e2e": {"value": e2e_steps_per_s, "unit": "steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "what": "nb_upload_bodies (pinned host) + nb_step + nb_download_bodies per step"},
        "gpu_launches": int(launches), "clocks": sampler.summary(),
    }
    if tp_leg:
        line["throughput_mode"] = tp_leg
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_sample(args)
        line["dropin_seven_call_steps_per_s"] = dropin_sample()
    emit(line)
    if world > 1: dist.destroy_process_group()


def dump_bodies(sim, out_dir):
    """What a caller of nb_step receives after the last timed step (nb_download_bodies): every body's transform, momentum and idle counter,
    float32, one .npy per field: 3.7 MB for the default 65,537 bodies, 59 MB for the largest config (c4).  The scene and its settling are
    seeded, so two builds given the same arguments can be compared file for file.  Under --replicas, rank 0's scene."""
    sim.download_bodies()
    os.makedirs(out_dir, exist_ok=True)
    fields = {"position": sim.transforms["position"], "rotation": sim.transforms["rotation"], "velocity": sim.momentum["velocity"],
              "angular_velocity": sim.momentum["angular_velocity"], "idle_counter": sim.idle}
    for name, a in fields.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def throughput_leg(sim, scene, flush, K):
    """The workload of the line, continued from the state the timed loop left, with nb_set_solver_mode(NB_SOLVER_THROUGHPUT): same
    timing rules (L2 flush between steps, CUDA events around nb_step), and the roofline of ITS dominant kernel, k_jacobi_sweep, from
    the library's own events around each launch.  The solver mode is switched back afterwards."""
    import torch
    E = lambda: torch.cuda.Event(enable_timing=True)
    sim.set_solver_mode("throughput")
    try:
        for _ in range(5):
            sim.step()
        ev = [(E(), E()) for _ in range(K)]
        torch.cuda.synchronize()
        for k in range(K):
            flush.fill_(k & 255)
            ev[k][0].record(); sim.step(); ev[k][1].record()
        torch.cuda.synchronize()
        ms = float(sum(a.elapsed_time(b) for a, b in ev))
        sim.timing_enable(True)
        nl, kms = 0, 0.0
        for k in range(min(K, 5)):
            flush.fill_(k & 255)
            sim.collide(); sim.apply_gravity_damping(); sim.read_cached_impulses(); sim.setup_contact_constraints()
            sim.apply_impulses(scene.iterations)
            sim.update_cached_impulses(); sim.write_cached_impulses(); sim.advance()
            a, b = sim.timing(); nl += a; kms += b
        sim.timing_enable(False)
        cnt = sim.counts()
    finally:
        sim.set_solver_mode("parity")
    peak, peak_src = peaks()
    alg = 184.0 * cnt.contacts + 64.0 * cnt.active
    avg = kms / max(nl, 1)
    achieved = alg / (avg * 1e-3) / 1e9
    return {"value": K / (ms * 1e-3), "unit": "steps/s", "ms_per_step": ms / K, "contacts": int(cnt.contacts),
            "solver_mode": "throughput: mass-splitting Jacobi over the reference's rows (nb_set_solver_mode; not bit-comparable with the reference, DESIGN.md 2.11)",
            "roofline": {"bound": "hbm", "kernel": "k_jacobi_sweep (one sweep per launch)", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "traffic_note": "measured on c4 only (1M boxes): profiles/solver_traffic_throughput.json, 1.11x the algorithmic bytes", "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg, "avg_launch_ms": avg, "timed_launches": int(nl),
                         "note": "on a 64k-body scene the rows (184 B/contact) fit the 126 MB L2 and the flush only evicts them once per step, so this figure mixes "
                                 "L2 and HBM streaming; the HBM-bound case is --config c4 --solver throughput"}}


def dropin_sample():
    """Cost of the LITERAL drop-in (libnudge_compat.so: the seven nudge:: calls with HOST pointers, every call uploading what it reads and
    downloading what it writes): oracle/_ref/headless_gpu, an application loop in the shape of example/main.cpp:274-328 on 1024 boxes + 1024
    spheres (BASELINE configs[0]), next to the same binary linked with the reference's nudge.cpp.  Not the fast path (nb_step is)."""
    d = os.path.join(ROOT, "oracle", "_ref")
    out = {}
    for name in ("headless_gpu", "headless_ref"):
        exe = os.path.join(d, name)
        if not os.path.exists(exe):
            return None
        try:
            r = subprocess.run([exe, "1024", "1024", "400", "8"], capture_output=True, text=True, timeout=300)
            out[name] = float([l for l in r.stdout.splitlines() if l.startswith("steps_per_s")][0].split()[1])
        except Exception as e:  # noqa: BLE001
            out[name] = None; out[name + "_error"] = repr(e)[:200]
    return {"gpu_dropin": out.get("headless_gpu"), "reference_cpu_1_thread": out.get("headless_ref"),
            "scene": "1024 boxes + 1024 spheres falling, 400 steps from the drop, 8 iterations, gravity loop on the host between the calls"}


def cpu_baseline_sample(args):
    """The unmodified reference (oracle/_ref, -O3 -mavx2 -mfma, FTZ/DAZ on like example/main.cpp:338-339) on the host: one
    8191-box pile of the same generator (the reference's 2^13 collider limit, nudge.cpp:3010), settled on the GPU, then timed."""
    import nudge_b200
    from oracle import pyref
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libnudge_ref_fast.so")):
        return None                               # the reference is not built in this tree (oracle/Makefile needs its sources)
    s = CONFIGS[args.config]["small"](args, 77)
    g = nudge_b200.Sim(s)
    settle_gpu(g, args.presim)
    g.download_bodies(); g.download_cache()
    r = pyref.RefSim(s, fast=True, ftz=True, contact_capacity=g.cap)
    r.transforms[:] = g.transforms; r.momentum[:] = g.momentum; r.idle[:] = g.idle
    from nudge_b200 import abi
    n = g.cache.count
    r.cache_tags[:n] = abi.wide_tag_to_ref(g.cache_tags[:n], g.cache_features[:n]); r.cache_data[:n] = g.cache_data[:n]; r.cache.count = n
    g.close()
    for _ in range(5):
        r.step()
    t0 = time.perf_counter(); k = 0
    while time.perf_counter() - t0 < 10.0:
        r.step(); k += 1
    dt = time.perf_counter() - t0
    return {"value": k / dt, "unit": "steps/s", "cores": 1, "kind": "reference",
            "sample": "one %d-body settled scene (%d contacts) of the same generator (%s), %d steps in %.1f s; the reference cannot run more than 8192 colliders (nudge.cpp:3010)" % (s.n_bodies - 1, r.contacts.count, s.name, k, dt),
            "host_cpus": os.cpu_count()}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation (oracle/_ref) with all the host threads it can use.  The library is
    single threaded and capped at 8192 colliders, so the arm's scene is run as independent piles of the reference's maximum size, one
    host thread each: 8 piles for the 65,536-box workload, and - like the repo's arm, whose c1 / c2 scene grows with the GPU count
    (weak scaling) - N times as many under `--gpus N`; the fixed-size scenes c3 / c4 / c5 take as many piles as cover them."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oracle import pyref
    world = int(os.environ.get("WORLD_SIZE", 1))
    weak = CONFIGS[args.config]["scaling"] == "weak"
    tiles = {"c1": 1, "c2": 8, "c3": 32, "c4": 128, "c5": 32}[args.config] * (world if weak else 1)
    threads = min(tiles, os.cpu_count() or 1)
    sims = [None] * tiles

    def work(fn):
        ths = [threading.Thread(target=fn, args=(t,)) for t in range(tiles)]
        # at most `threads` run at once
        for b in range(0, tiles, threads):
            for th in ths[b:b + threads]: th.start()
            for th in ths[b:b + threads]: th.join()

    def make(t):
        s = CONFIGS[args.config]["small"](args, 100 + t)
        sims[t] = pyref.RefSim(s, fast=True, ftz=True)
        for _ in range(args.ref_presim):
            sims[t].step()

    def step(t):
        sims[t].lib.ref_set_ftz_daz(1)
        sims[t].step()

    work(make)
    for _ in range(max(args.warmup, 1)):
        work(step)
    K = args.steps
    t0 = time.perf_counter()
    for _ in range(K):
        work(step)
    dt = time.perf_counter() - t0
    # the repo's arm counts a weak-scaling job in units of the one-GPU scene (N x 65,536 boxes stepped once = N steps): same here
    value = (world if weak else 1) * K / dt
    contacts = sum(s.contacts.count for s in sims)
    line = {"impl": "reference", "metric": "simulation steps/s", "value": value, "unit": "steps/s", "n_gpus": world, "steps": K,
            "warmup": max(args.warmup, 1), "ms_per_step": dt * 1e3 / K, "higher_is_better": True, "scaling": CONFIGS[args.config]["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": CONFIGS[args.config]["workload"], "config": args.config,
                       "sample": "%d independent scenes of the same generator at the reference's size limit (%s: %d bodies each, %d contacts in all) stepped together, %d host threads" % (tiles, sims[0].scene.name, sims[0].scene.n_bodies - 1, contacts, threads),
                       "solver_iterations": int(sims[0].scene.iterations), "presim_steps": args.ref_presim,
                       "value_definition": ("job steps/s x N: the job steps N one-GPU scenes (N x %d piles) at once" % (tiles // world) if weak else "steps/s of the fixed-size scene, run as %d piles" % tiles)},
            "cpu_baseline": {"value": value, "unit": "steps/s", "cores": threads, "kind": "reference",
                             "sample": "%d scenes (%s) per step; unmodified nudge.cpp, g++ -O3 -mavx2 -mfma, FTZ/DAZ on" % (tiles, sims[0].scene.name)},
            "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def main():
    _own_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--boxes", type=int, default=65536)
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json configs[0..4] = c1..c5 (default c2, the configuration the metric is quoted on)")
    ap.add_argument("--iterations", type=int, default=0, help="solver sweeps per step (0 = the config's own)")
    ap.add_argument("--presim", type=int, default=-1, help="untimed settling steps before the measurement (-1 = the config's own)")
    ap.add_argument("--ref-presim", type=int, default=700)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-throughput-leg", action="store_true", help="skip the extra throughput-mode measurement of the same scene (key throughput_mode)")
    ap.add_argument("--solver", default="parity", choices=["parity", "throughput"], help="parity = the reference's exact Gauss-Seidel order (default, bit-identical results); throughput = mass-splitting Jacobi")
    ap.add_argument("--transport", default="peer", choices=["peer", "nccl"], help="N > 1: ghost exchange through the library's peer-memory kernels (default) or one ncclAllGather; both are timed, `value` is this one")
    ap.add_argument("--margin", type=float, default=0.5, help="N > 1: extra halo width beyond the bounding radii (room for motion between re-partitions)")
    ap.add_argument("--no-parity-check", action="store_true", help="N > 1: skip the NCCL / peer / host-exchange bit-equality check before the timed region")
    ap.add_argument("--replicas", action="store_true", help="N > 1: run N independent copies of the workload instead of one sharded scene")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the bodies' state after the last timed step as DIR/<field>.npy (float32; one scene per GPU only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none")
    if args.presim < 0:
        args.presim = CONFIGS[args.config]["presim"]
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
    sys.stdout.flush(); sys.stderr.flush()
