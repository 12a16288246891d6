"""Ray-cast throughput on a settled pile (nb_build_query_tree + nb_raycast, DESIGN.md section 8.5).

Scenes: c2 (65,536-box settled pile, scenes.box_drop seed 2) and c4 (1M boxes), settled with nb_step as bench.py does.  Times the build and
2^20 / 2^24 rays with device I/O in two sets: coherent (downward rays from a grid above the pile) and incoherent (random directions from
random points inside the pile's bounds).  CUDA events around windows of back-to-back calls, each window longer than --window-s; the
reported figure is the median of --windows windows after warm-up.  The tree and leaf records (a few MB to tens of MB) fit the 126 MB L2
and are read from there after the first pass; rays and hits stream through HBM.  Prints one JSON object and writes it to --out.

    python scripts/bench_raycast.py --configs c2,c4 --out profiles/r03a_raycast.json"""
import argparse, json, os, subprocess, sys, time
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCENES = {"c2": (65536, 900), "c4": (1 << 20, 900)}   # boxes, settling steps (bench.py's presim)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def timed(fn, torch, windows, window_s):
    """Median seconds per call over `windows` CUDA-event windows, each at least window_s long."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter(); fn(); torch.cuda.synchronize(); one = max(time.perf_counter() - t0, 1e-6)
    reps = max(1, int(window_s / one) + 1)
    per = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record(); b.synchronize()
        per.append(a.elapsed_time(b) / 1e3 / reps)
    return float(np.median(per)), reps, [float(x) for x in per]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c4")
    ap.add_argument("--log2-rays", default="20,24")
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--window-s", type=float, default=0.5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import nudge_b200
    from nudge_b200 import scenes
    if not torch.cuda.is_available():
        raise SystemExit("bench_raycast: no CUDA device (there is no CPU path)")
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    res = dict(metric="rays/s", gpu=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit_max_sm_clock=gpu_info(),
               method="CUDA events around back-to-back nb_raycast calls (device I/O); median of %d windows of >= %.2f s after 3 warm-up calls" % (a.windows, a.window_s),
               results=[])
    for cfg in a.configs.split(","):
        nbox, settle = SCENES[cfg]
        s = scenes.box_drop(nbox, iterations=8, seed=2)
        sim = nudge_b200.Sim(s, stream=side.cuda_stream)
        for _ in range(settle):
            sim.step()
        sim.download_bodies()
        c = sim.counts()
        K = s.n_colliders
        nodes, m = K, K
        while m > 8:
            m = (m + 7) // 8; nodes += m
        tree_bytes = 32 * nodes + 48 * K
        build_s, build_reps, _ = timed(sim.build_query_tree, torch, a.windows, a.window_s)
        pos = torch.from_numpy(sim.transforms["position"][1:].copy()).cuda()
        lo, hi = pos.min(0).values, pos.max(0).values
        gen = torch.Generator(device="cuda"); gen.manual_seed(1)
        for lg in (int(x) for x in a.log2_rays.split(",")):
            n = 1 << lg
            for kind in ("coherent", "incoherent"):
                rays = torch.zeros((n, 8), dtype=torch.float32, device="cuda")
                if kind == "coherent":
                    side_n = int(np.ceil(np.sqrt(n)))
                    i = torch.arange(n, device="cuda")
                    u, v = (i % side_n).float() / max(side_n - 1, 1), (i // side_n).float() / max(side_n - 1, 1)
                    rays[:, 0] = lo[0] + u * (hi[0] - lo[0]); rays[:, 2] = lo[2] + v * (hi[2] - lo[2]); rays[:, 1] = hi[1] + 5.0
                    rays[:, 5] = -1.0
                else:
                    rays[:, 0:3] = lo + torch.rand((n, 3), device="cuda", generator=gen) * (hi - lo)
                    rays[:, 4:7] = torch.randn((n, 3), device="cuda", generator=gen)
                rays[:, 3] = float("inf")
                rays.view(torch.int32)[:, 7] = -1           # ignore_body = NB_NO_BODY
                hits = torch.empty((n, 8), dtype=torch.float32, device="cuda")
                fn = lambda: sim.raycast(device_ptr=rays.data_ptr(), hits_ptr=hits.data_ptr(), n=n)
                sec, reps, per = timed(fn, torch, a.windows, a.window_s)
                frac = float((hits.view(torch.int32)[:, 1] != -1).float().mean())
                res["results"].append(dict(config=cfg, colliders=K, contacts=c.contacts, rays=n, set=kind, hit_fraction=frac,
                                           ms_per_call=sec * 1e3, rays_per_s=n / sec, calls_per_window=reps, window_ms=[x * 1e3 for x in per],
                                           io_bytes_per_ray=64, io_GB_per_s=64 * n / sec / 1e9))
                print(json.dumps(res["results"][-1]), flush=True)
                del rays, hits
        res["results"].append(dict(config=cfg, colliders=K, build_ms=build_s * 1e3, builds_per_window=build_reps,
                                   tree_and_leaf_bytes=tree_bytes, l2_resident=tree_bytes < 126e6))
        print(json.dumps(res["results"][-1]), flush=True)
        sim.close()
        torch.cuda.synchronize()
    out = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(out + "\n")
    print(out)


if __name__ == "__main__":
    main()
