"""Per-frame tracking (RandomOptimizer -> GO) at two shapes, three arms alternated frame by frame in one run:
  composed: RandomOptimizer.optimize (pose read to the host) + sample_pixels_mix + FusedPoseRefiner.refine (its CUDA graph),
            then c2w.cpu() -- the route the reference consumes (bench.py's frame, scripts/prof_frame.py);
  graph:    FusedTracker.track with its CUDA graph, then c2w.cpu();
  eager:    FusedTracker.track(graph=False), then c2w.cpu().
Shapes: the reference's (FastCaMo-synth: RO 5 x 2000 particles x 16 x 24 pixels, GO 10 x 1000 rays x 75 samples) and BASELINE
configs[1] (RO 1024 particles x 32 x 64 pixels, 5 RO iterations as the reference's iter_RO, GO 20 x 1000 rays x 75 samples),
on one synthetic 620 x 460 frame, hash 2^19.

Per arm: host wall time from the call to the pose on the host (median over --frames frames after a warm-up), the device span
of the same frame (CUDA events around it), and -- in a separate torch.profiler pass of a few frames -- device kernels per
frame, host-issued launches per frame (kernel / graph launches, async copies and memsets seen by the profiler) and blocking
synchronisations per frame.  GPU name and power limit are read in the same run.  Prints one JSON line; --out writes it."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import torch  # noqa: E402

SHAPES = {
    "reference": dict(particles=2000, lattice=(16, 24), n_ro=5, n_go=10, n_px=1000),
    "baseline_c2": dict(particles=1024, lattice=(32, 64), n_ro=5, n_go=20, n_px=1000),
}


def gpu_info(index):
    try:
        q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"gpu": torch.cuda.get_device_name(index), "nvidia_smi": q}


def setup(shape, dev):
    import helpers as H
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    cfg = H.make_config(19, n_samples_d=50, n_range_d=25)
    lh, lw = shape["lattice"]
    cfg["tracking"] = {"RO": {"particle_size": shape["particles"], "initial_scaling_factor": 0.02, "rescaling_factor": 0.5,
                              "n_rows": lh, "n_cols": lw},
                       "ignore_edge_W": 20, "ignore_edge_H": 20, "lr_rot": 1e-3, "lr_trans": 1e-3, "wait_iters": 100, "best": True,
                       "iter_RO": shape["n_ro"], "iter": shape["n_go"], "sample": shape["n_px"]}
    model = H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=13)))
    dirs = synth.camera_rays()
    c2w = synth.trajectory(4)[1]
    frame = synth.render_frame(c2w, dirs)
    ds = types.SimpleNamespace(H=460, W=620, fx=320.0, fy=320.0, cx=309.5, cy=229.5, rays_d=dirs)
    g = torch.Generator().manual_seed(5)
    particles = torch.randn(shape["particles"], 6, generator=g).clamp(-2, 2)
    particles[0] = 0
    ro = mf.RandomOptimizer(cfg, types.SimpleNamespace(dataset=ds, device=str(dev)), particles=particles)
    init = c2w.clone()
    init[:3, 3] += torch.tensor([0.01, -0.008, 0.006])
    return types.SimpleNamespace(model=model, ro=ro, refiner=mf.FusedPoseRefiner(model), tracker=mf.FusedTracker(model, ro),
                                 depth=frame["depth"].to(dev), rgb=frame["rgb"].to(dev), dirs=dirs.to(dev), init=init.to(dev))


def arms(s, shape):
    from mipsfusion_b200 import sampling_helper as sh

    def composed():
        pose = s.ro.optimize(s.model, s.depth, s.init, s.init, n_iter=shape["n_ro"]).to(s.init.device)
        rows, cols = sh.sample_pixels_mix(460, 620, 16, 24, s.depth, shape["n_px"])
        c2w, _ = s.refiner.refine(pose, s.dirs[rows, cols], s.rgb[rows, cols], s.depth[rows, cols], shape["n_go"])
        return c2w.cpu()

    def graph():
        return s.tracker.track(s.depth, s.rgb, s.init)[0].cpu()

    def eager():
        return s.tracker.track(s.depth, s.rgb, s.init, graph=False)[0].cpu()
    return {"composed": composed, "graph": graph, "eager": eager}


def profile_counts(fn, frames):
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(frames):
            fn()
        torch.cuda.synchronize()
    kernels = launches = syncs = 0
    for e in prof.events():
        name = e.name
        if e.device_type == torch.autograd.DeviceType.CUDA:
            kernels += 1
        elif name.startswith(("cudaLaunchKernel", "cuLaunchKernel", "cudaGraphLaunch", "cudaMemcpyAsync", "cudaMemsetAsync")):
            launches += 1
        elif "Synchronize" in name:
            syncs += 1
    return {"device_ops_per_frame": kernels / frames, "host_launches_per_frame": launches / frames,
            "blocking_syncs_per_frame": syncs / frames}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--profile-frames", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_track.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"script": "scripts/bench_track.py", **gpu_info(0), "frames": a.frames, "shapes": {}}
    for name, shape in SHAPES.items():
        s = setup(shape, dev)
        fns = arms(s, shape)
        for _ in range(a.warmup):
            for fn in fns.values():
                fn()
        wall = {k: [] for k in fns}
        span = {k: [] for k in fns}
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.frames * len(fns))]
        torch.cuda.synchronize()
        i = 0
        for _ in range(a.frames):
            for k, fn in fns.items():
                e0, e1 = ev[i]
                i += 1
                t0 = time.perf_counter()
                e0.record()
                fn()
                e1.record()
                wall[k].append((time.perf_counter() - t0) * 1e3)
                span[k].append((e0, e1))
        torch.cuda.synchronize()
        out = {"shape": shape}
        for k in fns:
            dev_ms = [e0.elapsed_time(e1) for e0, e1 in span[k]]
            out[k] = {"host_ms_to_pose_median": round(statistics.median(wall[k]), 4),
                      "host_ms_min": round(min(wall[k]), 4), "device_span_ms_median": round(statistics.median(dev_ms), 4),
                      **profile_counts(fns[k], a.profile_frames)}
        out["graph_error"] = s.tracker.__dict__.get("_graph_error")
        out["host_ms_saved_graph_vs_composed"] = round(out["composed"]["host_ms_to_pose_median"] - out["graph"]["host_ms_to_pose_median"], 4)
        res["shapes"][name] = out
        del s, fns
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
