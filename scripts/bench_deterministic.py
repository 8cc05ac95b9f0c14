"""Cost of deterministic mode (mipsfusion_b200.set_deterministic) on three routes, default and deterministic alternated call by
call in one process:
  map    FusedMapper.step at bench.py's shape (C1: 4096 rays x 43 samples, T = 2^19), L2 flushed (256 MB write) before each
         timed step as bench.py does;
  ba     FusedMapper.local_ba at C3, S = 43 (scripts/bench_ba.py's shape: 50 keyframes, 4096 rays, 15 iterations, pose step every 5);
  track  FusedTracker.track (graph) at the reference shape (scripts/bench_track.py: 2000 particles, 5 RO + 10 GO iterations, 1000 px).
Then, in a separate pass with torch.profiler, the deterministic map step's own kernels (rows are written by the backward; the
fixed-point passes det_pass1 / det_pass2 / det_finalize) and the library-owned workspace size.  Card name and power limit are
read in the same run.  Prints one JSON line; --out also writes it."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")]

import torch  # noqa: E402


def alternate(fns, reps, warmup, before=None):
    """fns: mode -> callable; -> mode -> list of ms (CUDA events), modes alternated call by call."""
    import mipsfusion_b200 as mf
    prev = mf.get_deterministic()
    out = {k: [] for k in fns}
    try:
        for i in range(warmup + reps):
            for k, f in fns.items():
                mf.set_deterministic(k == "det")
                if before:
                    before()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                f()
                b.record()
                b.synchronize()
                if i >= warmup:
                    out[k].append(a.elapsed_time(b))
    finally:
        mf.set_deterministic(prev)
    return out


def summary(t):
    res = {}
    for k, v in t.items():
        s = sorted(v)
        res[k] = {"ms_median": s[len(s) // 2], "ms_min": s[0], "ms_max": s[-1], "n": len(s)}
    res["det_over_default"] = res["det"]["ms_median"] / res["default"]["ms_median"]
    res["det_minus_default_ms"] = res["det"]["ms_median"] - res["default"]["ms_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--routes", default="map,ba,track")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_deterministic.py needs a GPU")
    import bench
    import bench_ba
    import bench_track
    import helpers as H
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200.mapper import FusedMapper
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"script": "scripts/bench_deterministic.py", **bench_track.gpu_info(0), "reps": args.reps}
    routes = args.routes.split(",")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    if "map" in routes:
        cfg, of = bench.build_model()
        state = H.state_of(of)
        rays_o, rays_d, rgb, d, _ = bench.make_inputs(0)
        ro, rd, tc, td = (t.to(dev).contiguous() for t in (rays_o, rays_d, rgb, d.reshape(-1)))
        m = {k: FusedMapper(H.cuda_model(cfg, state)) for k in ("default", "det")}
        fns = {k: (lambda k=k: m[k].step(ro, rd, tc, td)) for k in m}
        res["map"] = summary(alternate(fns, args.reps, args.warmup, before=flush.zero_))
        res["map"]["shape"] = f"{bench.R_RAYS} rays x {bench.S} samples, T = 2^{bench.HASH}"
        # the deterministic step's kernels, profiled in a pass of their own
        from torch.profiler import ProfilerActivity, profile
        prev = mf.get_deterministic()
        mf.set_deterministic(True)
        try:
            for _ in range(3):
                m["det"].step(ro, rd, tc, td)
            torch.cuda.synchronize()
            steps = 20
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(steps):
                    flush.zero_()
                    m["det"].step(ro, rd, tc, td)
                torch.cuda.synchronize()
        finally:
            mf.set_deterministic(prev)
        kern = {}
        for e in prof.key_averages():
            if e.device_type is not None and "CUDA" in str(e.device_type) and e.count > 0:
                name = e.key.split("(")[0][:80]
                t_us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                kern[name] = {"us_per_step": t_us / steps, "calls_per_step": e.count / steps}
        res["map"]["det_kernels_us_per_step"] = dict(sorted(kern.items(), key=lambda kv: -kv[1]["us_per_step"])[:16])
        res["map"]["det_passes_us_per_step"] = sum(v["us_per_step"] for k, v in kern.items() if k.startswith("det_"))
        res["workspace_bytes_map"] = int(L.lib().mf_det_workspace_bytes())
        del m

    if "ba" in routes:
        n_kf, R, n_cur, iters = 50, 4096, 512, 15
        cfg = H.make_config(19, n_samples_d=32, n_range_d=11)
        cfg["sampling"] = {"kf_n_rays_h": 150, "kf_n_rays_w": 200}
        st, poses = bench_ba.build_store(cfg, n_kf, dev)
        poses_d = poses.to(dev)
        cur = st.rays[n_kf - 1, ::58][:n_cur].contiguous()
        state = H.state_of(H.oracle_field(cfg, grid_scale=0.3))
        hp = dict(n_iters=iters, pose_accum_step=5, lr_rot=1e-3, lr_trans=1e-3, optim_cur=True)
        m = {k: FusedMapper(H.cuda_model(cfg, state)) for k in ("default", "det")}
        fns = {k: (lambda k=k: m[k].local_ba(st, 0, list(range(n_kf)), poses_d, R - n_cur, cur_rays7=cur, seed=11, **hp)) for k in m}
        res["ba"] = summary(alternate(fns, max(args.reps // 5, 5), 2))
        res["ba"]["shape"] = "local_ba C3, S = 43: 50 keyframes, 4096 rays, 15 iterations, pose step every 5"
        del m, st

    if "track" in routes:
        shape = bench_track.SHAPES["reference"]
        s = {k: bench_track.setup(shape, dev) for k in ("default", "det")}
        fns = {k: (lambda k=k: s[k].tracker.track(s[k].depth, s[k].rgb, s[k].init)) for k in s}
        res["track"] = summary(alternate(fns, args.reps, args.warmup))
        res["track"]["shape"] = "FusedTracker.track (graph), reference shape: 2000 particles 16 x 24, 5 RO + 10 GO, 1000 px x 75"
    res["workspace_bytes_total"] = int(L.lib().mf_det_workspace_bytes())
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
