"""Submap initialisation (the reference's first_frame_mapping / initialize_new_localMLP) and the per-iteration current-frame
draw of local bundle adjustment, on one GPU.

Init arms, on a 620 x 460 synthetic frame with a T = 2^19 hash grid, alternated call by call, each call ending with the losses on
the host:
  (a) FusedMapper.first_frame_mapping: draw + map step per iteration on the device, no host sync inside the call;
  (b) the reference's loop body on the per-step API: host random.sample(range(H*W), n), the column-major gather from the host
      frame into pinned memory, then step_host (one copy and one synchronisation per iteration).
Shapes: the reference's init shape (500 iterations x 1800 rays x 75 samples) and the C1 ray shape (4096 rays x 43 samples, also
500 iterations).  Reported per arm and shape: median ms per call and per iteration, launches per iteration, and for (a) the host
time to enqueue a call next to its device time (both per iteration): when the first is the larger, eager issue leaves the GPU idle.

BA arm: local_ba at the C3 shape of scripts/bench_ba.py (50 keyframes, 3584 store rays + 512 current-frame rays, 15 iterations,
pose step every 5, S = 43) with ``cur_frame`` (512 pixels drawn afresh every iteration, keys on the device) against
``cur_rays7`` (the same 512 rows every iteration).

Prints one JSON line with the GPU name and power limit read in the same run; ``--out`` also writes it to a file."""
import argparse
import json
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")]

import numpy as np  # noqa: E402
import torch  # noqa: E402


def median(v):
    return sorted(v)[len(v) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--ba-reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_init.py needs a GPU")
    import helpers as H
    from bench_ba import build_store, gpu_info, time_calls
    from mipsfusion_b200 import synth
    from mipsfusion_b200.mapper import FusedMapper
    dev = torch.device("cuda", torch.cuda.current_device())
    traj = synth.trajectory(51)
    fr = synth.render_frame(traj[50], synth.camera_rays(), seed=3)
    frame_h = {k: fr[k].contiguous() for k in ("direction", "rgb", "depth")}
    frame_d = {k: v.to(dev) for k, v in frame_h.items()}
    Hh, W = frame_h["depth"].shape
    res = dict(workload="submap initialisation on a %d x %d frame, T = 2^19, %d iterations per call; local_ba current-frame draw at "
                        "C3" % (W, Hh, args.iters), **gpu_info(dev.index))
    host_flat = torch.cat([frame_h["direction"], frame_h["rgb"], frame_h["depth"][..., None]], -1).numpy()     # (H, W, 7)
    for label, R, (nsd, nrd) in (("ref_init_1800x75", 1800, (50, 25)), ("c1_4096x43", 4096, (32, 11))):
        cfg = H.make_config(19, n_samples_d=nsd, n_range_d=nrd)
        state = H.state_of(H.oracle_field(cfg, grid_scale=0.3))
        m_a, m_b = FusedMapper(H.cuda_model(cfg, state)), FusedMapper(H.cuda_model(cfg, state))
        eye = torch.eye(4, device=dev)[None]
        pinned = torch.empty(R, 7).pin_memory()
        rng = random.Random(0)
        seeds = iter(range(0, 10 ** 9, args.iters))
        host_ms = []

        def arm_a():
            t0 = time.perf_counter()
            losses = m_a.first_frame_mapping(frame_d, args.iters, pix_num=R, seed=next(seeds))
            host_ms.append((time.perf_counter() - t0) * 1e3)
            return losses.cpu()

        def arm_b():
            out = None
            for _ in range(args.iters):
                i = np.asarray(rng.sample(range(Hh * W), R))                # mipsfusion.py:176-180
                pinned.numpy()[:] = host_flat[i % Hh, i // Hh]
                out = m_b.step_host(pinned, None, eye)
            return out.clone()

        counts = {}
        for name, m, f in (("a_first_frame_mapping", m_a, arm_a), ("b_host_loop", m_b, arm_b)):
            l0 = m.launches
            f()
            counts[name] = (m.launches - l0) / args.iters
        host_ms.clear()
        t = time_calls({"a_first_frame_mapping": arm_a, "b_host_loop": arm_b}, args.reps, args.warmup)
        host_ms = host_ms[args.warmup:]
        out = {}
        for k, v in t.items():
            ms = median(v)
            out[k] = {"ms_per_call_median": ms, "ms_min": min(v), "ms_max": max(v), "ms_per_iteration": ms / args.iters,
                      "launches_per_iteration": counts[k]}
        out["b_host_loop"]["host_syncs_per_iteration"] = 1
        out["b_host_loop"]["h2d_copies_per_iteration"] = 1
        out["a_first_frame_mapping"]["host_enqueue_ms_per_iteration"] = median(host_ms) / args.iters
        out["a_first_frame_mapping"]["device_ms_per_iteration"] = out["a_first_frame_mapping"]["ms_per_iteration"]
        out["speedup"] = out["b_host_loop"]["ms_per_call_median"] / out["a_first_frame_mapping"]["ms_per_call_median"]
        res[label] = dict(rays=R, samples=nsd + nrd, **out)
        del m_a, m_b
        torch.cuda.empty_cache()
    # ---- BA arm: C3 with the current frame drawn every iteration vs fixed rows
    n_kf, Rb, n_cur, iters = 50, 4096, 512, 15
    pix = Rb - n_cur
    cfg = H.make_config(19, n_samples_d=32, n_range_d=11)
    cfg["sampling"] = {"kf_n_rays_h": 150, "kf_n_rays_w": 200}
    st, poses = build_store(cfg, n_kf, dev)
    poses_d = poses.to(dev)
    related = list(range(n_kf))
    state = H.state_of(H.oracle_field(cfg, grid_scale=0.3))
    m_f, m_r = FusedMapper(H.cuda_model(cfg, state)), FusedMapper(H.cuda_model(cfg, state))
    cur = st.rays[n_kf - 1, ::58][:n_cur].contiguous()
    hp = dict(n_iters=iters, pose_accum_step=5, lr_rot=1e-3, lr_trans=1e-3, optim_cur=True)
    seeds = iter(range(10 ** 6))
    fns = {"cur_frame": lambda: m_f.local_ba(st, 0, related, poses_d, pix, cur_frame=frame_d, n_cur=n_cur, seed=3 * iters * next(seeds), **hp),
           "cur_rays7": lambda: m_r.local_ba(st, 0, related, poses_d, pix, cur_rays7=cur, seed=3 * iters * next(seeds), **hp)}
    counts = {}
    for k, m in (("cur_frame", m_f), ("cur_rays7", m_r)):
        l0 = m.launches
        fns[k]()
        counts[k] = (m.launches - l0) / iters
    t = time_calls(fns, args.ba_reps, 2)
    ba = {k: {"ms_per_call_median": median(v), "ms_min": min(v), "ms_max": max(v), "launches_per_iteration": counts[k]} for k, v in t.items()}
    ba["draw_cost_ms_per_iteration"] = (ba["cur_frame"]["ms_per_call_median"] - ba["cur_rays7"]["ms_per_call_median"]) / iters
    res["ba_c3_cur_frame"] = dict(keyframes=n_kf, rays=Rb, n_cur=n_cur, iterations=iters, samples=43, **ba)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
