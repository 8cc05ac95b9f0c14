"""Local bundle adjustment at the C3 shape (BASELINE configs[2]): 50 keyframes of 640 x 480 stored as 150 x 200 rays each,
4096 rays per rank and iteration (3584 drawn from the store on the device + 512 current-frame rays, the split of bench.py's
store arm), 15 iterations with a pose step every 5, at S = 43 (the BASELINE map shape) and S = 75 (the reference's).

Arms, timed with CUDA events after a warm-up, alternated call by call:
  (a) FusedMapper.local_ba: the whole loop on the device, pose steps included;
  (b) the same 15 iterations of step_from_store without the pose leg (a - b = the cost of the pose optimisation);
  (d) the same 15 iterations of step_from_store(pose_grad=True): the ray-gradient backward without local_ba's pose steps
      (a - d = what local_ba adds around it);
  (c) the route local_ba replaces: step_host(pose_grad=True) on a host batch every iteration (one synchronisation each),
      poses_all.backward(d_poses) through qt_to_transform_matrix and torch.optim.Adam on the poses every 5 iterations.
Under ``torch.distributed.run --nproc_per_node G`` every rank runs (a) on its own 4096 rays (weak scaling) and rank 0 prints.
Prints one JSON line (GPU name and power limit read in the same run); ``--out`` also writes it to a file.
The keyframe contents are rendered at the stored ray lattice only (synth.render_frame on the 150 x 200 directions): the
store holds exactly what add_keyframe would keep of a full frame, without rendering the other 277,200 pixels."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import torch  # noqa: E402


def gpu_info(index):
    try:
        q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"gpu": torch.cuda.get_device_name(index), "nvidia_smi": q}


def build_store(cfg, n_kf, dev):
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    dirs = synth.camera_rays()
    st = mf.KeyframeRayStore(cfg, dirs.shape[0], dirs.shape[1], n_kf, dev)
    rows, cols = st.row_indices.cpu(), st.col_indices.cpu()
    lat = dirs[rows, cols].reshape(st.n_rays_h, st.n_rays_w, 3).contiguous()
    traj = synth.trajectory(n_kf + 1)
    for k in range(n_kf):
        st.rays[k].copy_(synth.frame_rays(synth.render_frame(traj[k], lat, seed=k)))
        st.frame_ids.append(k)
    return st, traj.to(torch.float32).contiguous()


def time_calls(fns, reps, warmup):
    """fns: name -> callable; alternated call by call; -> name -> list of ms."""
    for _ in range(warmup):
        for f in fns.values():
            f()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            out[k].append(a.elapsed_time(b))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", default="43,75")
    ap.add_argument("--iters", type=int, default=15)
    ap.add_argument("--accum", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ba.py needs a GPU")
    import helpers as H
    from mipsfusion_b200.mapper import FusedMapper
    from oracle.tracking import qt_to_transform_matrix
    from oracle.shims.pytorch3d.transforms import matrix_to_quaternion
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    group = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
        group = dist.group.WORLD
    dev = torch.device("cuda", torch.cuda.current_device())
    n_kf, R, n_cur = 50, 4096, 512
    pix = R - n_cur
    related = list(range(n_kf))
    res = dict(workload="local_ba C3: %d keyframes (150 x 200 rays each), K = %d poses, %d rays per rank (%d store draws + %d "
                        "current-frame rays), %d iterations, pose step every %d" % (n_kf, n_kf + 1, R, pix, n_cur, args.iters, args.accum),
               world=world, **gpu_info(dev.index))
    for S in [int(s) for s in args.samples.split(",")]:
        nsd, nrd = {43: (32, 11), 75: (50, 25)}[S]
        cfg = H.make_config(19, n_samples_d=nsd, n_range_d=nrd)
        cfg["sampling"] = {"kf_n_rays_h": 150, "kf_n_rays_w": 200}
        st, poses = build_store(cfg, n_kf, dev)
        poses_d = poses.to(dev)
        cur = st.rays[n_kf - 1, ::58][:n_cur].contiguous()
        state = H.state_of(H.oracle_field(cfg, grid_scale=0.3))
        hp = dict(n_iters=args.iters, pose_accum_step=args.accum, lr_rot=1e-3, lr_trans=1e-3, optim_cur=True)
        m_a = FusedMapper(H.cuda_model(cfg, state), group=group)
        seeds = iter(range(10 ** 6))
        fns = {"a_local_ba": lambda: m_a.local_ba(st, 0, related, poses_d, pix, cur_rays7=cur, seed=3 * args.iters * world * next(seeds), **hp)}
        if world == 1:
            m_b = FusedMapper(H.cuda_model(cfg, state))
            m_c = FusedMapper(H.cuda_model(cfg, state))

            def arm_b():
                for _ in range(args.iters):
                    m_b.step_from_store(st, 0, related, poses_d, pix, cur_rays7=cur)
            # (c): host batches drawn beforehand (outside the timed window), the reference's host-side pose parametrisation
            batches = []
            for i in range(args.iters):
                rays, _, kidx = st.sample_rays_in_submap(0, related, pix, seed=7 + 3 * i)
                batches.append((torch.cat([rays, cur]).cpu().pin_memory(),
                                torch.cat([kidx, torch.full((n_cur,), -1, device=dev, dtype=torch.int64)]).cpu().pin_memory()))

            def arm_c():
                rot = torch.nn.Parameter(matrix_to_quaternion(poses_d[1:, :3, :3]).clone())
                trans = torch.nn.Parameter(poses_d[1:, :3, 3].clone())
                opt = torch.optim.Adam([{"params": rot, "lr": 1e-3}, {"params": trans, "lr": 1e-3}])
                P = torch.cat([poses_d[:1], qt_to_transform_matrix(rot, trans)])
                for i in range(args.iters):
                    _, d_poses = m_c.step_host(batches[i][0], batches[i][1], P.detach(), pose_grad=True)
                    P.backward(d_poses, retain_graph=True)
                    if (i + 1) % args.accum == 0:
                        opt.step(); opt.zero_grad()
                        P = torch.cat([poses_d[:1], qt_to_transform_matrix(rot, trans)])
            m_d = FusedMapper(H.cuda_model(cfg, state))

            def arm_d():
                for _ in range(args.iters):
                    m_d.step_from_store(st, 0, related, poses_d, pix, cur_rays7=cur, pose_grad=True)
            fns["b_store_no_poses"] = arm_b
            fns["d_store_pose_grads_no_pose_step"] = arm_d
            fns["c_host_pose_route"] = arm_c
        launches0 = m_a.launches
        m_a.local_ba(st, 0, related, poses_d, pix, cur_rays7=cur, seed=11, **hp)
        launches_per_iter = (m_a.launches - launches0) / args.iters
        t = time_calls(fns, args.reps, args.warmup)
        out = {}
        for k, v in t.items():
            ms = sorted(v)[len(v) // 2]
            out[k] = {"ms_per_call_median": ms, "ms_min": min(v), "ms_max": max(v),
                      "rays_per_s": R * world * args.iters / (ms * 1e-3)}
        if world > 1:
            import torch.distributed as dist
            mx = torch.tensor([out["a_local_ba"]["ms_per_call_median"]], device=dev)
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            out["a_local_ba"]["ms_per_call_median_slowest_rank"] = float(mx)
        else:
            out["pose_leg_overhead_pct"] = 100.0 * (out["a_local_ba"]["ms_per_call_median"] / out["b_store_no_poses"]["ms_per_call_median"] - 1)
            out["speedup_vs_host_pose_route"] = out["c_host_pose_route"]["ms_per_call_median"] / out["a_local_ba"]["ms_per_call_median"]
        out["local_ba_launches_per_iteration"] = launches_per_iter
        res["S%d" % S] = out
        del st
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
