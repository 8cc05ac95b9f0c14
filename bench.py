#!/usr/bin/env python
"""Benchmark of the MIPSFusion per-frame neural-field hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Headline metric (BASELINE.json): map-step rays/s -- one mapping iteration = z-sampling, fused
encode+MLP forward, SDF->weight render + losses, full backward, dense Adam -- on the BASELINE shape
4096 rays x 43 samples, T = 2^19 hash grid, synthetic SDF-room frame.  The same JSON line also carries
the tracking metric (pose candidates/s at 1024 x 2048) under "also".

--dump-outputs DIR: after the K timed steps, writes what the last of them computed as DIR/<name>.npy (float32, see
dump_outputs).  The inputs, the initial model and the device draws of the step are seeded, so two builds run with the same
arguments can be compared output for output.

N > 1 (torchrun): data-parallel mapping, one 4096-ray batch per rank (weak scaling), global mask counts
all-reduced before the loss and gradients all-reduced before Adam (NCCL).
--impl reference: the CPU implementation of the same step (the oracle port of the reference's PyTorch
path; the reference checkout itself does not travel to the GPU box) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

R_RAYS, N_SAMPLES_D, N_RANGE_D, HASH = 4096, 32, 11, 19
S = N_SAMPLES_D + N_RANGE_D
ALG_BYTES_PER_POINT = 1024              # SURVEY 8d: 16 levels x 8 corners x 2 features x 4 B gathered (forward) / scattered (backward)
ADAM_BYTES_PER_PARAM = 32
DTYPE = "f32 (decoder contractions as bf16x3 hi/lo splits on tcgen05, fp32 accumulate; encodings, render, losses, Adam in fp32)"


def ncu_traffic():
    """DRAM bytes per launch from the committed ncu --set full capture (kernel name -> bytes), {} if none is committed."""
    p = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def pause(self):
        """Stops polling (the rows collected so far are kept); start() resumes."""
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.t.join(timeout=1.0)
            except Exception:
                pass
            self.proc = None
            self.started = True

    def stop(self):
        if self.proc is None and not getattr(self, "started", False):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(parts[0])); mx = float(parts[1])
            except Exception:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_inputs(seed):
    import helpers as H
    return H.synth_batch(R_RAYS, S, seed=seed, invalid=64)


def build_model(seed=0):
    import helpers as H
    cfg = H.make_config(HASH, n_samples_d=N_SAMPLES_D, n_range_d=N_RANGE_D)
    of = H.oracle_field(cfg, seed=seed)            # same init as the CPU arm: grid U(-1e-4,1e-4) seed 1337, nn.Linear default
    return cfg, of


# ------------------------------------------------------------------------------------------------
def cpu_step_fn(n_rays, threads=None):
    """The CPU arm: oracle port of JointEncoding.forward + loss.backward() + torch.optim.Adam.step()."""
    import torch
    from oracle import adam as oadam
    torch.set_num_threads(threads or os.cpu_count())
    cfg, of = build_model()
    opt = oadam.make_optimizer(of)
    rays_o, rays_d, rgb, d, u = make_inputs(0)
    sl = slice(0, n_rays)
    args = (rays_o[sl], rays_d[sl], rgb[sl], d[sl], u[sl])

    def step():
        opt.zero_grad()
        ret = of.forward(*args)
        loss = of.total_loss(ret)
        loss.backward()
        opt.step()
        return float(loss)
    return step


def run_reference(args):
    """`--impl reference`: CPU implementation on the host cores, bounded sample per step."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_rays = R_RAYS                    # the full 4096-ray batch of the GPU arm (about 0.5 s per step on 16 host threads)
    step = cpu_step_fn(n_rays)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = n_rays * args.steps / dt
    cores = torch.get_num_threads()
    sample = (f"{args.steps} steps x {n_rays} rays x {S} samples (the full batch of the GPU arm), full T=2^19 grid + dense Adam, "
              f"oracle port of the reference's PyTorch path on the host cores, torch {torch.__version__}")
    emit(({
        "impl": "reference", "metric": "map_step_rays_per_s", "value": val, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(n):
    return {"workload": f"C1 mapping step: {R_RAYS} rays x {S} samples ({N_SAMPLES_D} uniform + {N_RANGE_D} around depth) per GPU, "
                        f"HashGrid T=2^{HASH} (9,014,144 params) + MLP_reg (36,577), forward + backward + dense Adam, one synthetic "
                        "SDF-room 640x480 frame (BASELINE.json configs[0] shape; configs[1] tracking shape reported under 'also')",
            "rays_per_gpu": R_RAYS, "samples_per_ray": S, "hash_size": HASH, "parallelism": f"dp{n}" if n > 1 else "single",
            "l2": "per-step working set (grid p,g,m,v = 144 MB) exceeds the 126 MB L2; L2 additionally flushed (256 MB write) between timed steps"}


# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import helpers as H
    import mipsfusion_b200 as mf
    from mipsfusion_b200.mapper import FusedMapper

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"           # keep NCCL's version banner off the JSON stream
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    cfg, of = build_model()
    model = H.cuda_model(cfg, H.state_of(of))
    rays_o, rays_d, rgb, d, _ = make_inputs(rank)
    host = torch.cat([rays_o, rays_d, rgb, d], -1).contiguous().pin_memory()        # (R, 10) pinned host batch
    dv = host.to(dev)
    ro, rd, tc, td = dv[:, 0:3].contiguous(), dv[:, 3:6].contiguous(), dv[:, 6:9].contiguous(), dv[:, 9].contiguous()
    mapper = FusedMapper(model, group=group)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        mapper.step(ro, rd, tc, td)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- timed region: exactly K steps, device time per step (events), L2 flushed between steps ----
    mapper.launches = 0
    evs = []
    barrier()
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        losses = mapper.step(ro, rd, tc, td)
        b.record()
        evs.append((a, b))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    launches = mapper.launches
    t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t)
    value = world * R_RAYS * args.steps / (dev_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        sampler.pause()                 # (the copy and the file writes leave the GPU idle: kept out of the clock samples)
        dump_outputs(args.dump_outputs, mapper, losses)
        sampler.start()

    if args.quick:                    # profiling runs (ncu): only the timed steps above
        if rank == 0:
            emit({"metric": "map_step_rays_per_s", "value": value, "ms_per_step": dev_ms / args.steps, "quick": True})
        return
    # ---- per-kernel timing of the dominant kernel (separate pass, events around each launch) ----
    import ctypes as C
    from mipsfusion_b200 import _lib as L
    mapper.timing = {}
    kernel_acc = {"field_fwd": [], "field_bwd": []}
    L.call("mf_debug_kernel_timer", 1)
    for _ in range(args.steps):
        flush.zero_()
        mapper.step(ro, rd, tc, td)
        for slot, name in ((0, "field_fwd"), (1, "field_bwd")):
            ms = C.c_float(0.0)
            L.call("mf_debug_kernel_ms", slot, C.byref(ms))
            kernel_acc[name].append(ms.value)
    torch.cuda.synchronize()
    L.call("mf_debug_kernel_timer", 0)
    phase_ms = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in mapper.timing.items()}
    kernel_ms = {k: sum(v) / len(v) for k, v in kernel_acc.items()}
    mapper.timing = None

    # ---- e2e: public API with HOST buffers; every step copies the pinned host batch H2D and reads the loss back ----
    # (a) the drop-in route through the reference's UNCHANGED call surface (north_star): JointEncoding.forward +
    #     loss.backward() + the optimiser's step, exactly the body of the reference's mapping loop (mipsfusion.py:316-335)
    #     -- the headline e2e;
    # (b) FusedMapper.step_host: the one-call replacement of that loop body (INTEGRATION.md section 1), reported under also.
    def timed_e2e(fn):
        for _ in range(10):                                  # (allocator / lazy-initialisation warm-up of the host path)
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        barrier()
        te = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return world * R_RAYS * args.steps / float(te)

    rays7, pose_idx, poses_h, _ = H.synth_batch_packed(R_RAYS, seed=rank, invalid=64)
    rays7, pose_idx, poses_d = rays7.pin_memory(), pose_idx.pin_memory(), poses_h.to(dev)
    e2e_val = timed_e2e(lambda: mapper.step_host(rays7, pose_idx, poses_d))
    h2d_bytes, d2h_bytes = rays7.numel() * 4 + pose_idx.numel() * 8, 8 * 4

    # (the clock / throttle sampler has covered the device-timed regions and the GPU-bound loop above; it pauses here because the
    # nvidia-smi poll takes the driver lock every 50 ms, which the HOST-bound drop-in loop below would feel, and resumes for the
    # GPU-bound tracking / frame / joint-query measurements)
    if rank == 0:
        sampler.pause()
    model2 = H.cuda_model(cfg, H.state_of(of))
    opt = mf.create_map_optimizer(model2, cfg["mapping"]["lr_decoder"], cfg["mapping"]["lr_embed"])
    tw = cfg["training"]

    def autograd_step():
        batch = host.to(dev, non_blocking=True)
        ret = model2(batch[:, 0:3], batch[:, 3:6], batch[:, 6:9], batch[:, 9:10])
        loss = tw["rgb_weight"] * ret["rgb_loss"] + tw["sdf_weight"] * ret["sdf_loss"] + tw["fs_weight"] * ret["fs_loss"]
        loss.backward()
        if world > 1:
            import torch.distributed as dist
            # (the decoder's ten gradients are views of one flat buffer: two all-reduces instead of eleven)
            fg = model2.decoder.__dict__.get("_flat_grad")
            gl = [model2.embed_fn.params.grad] + ([fg] if fg is not None else [p.grad for p in model2.decoder.parameters()])
            for g_ in gl:
                if g_ is not None:
                    dist.all_reduce(g_); g_.mul_(1.0 / world)
        opt.step(zero_grad=True)
        return float(loss.detach())                          # D2H read of the step's result
    e2e_autograd = timed_e2e(autograd_step)
    del model2, opt
    if rank == 0:
        sampler.start()


    # ---- tracking metric (BASELINE configs[1] shape): RandomOptimizer scoring 1024 candidates x 2048 pixels ----
    also = {"e2e_fused_step_host_rays_per_s": e2e_val,
            "e2e_fused_step_host": "FusedMapper.step_host(rays7 (R,7) pinned host batch, pose_idx, poses) -> ray generation + map step "
                                   "-> 8 loss terms on the host: the one-call replacement of the reference's loop body (%d B H2D, %d B D2H per step)"
                                   % (h2d_bytes, d2h_bytes)}
    if world > 1:                      # the two other sharded paths, strong scaling on the single-GPU shapes
        also.update(tracking_bench(model, cfg, dev, group=group))
        also.update(joint_query_bench(dev, group=group))
        also.update(joint_query_bench(dev, group=group, shard="submaps", prefix="joint_query_submap_sharded"))
        also.update(submap_parallel_bench(dev, group))
    if world == 1:
        also.update(tracking_bench(model, cfg, dev))
        also.update(frame_bench(dev))
        also.update(joint_query_bench(dev))
        also.update(store_bench(mapper, dev, args.steps))
        also.update(render_full_bench(dev))
        also.update(marching_cubes_bench(dev))
        also.update(mesh_pipeline_bench(dev))
    clocks = sampler.stop() if rank == 0 else None          # (before the CPU baselines: only GPU-loaded intervals are sampled)
    also_roof = {k[len("_roof_"):]: also.pop(k) for k in [k for k in also if k.startswith("_roof_")]}
    also_roof = {k: v for k, v in also_roof.items() if v}

    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return
    hbm, tf, which = peaks()
    P = R_RAYS * S
    n_params = 9014144 + 36577
    # ---- roofline (SURVEY 8d): algorithmic bytes / launch of the dominant kernel over its own CUDA-event duration ----
    # field backward: 1,024 B of scatter per point x ALL points of the launch (the kernel only visits the points whose
    # upstream gradient row is non-zero, the algorithmic count is the work the reference's autograd does); duration = the
    # event pair the library records around the kernel launch itself (mf_debug_kernel_timer), not the phase around it
    bwd_ms = kernel_ms.get("field_bwd", float("nan"))
    fwd_ms = kernel_ms.get("field_fwd", float("nan"))
    d_raw = mapper._bufs[(R_RAYS, S)]["d_raw"]
    n_active = int((d_raw.view(-1, d_raw.shape[-1]) != 0).any(-1).sum())
    alg_bytes = ALG_BYTES_PER_POINT * P
    achieved = alg_bytes / (bwd_ms * 1e-3) / 1e9
    step_ms = dev_ms / args.steps
    step_bytes = 2 * ALG_BYTES_PER_POINT * P + ADAM_BYTES_PER_PARAM * n_params + (28 + 4 * S + 44) * R_RAYS     # 651.3 MB
    traffic = ncu_traffic()
    roof = {"bound": "hbm", "kernel": "field_bwd_tc2_kernel (role-split tcgen05 backward: recompute-forward + dgrad chain | wgrad read-out | grid scatter)",
            "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
            "traffic": traffic.get("field_bwd_tc2_kernel"), "traffic_unit": "bytes/launch (dram__bytes_read.sum + dram__bytes_write.sum, "
            "ncu --set full, profiles/r2_ncu_traffic.json)", "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)",
            "ms_per_launch": bwd_ms, "alg_bytes_per_launch": alg_bytes, "alg_bytes_per_point": ALG_BYTES_PER_POINT,
            "points_per_launch": P, "active_points_per_launch": n_active,
            "step": {"alg_bytes": step_bytes, "ms": step_ms, "achieved": step_bytes / (step_ms * 1e-3) / 1e9,
                     "frac": step_bytes / (step_ms * 1e-3) / 1e9 / hbm,
                     "what": "2,048 B x points (gather + scatter) + 32 B x parameters (Adam) + ray I/O over the whole map step"},
            "kernels": {
                "field_fwd_tc3_kernel": {"alg_bytes": ALG_BYTES_PER_POINT * P, "ms": fwd_ms,
                                         "achieved": ALG_BYTES_PER_POINT * P / (fwd_ms * 1e-3) / 1e9,
                                         "frac": ALG_BYTES_PER_POINT * P / (fwd_ms * 1e-3) / 1e9 / hbm,
                                         "traffic": traffic.get("field_fwd_tc3_kernel")},
                "adam_pair_kernel": {"alg_bytes": ADAM_BYTES_PER_PARAM * n_params, "ms": phase_ms.get("adam"),
                                     "achieved": ADAM_BYTES_PER_PARAM * n_params / (phase_ms.get("adam", float("nan")) * 1e-3) / 1e9,
                                     "frac": ADAM_BYTES_PER_PARAM * n_params / (phase_ms.get("adam", float("nan")) * 1e-3) / 1e9 / hbm,
                                     "note": "phase = Adam (grid + decoder, one launch) + weight re-layout",
                                     "traffic": traffic.get("adam_pair_kernel")}},
            "phase_ms": phase_ms}
    for k in ("ro_field_query", "joint_query", "render_full_img", "marching_cubes"):
        if k in also_roof:
            also_roof[k]["frac"] = also_roof[k]["achieved"] / hbm
            roof["kernels"][k] = also_roof[k]
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        n_rays, steps = R_RAYS, 3
        step = cpu_step_fn(n_rays)
        step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
        cpu = {"value": n_rays * steps / dt, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"{steps} steps x {n_rays} rays x {S} samples (the full batch), full T=2^19 grid + dense Adam, "
                         f"oracle port of the reference's PyTorch path, torch {torch.__version__}"}
        # the other metrics of BASELINE.json beside their GPU numbers (BASELINE.md section 3): tracking, ms/frame, joint query
        cpu["also"] = cpu_also_baselines(cfg, also)
    out = {"metric": "map_step_rays_per_s", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": workload_config(world),
           "roofline": roof, "cpu_baseline": cpu,
           "e2e": {"value": e2e_autograd, "unit": "rays/s", "h2d_bytes_per_step": host.numel() * 4, "d2h_bytes_per_step": 4,
                   "api": "the reference's unchanged call surface: pinned host batch (R,10) -> .to(device) -> JointEncoding.forward(rays_o, rays_d, "
                          "rgb, depth) -> weighted loss -> loss.backward() -> create_map_optimizer(...).step() -> float(loss) on the host"},
           "gpu_launches": launches, "clocks": clocks, "wall_s_timed_region": t_wall, "also": also}
    emit(out)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def dump_outputs(out_dir, mapper, losses):
    """Writes what the last timed map step computed, as float32 .npy files under out_dir (36 MB in all): the (8,) vector
    FusedMapper.step returns, the rendered colour and depth of every ray, and the model the step leaves behind: the whole hash
    grid (9,014,144 parameters) and the decoder's flat weights (36,577).
    The backward accumulates the grid and decoder gradients with atomics in no fixed order, and Adam turns those last-bit
    differences into whole steps wherever a gradient nearly cancels.  So two runs of one build do not agree bit for bit.
    profiles/r3_dump_spread.txt records the per-array differences between two such runs (GPU, power limit and command included;
    scripts/compare_dumps.py computes them).  They show the size of the spread from one pair of runs and are not a tolerance:
    compare two builds against repeated runs of one of them."""
    import numpy as np
    import torch
    b = mapper._bufs[(R_RAYS, S)]
    arrays = {"losses": losses, "rgb": b["rgb"], "depth": b["depth"], "grid_params": mapper.grid, "decoder_params": mapper.mlp}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to(torch.float32).cpu().numpy())


def _max_over_ranks(x, dev, group):
    import torch
    t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
    if group is not None:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t)


def tracking_bench(model, cfg, dev, iters=5, group=None):
    """pose candidates/s of RandomOptimizer scoring at the BASELINE tracking shape.  With a process group the SAME 1024
    candidates are sharded across the ranks (strong scaling; one all-gather of 9 floats per candidate per iteration)."""
    import types
    import torch
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    from mipsfusion_b200.sampling_helper import sample_pixels_uniformly        # (the product's own lattice kernel: the oracle stays in the CPU legs)
    Cn, nr, nc = 1024, 32, 64
    tcfg = dict(cfg)
    tcfg["tracking"] = {"RO": {"particle_size": Cn, "initial_scaling_factor": 0.02, "rescaling_factor": 0.5, "n_rows": nr, "n_cols": nc},
                        "ignore_edge_W": 20, "ignore_edge_H": 20}
    dirs = synth.camera_rays()
    c2w = synth.trajectory(4)[1]
    rows, cols = (t.cpu() for t in sample_pixels_uniformly(460, 620, nr, nc, device=dev))
    sub = synth.render_frame(c2w, dirs[rows, cols][None].contiguous())
    ds = types.SimpleNamespace(H=460, W=620, fx=320.0, fy=320.0, cx=309.5, cy=229.5, rays_d=dirs)
    g = torch.Generator().manual_seed(0)
    particles = torch.randn(Cn, 6, generator=g).clamp(-2, 2); particles[0] = 0
    ro = mf.RandomOptimizer(tcfg, types.SimpleNamespace(dataset=ds, device=str(dev)), particles=particles, group=group)
    model.eval()
    target_d = sub["depth"].reshape(-1).to(dev); rays_d = dirs[rows, cols].contiguous().to(dev)
    rot, trans = c2w[:3, :3].contiguous().to(dev), c2w[:3, 3].contiguous().to(dev)
    search = torch.full((6,), 0.02, device=dev)
    # the loop body of RandomOptimizer.optimize (score + swarm update, in place on copies of the pose state) on a fixed lattice
    rot_s, trans_s, search_s = rot.clone(), trans.clone(), search.clone()
    def body():
        ro.iterate(model, rot_s, trans_s, search_s, target_d, rays_d)
    for _ in range(2):
        body()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        body()
    b.record(); torch.cuda.synchronize()
    ms_it = _max_over_ranks(a.elapsed_time(b) / iters, dev, group)
    model.train()
    P_ = nr * nc
    ro_bytes = Cn * (P_ * (ALG_BYTES_PER_POINT + 12) + 28)          # SURVEY 8d: per candidate Pix x (1,024 B + 12 B) + 28 B
    roof = {"alg_bytes": ro_bytes, "ms": ms_it, "achieved": ro_bytes / (ms_it * 1e-3) / 1e9,
            "what": "one RandomOptimizer iteration (pose kernel + SDF-only field query + per-candidate reduction + swarm update) "
                    f"at {Cn} candidates x {P_} pixels; per candidate Pix x 1,036 B + 28 B"}
    return {"_roof_ro_field_query": roof,
            "tracking_pose_candidates_per_s": Cn / (ms_it * 1e-3), "tracking_ms_per_ro_iteration": ms_it,
            "tracking_shape": f"{Cn} candidates x {nr * nc} pixels, SDF-only field query + per-candidate reduction + swarm update"
                              + ("" if group is None else "; the candidates are sharded across the GPUs (strong scaling)")}


def cpu_also_baselines(cfg, also):
    """CPU (oracle port, all host threads) numbers for the metrics reported under `also`, each on a bounded sample:
    one RandomOptimizer iteration at 256 of the 1024 candidates x 2048 pixels; the reference's per-frame work at its shipped
    sizes (RO 5 x 2000 x 384, 10 pose-refinement iterations x 1000 rays x 75, 15 mapping iterations x 2600 x 75 every 3rd
    frame), each component timed once; the joint query on a 128^3 sub-grid x 16 submaps (x 64 = 512^3)."""
    import types
    import numpy as np
    import torch
    import helpers as H
    from mipsfusion_b200 import synth
    from oracle import ro as oro, sampling as osamp, joint_query as ojq, adam as oadam
    out = {"cores": torch.get_num_threads(), "kind": "port"}
    dirs = synth.camera_rays()
    c2w = synth.trajectory(4)[1]
    # ---- C2: RandomOptimizer iteration ----
    _, of = build_model()
    Cn, nr, nc, sub = 1024, 32, 64, 256
    rows, cols = osamp.sample_pixels_uniformly(460, 620, nr, nc)
    fr = synth.render_frame(c2w, dirs[rows, cols][None].contiguous())
    g = torch.Generator().manual_seed(0)
    particles = torch.randn(Cn, 6, generator=g).clamp(-2, 2); particles[0] = 0
    td, rdc = fr["depth"].reshape(-1, 1), dirs[rows, cols].contiguous()
    with torch.no_grad():
        t0 = time.perf_counter()
        oro.ro_iteration(of, c2w[:3, :3], c2w[:3, 3:], 0.02, particles[:sub], td, rdc, cfg["training"]["trunc"])
        dt = time.perf_counter() - t0
    out["tracking_pose_candidates_per_s"] = sub / dt
    out["tracking_sample"] = f"1 RandomOptimizer iteration, {sub} of the {Cn} candidates x {nr * nc} pixels"
    if "tracking_pose_candidates_per_s" in also:
        out["tracking_gpu_over_cpu"] = also["tracking_pose_candidates_per_s"] / out["tracking_pose_candidates_per_s"]
    # ---- ms / frame at the reference's shipped sizes ----
    fcfg = H.make_config(HASH, n_samples_d=50, n_range_d=25)
    off = H.oracle_field(fcfg)
    frame = synth.render_frame(c2w, dirs)
    rows, cols = osamp.sample_pixels_uniformly(460, 620, 16, 24)
    g = torch.Generator().manual_seed(1)
    p2000 = torch.randn(2000, 6, generator=g).clamp(-2, 2); p2000[0] = 0
    td, rdc = frame["depth"][rows, cols].reshape(-1, 1), dirs[rows, cols].contiguous()
    with torch.no_grad():
        t0 = time.perf_counter()
        oro.ro_iteration(off, c2w[:3, :3], c2w[:3, 3:], 0.02, p2000, td, rdc, fcfg["training"]["trunc"])
        t_ro = (time.perf_counter() - t0) * 5                        # 5 RO iterations per frame
    idx = torch.randint(0, 460 * 620, (1000,), generator=g)
    r_, c_ = idx // 620, idx % 620
    d_cam, t_rgb, t_d = dirs[r_, c_], frame["rgb"][r_, c_], frame["depth"][r_, c_].unsqueeze(-1)
    trans = c2w[:3, 3].clone().requires_grad_(True); rot = c2w[:3, :3].clone().requires_grad_(True)
    popt = torch.optim.Adam([rot, trans], lr=1e-3)
    u = torch.rand(1000, 75, generator=g)
    t0 = time.perf_counter()
    for _ in range(2):                                               # 2 of the 10 pose-refinement iterations
        popt.zero_grad()
        ret = off.forward(trans[None, :].repeat(1000, 1), torch.sum(d_cam[..., None, :] * rot[None], -1), t_rgb, t_d, u, EMD_w=0.0)
        off.total_loss(ret).backward()
        popt.step()
    t_go = (time.perf_counter() - t0) * 5
    for q in off.parameters():
        q.grad = None
    mopt = oadam.make_optimizer(off)
    idx = torch.randint(0, 460 * 620, (2600,), generator=g)
    r_, c_ = idx // 620, idx % 620
    ro_ = c2w[None, :3, 3].repeat(2600, 1); rd_ = torch.sum(dirs[r_, c_][..., None, :] * c2w[None, :3, :3], -1)
    u = torch.rand(2600, 75, generator=g)
    t0 = time.perf_counter()
    for _ in range(2):                                               # 2 of the 15 mapping iterations
        mopt.zero_grad()
        off.total_loss(off.forward(ro_, rd_, frame["rgb"][r_, c_], frame["depth"][r_, c_].unsqueeze(-1), u)).backward()
        mopt.step()
    t_map = (time.perf_counter() - t0) * 7.5
    out["ms_per_frame_640x480"] = 1e3 * (t_ro + t_go + t_map / 3.0)
    out["frame_sample"] = ("RO: 1 of 5 iterations (2000 x 384) x 5; pose refinement: 2 of 10 iterations (1000 rays x 75) x 5; mapping: "
                           "2 of 15 iterations (2600 rays x 75) x 7.5, every 3rd frame; components "
                           f"{1e3 * t_ro:.0f} + {1e3 * t_go:.0f} + {1e3 * t_map:.0f}/3 ms")
    if "ms_per_frame_640x480" in also:
        out["frame_cpu_over_gpu"] = out["ms_per_frame_640x480"] / also["ms_per_frame_640x480"]
    # ---- C5: joint query, 128^3 sub-grid x 16 submaps (scaled x 64 to 512^3) ----
    jcfg = H.make_config(HASH)
    jcfg["grid"]["use_bound_normalize"] = False
    jf = H.oracle_field(jcfg)
    lo, hi = np.array([-0.6, 0.5, -1.15]), np.array([2.95, 7.05, 3.05])
    ext = hi - lo
    poses, amin, amax, cents = [], [], [], []
    for m in range(16):
        ix, iy = m % 4, m // 4
        a = lo + ext * np.array([ix / 4.0 - 0.08, iy / 4.0 - 0.08, 0.0])
        b = lo + ext * np.array([(ix + 1) / 4.0 + 0.08, (iy + 1) / 4.0 + 0.08, 1.0])
        T = torch.eye(4); T[:3, 3] = torch.tensor((a + b) / 2, dtype=torch.float32)
        poses.append(T); amin.append(a); amax.append(b); cents.append(((a + b) / 2).astype(np.float32))
    axes = [np.linspace(lo[k], hi[k], 128) for k in range(3)]
    xx, yy, zz = np.meshgrid(*axes)
    pts = np.vstack([xx.ravel(), yy.ravel(), zz.ravel()]).T.astype(np.float32)
    t0 = time.perf_counter()
    ojq.joint_query(pts, [jf] * 16, poses, amin, amax, cents)
    dt = time.perf_counter() - t0
    out["joint_query_grid_points_per_s"] = pts.shape[0] / dt
    out["joint_query_sample"] = "128^3 grid over the same volume x 16 submaps (1/64 of the 512^3 points; same submaps-per-point ratio)"
    if "joint_query_grid_points_per_s" in also:
        out["joint_query_gpu_over_cpu"] = also["joint_query_grid_points_per_s"] / out["joint_query_grid_points_per_s"]
    # ---- N2: marching cubes (the reference's NumpyMarchingCubes restated in C++, one thread -- the reference routine is serial) ----
    from oracle import marching_cubes as omc
    sub = mc_volume(512, "cpu")[192:320, 192:320, 192:320].contiguous().numpy()
    t0 = time.perf_counter()
    _, f = omc.marching_cubes(sub, 0.0, 3.0)
    dt = time.perf_counter() - t0
    out["marching_cubes_voxels_per_s"] = sub.size / dt
    out["marching_cubes_sample"] = (f"128^3 centre block of the 512^3 volume ({f.shape[0]} faces), 1 thread (the reference routine is serial); "
                                    "oracle/_ref (the reference's own sources) runs the same block 2-5x slower than this restatement")
    if "marching_cubes_voxels_per_s" in also:
        out["marching_cubes_gpu_over_cpu"] = also["marching_cubes_voxels_per_s"] / out["marching_cubes_voxels_per_s"]
    return out


def mc_volume(n, dev):
    """Room-like SDF on an n^3 grid (two walls, a floor, a ball), tanh-compressed like the decoder's output in (-1, 1)."""
    import torch
    ax = torch.linspace(0, 1, n, device=dev)
    X, Y, Z = ax[:, None, None], ax[None, :, None], ax[None, None, :]
    d = torch.minimum(torch.minimum(X - 0.12, 0.9 - Y),
                      torch.minimum(Z - 0.2, torch.sqrt((X - 0.55) ** 2 + (Y - 0.55) ** 2 + (Z - 0.55) ** 2) - 0.17))
    return torch.tanh(d * 12.0).contiguous()


def mesh_pipeline_bench(dev, res=512, n_submaps=16):
    """C5 end to end on the device: blended SDF over 512^3 x 16 submaps -> marching cubes -> blended vertex colours
    (JointSubmapQuery.extract_mesh = Mesher.extract_mesh_jointly steps 4, 5 and 9).  The decoders are randomly initialised (no
    checkpoints offline), so the surface is whatever level set the random field has; the work per grid point is the real one."""
    import torch
    jq, axes, _, _ = joint_query_setup(dev, res, n_submaps)
    small = [a_[:96] for a_ in axes]
    jq.extract_mesh(small)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = jq.extract_mesh(axes)                                   # allocations of the full-size buffers
    del out
    a.record()
    out = jq.extract_mesh(axes)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    return {"mesh_pipeline_ms": ms, "mesh_pipeline_grid_points_per_s": res ** 3 / (ms * 1e-3),
            "mesh_pipeline": f"{res}^3 grid x {n_submaps} submaps -> blended SDF -> marching cubes ({out['vertices'].shape[0]} vertices, "
                             f"{out['faces'].shape[0]} faces) -> blended vertex colours, device resident"}


def marching_cubes_bench(dev, n=512):
    """SURVEY 8f row N2: marching cubes over the 512^3 blended-SDF grid of C5 (utils/utils.py:78 -> NumpyMarchingCubes), device
    volume in, device mesh out; the two C-ABI calls and their host read-backs of the data-dependent sizes are inside the events."""
    import torch
    import mipsfusion_b200 as mf
    vol = mc_volume(n, dev)
    mf.marching_cubes_device(vol, 0.0, 3.0)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(3):
        v, f, info = mf.marching_cubes_device(vol, 0.0, 3.0, return_info=True)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 3
    alg = 4 * n ** 3 + 12 * v.shape[0] + 12 * f.shape[0]
    return {"marching_cubes_ms": ms, "marching_cubes_voxels_per_s": n ** 3 / (ms * 1e-3),
            "marching_cubes_mesh": f"{n}^3 volume -> {v.shape[0]} vertices, {f.shape[0]} faces ({info['soup_triangles']} triangles before "
                                   f"merging, {info['rounds']} clustering round(s)); bit-identical to the reference routine",
            "_roof_marching_cubes": {"alg_bytes": alg, "ms": ms, "achieved": alg / (ms * 1e-3) / 1e9,
                                     "what": "whole call (15 kernels + 3 scans + 2 host read-backs of data-dependent sizes): 4 B per voxel read once + 12 B per output vertex and face"}}


def render_full_bench(dev):
    """SURVEY 8f row N4: Logger.render_full_img (Logger.py:193-214) -- 620 x 460 rays x 75 samples in one forward launch; the
    large-batch benchmark of the forward field kernel (21.4 M points)."""
    import torch
    import helpers as H
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    cfg = H.make_config(HASH, n_samples_d=50, n_range_d=25)
    cfg["training"]["perturb"] = 0
    model = H.cuda_model(cfg, H.state_of(H.oracle_field(cfg)), train=False)
    dirs = synth.camera_rays()
    c2w = synth.trajectory(4)[1]
    frame = synth.render_frame(c2w, dirs)
    dirs_d, depth_d, pose_d = dirs.to(dev), frame["depth"].to(dev), c2w.to(dev)
    mf.render_full_img(model, dirs_d, pose_d, depth_d)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(3):
        rgb, depth = mf.render_full_img(model, dirs_d, pose_d, depth_d)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 3
    R, Sx = dirs.shape[0] * dirs.shape[1], 75
    return {"render_full_img_ms": ms, "render_full_img_rays_per_s": R / (ms * 1e-3),
            "_roof_render_full_img": {"alg_bytes": ALG_BYTES_PER_POINT * R * Sx, "ms": ms, "achieved": ALG_BYTES_PER_POINT * R * Sx / (ms * 1e-3) / 1e9,
                                      "what": f"{dirs.shape[1]} x {dirs.shape[0]} image, {R} rays x {Sx} samples: ray generation + z sampling + one forward "
                                              "field launch over 21.4 M points + SDF-to-weight render (no losses); 1,024 B per point"},
            "render_full_img_shape": f"{dirs.shape[1]}x{dirs.shape[0]} image (640x480 cropped by 10), {Sx} samples per ray, one launch"}


def submap_parallel_bench(dev, group):
    """BASELINE configs[3] (C4) pieces on G GPUs: 16 submaps placed round robin (2 per GPU at G = 8).
    (a) weight hand-off of one T=2^19 submap (36.2 MB) rank 0 -> rank 1 and as a broadcast (mipsfusion.py:607-653);
    (b) cross-rank overlap SDF difference with pose gradients, 768 rays (InactiveMap.py:128-192);
    (c) rank 0 tracks + maps the active submap (the frame of frame_bench) while every other rank runs the inactive-submap BA
        (InactiveMap.local_BA: 2600 rays x 75 samples per iteration) on its own submaps: rank-0 ms/frame and the BA iterations/s
        of the other ranks, running concurrently."""
    import torch
    import torch.distributed as dist
    import helpers as H
    from mipsfusion_b200.mapper import FusedMapper
    from mipsfusion_b200.submap_parallel import SubmapParallel
    sp = SubmapParallel(group)
    out = {}
    cfg = H.make_config(HASH, n_samples_d=50, n_range_d=25)
    of = H.oracle_field(cfg)
    local_ids = sp.local_ids(16)
    models = {m: H.cuda_model(cfg, H.state_of(of)) for m in local_ids[:2]}
    m0 = models[local_ids[0]]
    # (a) hand-off
    for dst, key in ((1, "submap_handoff_p2p"), (None, "submap_handoff_broadcast")):
        sp.handoff(m0, 0, dst)                                         # warm-up (NCCL channel set-up)
        torch.cuda.synchronize(); dist.barrier(group=group)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            nbytes = sp.handoff(m0, 0, dst)
        b.record(); torch.cuda.synchronize()
        ms = _max_over_ranks(a.elapsed_time(b) / 5, dev, group)
        out[key + "_ms"] = ms
        out[key + "_gbs"] = 36.2e6 * 1.004 / (ms * 1e-3) / 1e9
    # (b) cross-rank overlap query: submaps 0 and 1 (ranks 0 and 1), 768 rays
    g = torch.Generator().manual_seed(5)
    rays7 = H.synth_batch_packed(768, seed=3)[0].to(dev)
    pose = H.synth_batch_packed(4, seed=3)[2][0].to(dev)
    local = {m: models[m] for m in local_ids[:2] if m in (0, 1)}
    for mm in local.values():
        mm.eval()
    target_d, dirs = rays7[:, 6:7].contiguous(), rays7[:, :3].contiguous()
    mask = (target_d > 0).float()
    def ovl():
        f1 = torch.eye(4, device=dev).requires_grad_(True); f2 = torch.eye(4, device=dev).requires_grad_(True)
        loss = sp.overlap_sdf_difference(local, 0, 1, target_d, dirs, mask, pose, f1, f2, 0.1)
        if loss.requires_grad:
            loss.backward()
        return loss
    for _ in range(3):
        ovl()
    torch.cuda.synchronize(); dist.barrier(group=group)
    t0 = time.perf_counter()
    for _ in range(10):
        ovl()
    torch.cuda.synchronize()
    out["overlap_query_ms"] = _max_over_ranks((time.perf_counter() - t0) / 10 * 1e3, dev, group)
    out["overlap_query_shape"] = "768 rays, submaps 0 / 1 on ranks 0 / 1: two field queries + one 2 x 768-float all-reduce + pose gradients on each owner"
    for mm in local.values():
        mm.train()
    # (c) rank 0: frames; other ranks: inactive-submap BA, concurrently
    rank = sp.rank
    frames = 6
    torch.cuda.synchronize(); dist.barrier(group=group)
    if rank == 0:
        r = frame_bench(dev, frames=frames)
        ms_frame, ba_its = r["ms_per_frame_640x480"], 0.0
    else:
        mapper = FusedMapper(m0)
        ro, rd, rgb, d, _ = [t.to(dev).contiguous() for t in H.synth_batch(2600, 75, seed=10 + rank)]
        for _ in range(3):
            mapper.step(ro, rd, rgb, d.reshape(-1))
        torch.cuda.synchronize()
        t0 = time.perf_counter(); n = 0
        while time.perf_counter() - t0 < 0.25:                         # (about the span of rank 0's frames)
            for _ in range(10):
                mapper.step(ro, rd, rgb, d.reshape(-1))
            torch.cuda.synchronize(); n += 10
        ms_frame, ba_its = 0.0, n / (time.perf_counter() - t0)
    tt = torch.tensor([ms_frame, ba_its], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, group=group)
    out["c4_ms_per_frame_rank0"] = float(tt[0])
    out["c4_inactive_ba_iterations_per_s_other_ranks"] = float(tt[1])
    out["c4_shape"] = ("16 submaps round robin; rank 0: RO 5 x 2000 x 384 + 10 pose-refinement iterations + mapping every 3rd frame on the "
                       "active submap; ranks 1..G-1: InactiveMap.local_BA iterations (2600 rays x 75) on their submaps at the same time")
    return out


def emit(obj):
    """Write the single JSON line to the real stdout (fd 1 is pointed at stderr while the bench runs so that
    library banners such as NCCL's version line cannot pollute it)."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


_REAL_STDOUT = 1

def store_bench(mapper, dev, steps):
    """Map step fed from the device-resident keyframe ray store (SURVEY 8 "next" row N1): 3584 rays sampled on the device
    from 8 stored keyframes (150 x 200 rays each) + 512 rays of the current frame, ray generation, then the same step."""
    import torch
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    cfg = {"sampling": {"kf_n_rays_h": 150, "kf_n_rays_w": 200}}
    dirs = synth.camera_rays()
    poses = synth.trajectory(8)
    store = mf.KeyframeRayStore(cfg, dirs.shape[0], dirs.shape[1], 8, dev)
    for k, c2w in enumerate(poses):
        fr = synth.render_frame(c2w, dirs, seed=k)
        store.add_keyframe({"direction": dirs, "rgb": fr["rgb"], "depth": fr["depth"], "frame_id": k})
    poses_all = torch.stack(list(poses)).to(dev)
    cur = store.rays[7, ::58][:512].contiguous()
    related = list(range(8))
    for _ in range(3):
        mapper.step_from_store(store, 0, related, poses_all, R_RAYS - 512, cur_rays7=cur)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        losses = mapper.step_from_store(store, 0, related, poses_all, R_RAYS - 512, cur_rays7=cur)
    float(losses[0])
    dt = time.perf_counter() - t0
    return {"store_fed_rays_per_s": R_RAYS * steps / dt,
            "store_fed_shape": "KeyframeRayStore.sample_rays_in_submap (device draws, 8 keyframes) + 512 current-frame rays -> "
                               "mf_gen_rays_packed -> map step; no host data per step"}


def joint_query_setup(dev, res=512, n_submaps=16):
    """16 overlapping submap boxes (4 x 4 across x / y, full height) over the apartment-sized volume and the res^3 grid axes."""
    import numpy as np
    import torch
    import helpers as H
    import mipsfusion_b200 as mf
    cfg = H.make_config(HASH)
    cfg["grid"]["use_bound_normalize"] = False
    of = H.oracle_field(cfg)
    state = H.state_of(of)
    models, poses, amin, amax, cents = [], [], [], [], []
    lo, hi = np.array([-0.6, 0.5, -1.15]), np.array([2.95, 7.05, 3.05])
    ext = hi - lo
    for m in range(n_submaps):
        ix, iy = m % 4, m // 4
        a = lo + ext * np.array([ix / 4.0 - 0.08, iy / 4.0 - 0.08, 0.0])
        b = lo + ext * np.array([(ix + 1) / 4.0 + 0.08, (iy + 1) / 4.0 + 0.08, 1.0])
        models.append(H.cuda_model(cfg, state, train=False))
        T = torch.eye(4); T[:3, 3] = torch.tensor((a + b) / 2, dtype=torch.float32)
        poses.append(T); amin.append(a); amax.append(b); cents.append(((a + b) / 2).astype(np.float32))
    axes = [np.linspace(lo[k], hi[k], res) for k in range(3)]
    return mf.JointSubmapQuery(models, poses, amin, amax, cents), axes, amin, amax


def joint_query_bench(dev, res=512, n_submaps=16, group=None, shard="points", prefix="joint_query"):
    """BASELINE configs[4] shape: joint SDF grid query at res^3 over n_submaps submaps (Mesher / render_mesh path):
    containment + world->submap transform + field query (sdf, entropy) + entropy/distance-weighted blend."""
    import numpy as np
    import torch
    jq, axes, amin, amax = joint_query_setup(dev, res, n_submaps)
    kw = {} if group is None else dict(group=group, shard=shard)
    jq.query(axes=[a_[:64] for a_ in axes], **kw)                # warm-up: kernels, ...
    out = jq.query(axes=axes, **kw)                              # ... and the 1.3 GB of result / work buffers (cudaMalloc is not the query)
    del out
    torch.cuda.synchronize()
    if group is not None:
        import torch.distributed as dist
        dist.barrier()
    t0 = time.perf_counter()
    out = jq.query(axes=axes, **kw)
    torch.cuda.synchronize()
    dt = _max_over_ranks(time.perf_counter() - t0, dev, group)
    frac = float(out["mask"].float().mean())
    # (point, containing submap) pairs: the boxes are axis aligned, so the count factorises over the axes
    evals = float(sum(np.prod([np.count_nonzero((axes[k] >= amin[m][k]) & (axes[k] <= amax[m][k])) for k in range(3)])
                      for m in range(n_submaps)))
    del out
    roof = None
    if evals is not None:
        jb = evals * (ALG_BYTES_PER_POINT + 8)                        # SURVEY 8d: per point per containing submap 1,024 B + 8 B out
        roof = {"alg_bytes": jb, "ms": dt * 1e3, "achieved": jb / dt / 1e9, "evals": evals,
                "what": f"{res}^3 grid x {n_submaps} submaps: containment + SDF-only field query of every (point, containing submap) "
                        "pair + blend; per pair 1,032 B" + ("" if group is None else " (all ranks)")}
    if prefix != "joint_query":
        return {prefix + "_grid_points_per_s": res ** 3 / dt, prefix + "_s": dt,
                prefix + "_shape": f"{res}^3 grid x {n_submaps} submaps, submap m evaluated on GPU m mod G, partial sums (2 floats per grid "
                                   "point) all-reduced (what the online system needs: the submaps live on different GPUs)"}
    return {"_roof_joint_query": roof, "joint_query_grid_points_per_s": res ** 3 / dt, "joint_query_s": dt,
            "joint_query_shape": f"{res}^3 grid x {n_submaps} submaps (T=2^{HASH} each), {frac:.2f} of the points inside >= 1 submap"
                                 + ("" if group is None else "; the grid points are sharded across the GPUs (strong scaling, results stay sharded)")}


def frame_bench(dev, frames=3):
    """ms/frame of the reference's per-frame work at its shipped sizes (configs/FastCaMo-synth/FastCaMo-synth.yaml):
    RandomOptimizer 5 iterations x 2000 particles x 384 pixels, 10 gradient pose-refinement iterations x 1000 rays x 75
    samples, and 15 mapping iterations x 2600 rays x 75 samples every 3rd frame (amortised), on one synthetic 640x480 frame
    (cropped to 620x460).  Pose refinement: FusedPoseRefiner (the GO loop without autograd; the drop-in autograd route is timed
    beside it as ms_per_frame_640x480_autograd_go)."""
    import types
    import torch
    import helpers as H
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    from mipsfusion_b200.mapper import FusedMapper
    from mipsfusion_b200 import sampling_helper as sh
    cfg = H.make_config(HASH, n_samples_d=50, n_range_d=25)
    cfg["tracking"] = {"RO": {"particle_size": 2000, "initial_scaling_factor": 0.02, "rescaling_factor": 0.5, "n_rows": 16, "n_cols": 24},
                       "ignore_edge_W": 20, "ignore_edge_H": 20, "lr_rot": 1e-3, "lr_trans": 1e-3, "wait_iters": 100, "best": True}
    of = H.oracle_field(cfg)
    model = H.cuda_model(cfg, H.state_of(of))
    dirs = synth.camera_rays()
    c2w = synth.trajectory(4)[1]
    frame = synth.render_frame(c2w, dirs)
    depth_d, rgb_d, dirs_d = frame["depth"].to(dev), frame["rgb"].to(dev), dirs.to(dev)
    ds = types.SimpleNamespace(H=460, W=620, fx=320.0, fy=320.0, cx=309.5, cy=229.5, rays_d=dirs)
    ro = mf.RandomOptimizer(cfg, types.SimpleNamespace(dataset=ds, device=str(dev)))
    mapper = FusedMapper(model)
    refiner = mf.FusedPoseRefiner(model)
    tw = cfg["training"]

    def one_frame(do_map, fused_go=True):
        model.eval()
        pose = ro.optimize(model, frame["depth"], c2w.clone(), c2w.clone(), n_iter=5).to(dev)      # RO (returns a CPU pose, as the reference)
        model.train()
        rows, cols = sh.sample_pixels_mix(460, 620, 16, 24, depth_d, 1000)
        d_cam, t_rgb, t_d = dirs_d[rows, cols], rgb_d[rows, cols], depth_d[rows, cols].unsqueeze(-1)
        if fused_go:
            pose_f, _ = refiner.refine(pose, d_cam, t_rgb, t_d, 10)                               # GO (mipsfusion.py:501-556)
            pose = pose_f.clone()
        else:
            trans = pose[:3, 3].clone().requires_grad_(True)
            rot = pose[:3, :3].clone().requires_grad_(True)
            opt = torch.optim.Adam([rot, trans], lr=1e-3)
            for _ in range(10):
                opt.zero_grad()
                rays_o = trans[None, :].repeat(1000, 1)
                rays_d = torch.sum(d_cam[..., None, :] * rot[None], -1)
                ret = model(rays_o, rays_d, t_rgb, t_d, EMD_w=0.0)
                loss = tw["rgb_weight"] * ret["rgb_loss"] + tw["sdf_weight"] * ret["sdf_loss"] + tw["fs_weight"] * ret["fs_loss"]
                loss.backward()
                opt.step()
        if do_map:
            idx = torch.randint(0, 460 * 620, (2600,), device=dev)
            r_, c_ = idx // 620, idx % 620
            ro_, rd_ = pose[None, :3, 3].repeat(2600, 1).contiguous(), torch.sum(dirs_d[r_, c_][..., None, :] * pose[None, :3, :3], -1).contiguous()
            for _ in range(15):                                                                   # local BA (mipsfusion.py:293-335)
                mapper.step(ro_, rd_, rgb_d[r_, c_].contiguous(), depth_d[r_, c_].contiguous())
        return float(pose[0, 3])                                                                  # the frame's pose is read on the host

    out = {}
    for fused, key in ((True, "ms_per_frame_640x480"), (False, "ms_per_frame_640x480_autograd_go")):
        one_frame(True, fused)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(frames):
            one_frame(k % 3 == 0, fused)
        torch.cuda.synchronize()
        out[key] = (time.perf_counter() - t0) / frames * 1e3
    # the pose-refinement stage alone, device time
    rows, cols = sh.sample_pixels_mix(460, 620, 16, 24, depth_d, 1000)
    d_cam, t_rgb, t_d = dirs_d[rows, cols], rgb_d[rows, cols], depth_d[rows, cols].unsqueeze(-1)
    pose0 = c2w.to(dev)
    refiner.refine(pose0, d_cam, t_rgb, t_d, 10)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record()
    for _ in range(3):
        refiner.refine(pose0, d_cam, t_rgb, t_d, 10)
    b.record(); torch.cuda.synchronize()
    out["pose_refinement_10_iterations_ms"] = a.elapsed_time(b) / 3
    out["frame_shape"] = ("RO 5 x 2000 x 384, pose refinement 10 x 1000 rays x 75 (FusedPoseRefiner: tensor-core forward + ray-gradient-only "
                          "tensor-core backward, no autograd), mapping 15 x 2600 rays x 75 every 3rd frame")
    return out


if __name__ == "__main__":
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="timed steps only (for runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl b200)")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_gpu(a)
