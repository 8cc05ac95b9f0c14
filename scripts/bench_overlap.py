"""Overlap-region SDF consistency of the inactive-map global BA (InactiveMap.get_SDF_dif2) on one GPU.

Arms, alternated call by call, each ending with the pose gradients ready and a device synchronise:
  (a) composition: oracle/overlap.get_sdf_dif2 over the CUDA models (torch inverse and matmul, two run_network calls through the
      fp32 point route), summed over the pairs, then backward;
  (b) fused: mipsfusion_b200.OverlapSDF (get_SDF_dif2 for one pair, pairs() for many), then backward.
Both fill d loss / d first-keyframe poses and d loss / d overlap poses.  Shapes: one pair at N = 768 and at N = 500
(config["mapping"]["sample"] // 4 with sample = 2000), and 16 pairs over 16 submaps at N = 768 (T = 2^19 hash grids).
Reported per arm and shape: median host time to gradients ready (perf_counter around the call and a synchronise), median device
time (CUDA events), and, from a separate torch.profiler run, the device activities (kernels, memsets, copies) per call.

Prints one JSON line with the GPU name and power limit read in the same run; ``--out`` also writes it to a file."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")]

import torch  # noqa: E402


def median(v):
    return sorted(v)[len(v) // 2]


def make_inputs(n_submaps, P, N, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    def pose(scale):
        q = torch.randn(4, generator=g)
        q = q / q.norm()
        w, x, y, z = q.tolist()
        R = torch.tensor([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                          [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                          [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
        T = torch.eye(4)
        T[:3, :3], T[:3, 3] = R, scale * (torch.rand(3, generator=g) - 0.5)
        return T
    first = torch.stack([pose(1.0) for _ in range(n_submaps)])
    ovlp = torch.stack([torch.stack([pose(1.0)] * N) for _ in range(P)])
    dirs = torch.randn(P, N, 3, generator=g)
    dirs[..., 2] = -dirs[..., 2].abs() - 1.0
    depth = 0.5 + 2.5 * torch.rand(P, N, generator=g)
    mask = (torch.rand(P, N, generator=g) > 0.1).float()
    pair_ids = [(p % n_submaps, (p + 1 + p // n_submaps) % n_submaps) for p in range(P)]
    return dict(first=first.to(dev), ovlp=ovlp.to(dev), dirs=dirs.to(dev), depth=depth.to(dev), mask=mask.to(dev), pair_ids=pair_ids)


def arms(models, x, trunc):
    import mipsfusion_b200 as mf
    from oracle import overlap as oov
    ov = mf.OverlapSDF(models)
    P = len(x["pair_ids"])
    F = x["first"].clone().requires_grad_(True)
    O = x["ovlp"].clone().requires_grad_(True)

    def composition():
        F.grad = None; O.grad = None
        loss = sum(oov.get_sdf_dif2(models, x["depth"][p][:, None], x["dirs"][p], x["mask"][p][:, None], O[p], i1, i2, F[i1], F[i2],
                                    trunc) for p, (i1, i2) in enumerate(x["pair_ids"]))
        loss.backward()

    def fused():
        F.grad = None; O.grad = None
        if P == 1:
            i1, i2 = x["pair_ids"][0]
            loss = ov.get_SDF_dif2(x["depth"][0][:, None], x["dirs"][0], x["mask"][0][:, None], O[0], i1, i2, F[i1], F[i2], trunc)
        else:
            loss = ov.pairs(x["pair_ids"], x["depth"], x["dirs"], x["mask"], O, F, trunc).sum()
        loss.backward()

    return {"composition": composition, "fused": fused}


def measure(fns, reps, warmup):
    for _ in range(warmup):
        for f in fns.values():
            f()
    torch.cuda.synchronize()
    host = {k: [] for k in fns}
    dev = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record()
            f()
            b.record()
            torch.cuda.synchronize()
            host[k].append(1e3 * (time.perf_counter() - t0))
            dev[k].append(a.elapsed_time(b))
    return host, dev


def activities(f, calls=5):
    from torch.profiler import ProfilerActivity, profile
    f()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            f()
        torch.cuda.synchronize()
    n = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
    return n / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_overlap.py needs a GPU")
    import helpers as H
    from bench_ba import gpu_info
    dev = torch.device("cuda", torch.cuda.current_device())
    cfg = H.make_config(19)
    trunc = float(cfg["training"]["trunc"])
    n_sub = 16
    models = [H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, grid_scale=0.05, seed=i)), train=False) for i in range(n_sub)]
    res = dict(workload="overlap SDF consistency (get_SDF_dif2), gradients w.r.t. first-keyframe and overlap poses; T = 2^19",
               reps=args.reps, **gpu_info(dev.index))
    for label, P, N in (("1pair_768", 1, 768), ("1pair_500", 1, 500), ("16pairs_16submaps_768", 16, 768)):
        x = make_inputs(n_sub, P, N, dev, seed=P * 1000 + N)
        fns = arms(models if P > 1 else models[:2], x if P > 1 else {**x, "pair_ids": [(0, 1)]}, trunc)
        host, devt = measure(fns, args.reps, args.warmup)
        res[label] = {k: {"host_ms": round(median(host[k]), 4), "device_ms": round(median(devt[k]), 4)} for k in fns}
        for k, f in fns.items():
            res[label][k]["device_activities_per_call"] = activities(f)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
