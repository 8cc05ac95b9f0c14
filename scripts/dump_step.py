"""Every intermediate buffer of ONE FusedMapper.step at the bench shape, from the seeded bench model and batch, as DIR/<name>.npy:
z, counts, raw, rgb, depth, losses, d_raw, the active-point list, the decoder gradient and the grid gradient (before Adam),
then the decoder and grid after Adam.  Two builds (or two runs of one build) are compared with scripts/compare_dumps.py; all
buffers but the grid gradient and the grid (float atomic scatter) are expected to be bitwise equal.

With --deterministic (mipsfusion_b200.set_deterministic) the grid gradient is order-independent too, and --steps K dumps the
K-th step (K - 1 full steps with Adam before it, the same draw u every step).  DIR/mode.json records the mode; when both
directories are deterministic dumps, compare_dumps.py expects EVERY buffer bitwise equal and exits non-zero otherwise.

    python scripts/dump_step.py DIR [--deterministic] [--steps K]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main(out, deterministic=False, steps=1):
    import bench
    import mipsfusion_b200 as mf
    import helpers as H
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200.decoder import _Workspace
    from mipsfusion_b200.mapper import FusedMapper
    os.makedirs(out, exist_ok=True)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg, of = bench.build_model()
    model = H.cuda_model(cfg, H.state_of(of))
    rays_o, rays_d, rgb, d, _ = bench.make_inputs(0)
    dv = torch.cat([rays_o, rays_d, rgb, d], -1).contiguous().to(dev)
    ro, rd, tc, td = dv[:, 0:3].contiguous(), dv[:, 3:6].contiguous(), dv[:, 6:9].contiguous(), dv[:, 9].contiguous()
    mapper = FusedMapper(model)
    R = ro.shape[0]
    cfg_r, _ = model._render_cfg(True, 0.01, dev)
    S = cfg_r.n_samples_d + cfg_r.n_range_d
    u = torch.rand(R, S, generator=torch.Generator().manual_seed(1234)).to(dev)     # host-seeded draw: the same in every build
    mf.set_deterministic(deterministic)
    for _ in range(steps - 1):
        mapper.step(ro, rd, tc, td, u=u)
    losses = mapper.step(ro, rd, tc, td, u=u, update=False)
    torch.cuda.synchronize()
    b = mapper._buffers(R, S)
    arrs = {k: b[k] for k in ("z", "counts", "raw", "rgb", "depth", "d_raw")}
    arrs["losses"] = losses
    N = R * S
    ws = _Workspace.get(mapper.dev, field_points=N)
    off = int(L.lib().mf_mlp_grad_workspace_size())
    nb = (N + 1023) // 1024
    words = ws[off:off + N + nb * 33 + 1].view(torch.int32)
    arrs["active"] = words[:int(words[N + nb * 33])]
    arrs["g_mlp"] = mapper.g_mlp
    arrs["g_grid"] = mapper.g_grid
    arrs = {k: v.detach().cpu().numpy().copy() for k, v in arrs.items()}
    mapper.apply_gradients()
    torch.cuda.synchronize()
    arrs["mlp_after_adam"] = mapper.mlp.cpu().numpy().copy()
    arrs["grid_after_adam"] = mapper.grid.cpu().numpy().copy()
    for k, v in arrs.items():
        np.save(os.path.join(out, k + ".npy"), v)
    with open(os.path.join(out, "mode.json"), "w") as f:
        json.dump({"deterministic": bool(deterministic), "steps": steps}, f)
    print("dumped", sorted(arrs), "n_active", arrs["active"].size, "deterministic", bool(deterministic), "steps", steps)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("dir")
    ap.add_argument("--deterministic", action="store_true")
    ap.add_argument("--steps", type=int, default=1)
    a = ap.parse_args()
    main(a.dir, a.deterministic, max(a.steps, 1))
