"""Smoke check of programmatic dependent launch (mf_launch, mf_common.cuh) on the map step: one FusedMapper.step with it and one
in plain stream order, from the same seeded model and batch in one process, give the same z, raw, rendered colour / depth,
losses, d_raw, active-point list, decoder gradient and decoder after Adam bit for bit, and the hash-grid gradient (atomic
scatter) to fp32 rounding.  One run per mode can only catch an ordering hazard if the race fires in that run: the hazard rule
itself is argued in mf_common.cuh, not proven here."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers as H

pytestmark = pytest.mark.gpu


def _one_step(pdl, cfg, state, batch, update):
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200.decoder import _Workspace
    from mipsfusion_b200.mapper import FusedMapper
    prev = L.lib().mf_get_pdl()                  # (restored below: an MF_NO_PDL=1 session stays so for later tests)
    L.call("mf_set_pdl", 1 if pdl else 0)
    try:
        mapper = FusedMapper(H.cuda_model(cfg, state))
        ro, rd, rgb, d, u = batch
        R, S = ro.shape[0], u.shape[1]
        losses = mapper.step(ro, rd, rgb, d, u=u, update=update)
        torch.cuda.synchronize()
    finally:
        L.call("mf_set_pdl", prev)
    b = mapper._buffers(R, S)
    out = {k: b[k].cpu().numpy().copy() for k in ("z", "raw", "rgb", "depth", "d_raw", "counts")}
    out["losses"] = losses.cpu().numpy().copy()
    N = R * S
    ws = _Workspace.get(mapper.dev, field_points=N)
    off = int(L.lib().mf_mlp_grad_workspace_size())
    nb = (N + 1023) // 1024
    words = ws[off:off + N + nb * 33 + 1].view(torch.int32).cpu().numpy()
    n_active = int(words[N + nb * 33])
    out["active"] = words[:n_active].copy()
    out["g_mlp"] = mapper.g_mlp.cpu().numpy().copy()
    out["g_grid"] = mapper.g_grid.cpu().numpy().copy()
    out["mlp"] = mapper.mlp.cpu().numpy().copy()
    out["grid"] = mapper.grid.cpu().numpy().copy()
    return out


@pytest.mark.parametrize("update", [False, True])
def test_map_step_pdl_matches_stream_order(update):
    cfg = H.make_config(16, n_samples_d=32, n_range_d=11)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=7)
    state = H.state_of(of)
    R = 2048
    rays_o, rays_d, rgb, d, u = H.synth_batch(R, 43, seed=11)
    batch = tuple(t.cuda().contiguous() for t in (rays_o, rays_d, rgb, d.reshape(-1), u))
    a = _one_step(False, cfg, state, batch, update)
    b = _one_step(True, cfg, state, batch, update)
    assert 0 < a["active"].size < R * 43 and np.all(np.diff(a["active"]) > 0)
    for k in ("z", "raw", "rgb", "depth", "losses", "d_raw", "counts", "active", "g_mlp", "mlp"):
        assert a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), k
    # the grid gradient is a float atomic scatter: its summation order is not fixed, in either launch mode
    for k in ("g_grid", "grid"):
        np.testing.assert_allclose(b[k], a[k], rtol=1e-5, atol=1e-7 * max(1.0, float(np.abs(a[k]).max())), err_msg=k)
    if update:
        assert not np.any(a["g_mlp"]) and not np.any(b["g_mlp"])              # Adam zeroed the gradients it consumed
