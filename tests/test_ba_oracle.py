"""CPU checks of the local bundle adjustment oracle (oracle/ba.py): the pose gradient it applies, the loop with the pose
learning rates at zero, and the poses that are never optimised."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers as H
from oracle import adam as oadam
from oracle import ba as oba
from oracle.tracking import qt_to_transform_matrix


def _poses(K):
    from mipsfusion_b200 import synth
    return synth.trajectory(K).to(torch.float32).contiguous()


def test_pose_gradient_through_qt_to_transform_matrix_matches_central_differences():
    """d loss / d (q, t) through qt_to_transform_matrix and the ray generation, against fp64 central differences."""
    g = torch.Generator().manual_seed(4)
    P0 = _poses(5).double()
    rot, trans, build = oba.pose_parameters(P0, optim_cur=True)
    rays7 = torch.rand(200, 7, generator=g, dtype=torch.float64) - 0.5
    idx = torch.randint(-1, 4, (200,), generator=g)
    w = torch.randn(200, 6, generator=g, dtype=torch.float64)

    def loss_of(r, t):
        P = torch.cat([P0[:1], qt_to_transform_matrix(r, t)], 0)
        o, d = oba.gen_rays(rays7, idx, P)
        return (torch.sin(torch.cat([o, 3.0 * d], 1)) * w).sum()
    rot64 = rot.detach().double().requires_grad_(True)
    trans64 = trans.detach().double().requires_grad_(True)
    loss_of(rot64, trans64).backward()
    ana = torch.cat([rot64.grad, trans64.grad], 1)
    num = torch.zeros_like(ana)
    h = 1e-6
    for p in range(ana.shape[0]):
        for c in range(7):
            r, t = rot64.detach().clone(), trans64.detach().clone()
            tgt = r if c < 4 else t
            cc = c if c < 4 else c - 4
            tgt[p, cc] += h
            lp = float(loss_of(r, t))
            tgt[p, cc] -= 2 * h
            lm = float(loss_of(r, t))
            num[p, c] = (lp - lm) / (2 * h)
    assert H.rel_err(ana, num) < 1e-7, H.rel_err(ana, num)


def _fixture(K=5, iters=6, R=96):
    cfg = H.make_config(12, n_samples_d=16, n_range_d=7)
    cfg["training"]["perturb"] = 0
    rays7, _, _, g = H.synth_batch_packed(R * iters, seed=3)
    P = _poses(K)
    batches = [(rays7[i * R:(i + 1) * R], torch.randint(-1, K - 1, (R,), generator=g)) for i in range(iters)]
    return cfg, P, batches


def test_zero_pose_learning_rates_give_the_plain_map_loop():
    cfg, P, batches = _fixture()
    of = H.oracle_field(cfg, grid_scale=0.3, seed=1)
    plain = H.oracle_field(cfg, grid_scale=0.3, seed=1)
    res = oba.local_ba(of, batches, P, 2, 0.0, 0.0, optim_cur=True)
    _, _, build = oba.pose_parameters(P, optim_cur=True)
    P0 = build().detach()
    opt = oadam.make_optimizer(plain)
    lo = []
    for rays7, idx in batches:
        o, d = oba.gen_rays(rays7, idx, P0)
        ret = plain.forward(o, d, rays7[:, 3:6], rays7[:, 6:7], None)
        plain.total_loss(ret).backward()
        lo.append([float(ret[k].detach()) for k in ("rgb_loss", "depth_loss", "sdf_loss", "fs_loss")])
        opt.step()
        opt.zero_grad()
    # (the backward through ray directions that require a gradient sums in a different order: last-bit differences)
    np.testing.assert_allclose(res["losses"].numpy(), np.array(lo, dtype=np.float32), rtol=1e-5)
    assert torch.equal(res["poses"], P0)
    assert len(res["step_grads"]) == 3 and all(float(s.abs().max()) > 0 for s in res["step_grads"])


def test_frozen_poses_never_move():
    cfg, P, batches = _fixture()
    for optim_cur in (False, True):
        of = H.oracle_field(cfg, grid_scale=0.3, seed=1)
        res = oba.local_ba(of, batches, P, 2, 1e-2, 1e-2, optim_cur=optim_cur)
        out = res["poses"]
        assert torch.equal(out[0], P[0])
        assert torch.equal(out[-1], P[-1]) != optim_cur
        assert all(float((out[k] - P[k]).abs().max()) > 1e-3 for k in range(1, P.shape[0] - 1))
        assert res["step_grads"][0].shape[0] == P.shape[0] - (1 if optim_cur else 2)
