"""The analytic chain of the fused overlap SDF operator (mipsfusion_b200.OverlapSDF, overlap_kernels.cu) restated in fp64 and
checked against torch autograd of the composition oracle/overlap.py on tests/golden/overlap.npz, plus the batched form (a loop
over submap pairs) against single-pair calls.  CPU only."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers as H
from oracle import overlap as oov

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "overlap.npz")


def _state(fx, i):
    pre = f"w{i}:"
    return {k[len(pre):]: torch.from_numpy(v) for k, v in fx.items() if k.startswith(pre)}


def inverse_adjugate(F):
    """F^-1 the way mf_overlap_points forms it: fp64 adjugate (2x2 minors of rows {0,1} and {2,3}) / determinant, rounded
    once to fp32."""
    a = np.asarray(F, np.float64).reshape(16)
    s0, s1, s2 = a[0] * a[5] - a[4] * a[1], a[0] * a[6] - a[4] * a[2], a[0] * a[7] - a[4] * a[3]
    s3, s4, s5 = a[1] * a[6] - a[5] * a[2], a[1] * a[7] - a[5] * a[3], a[2] * a[7] - a[6] * a[3]
    c5, c4, c3 = a[10] * a[15] - a[14] * a[11], a[9] * a[15] - a[13] * a[11], a[9] * a[14] - a[13] * a[10]
    c2, c1, c0 = a[8] * a[15] - a[12] * a[11], a[8] * a[14] - a[12] * a[10], a[8] * a[13] - a[12] * a[9]
    det = s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0
    b = np.array([
        a[5] * c5 - a[6] * c4 + a[7] * c3, -a[1] * c5 + a[2] * c4 - a[3] * c3, a[13] * s5 - a[14] * s4 + a[15] * s3, -a[9] * s5 + a[10] * s4 - a[11] * s3,
        -a[4] * c5 + a[6] * c2 - a[7] * c1, a[0] * c5 - a[2] * c2 + a[3] * c1, -a[12] * s5 + a[14] * s2 - a[15] * s1, a[8] * s5 - a[10] * s2 + a[11] * s1,
        a[4] * c4 - a[5] * c2 + a[7] * c0, -a[0] * c4 + a[1] * c2 - a[3] * c0, a[12] * s4 - a[13] * s2 + a[15] * s0, -a[8] * s4 + a[9] * s2 - a[11] * s0,
        -a[4] * c3 + a[5] * c1 - a[6] * c0, a[0] * c3 - a[1] * c1 + a[2] * c0, -a[12] * s3 + a[13] * s1 - a[14] * s0, a[8] * s3 - a[9] * s1 + a[10] * s0])
    return torch.from_numpy((b / det).astype(np.float32).reshape(4, 4))


def pose_chain(finv, ovlp, target_d, rays_d_cam, d_pts):
    """fp64 restatement of mf_overlap_pose_bwd for one side.  finv (4,4); ovlp (N,4,4) or (1,4,4); target_d (N,); rays_d_cam
    (N,3); d_pts (N,3) = d loss / d point.  dA[:3,3] = dx, dA[i][k] = dx_i depth d_cam_k; d(F^-1) = sum_r dA_r O_r^T;
    dF = -F^-T d(F^-1) F^-T; dO_r = F^-T dA_r.  -> (dF (4,4), dO shaped like ovlp)."""
    d = lambda t: torch.as_tensor(t).detach().to(torch.float64)
    fi, O, dep, dc, dx = d(finv), d(ovlp), d(target_d).reshape(-1), d(rays_d_cam), d(d_pts)
    N = dx.shape[0]
    dA = torch.zeros(N, 4, 4, dtype=torch.float64)
    dA[:, :3, :3] = (dx * dep[:, None])[:, :, None] * dc[:, None, :]
    dA[:, :3, 3] = dx
    if O.shape[0] == 1:
        S = dA.sum(0)
        d_finv, dO = S @ O[0].T, (fi.T @ S)[None]
    else:
        d_finv, dO = (dA @ O.transpose(1, 2)).sum(0), fi.T @ dA
    return -fi.T @ d_finv @ fi.T, dO


def pair_chain(models, target_d, rays_d_cam, mask, ovlp, id1, id2, first1, first2, trunc, finv_fn=torch.inverse,
               want_pts_grad=False):
    """loss and its gradients w.r.t. the two first-keyframe poses and the overlap poses through the restated chain; the
    field's point gradients come from autograd of run_network on the points the chain forms (finv_fn(F) = F^-1)."""
    mask = mask.to(target_d)
    finvs, locals_, sdf = [], [], []
    for sid, F in ((id1, first1), (id2, first2)):
        fi = finv_fn(F.detach())
        A = fi @ ovlp.detach()
        rays_d = torch.sum(rays_d_cam[..., None, None, :] * A[..., None, :3, :3], -1).reshape(-1, 3)
        pts = (A[..., :3, 3].reshape(-1, 3) + rays_d * target_d).detach().requires_grad_(True)
        sdf.append(models[int(sid)].run_network(pts)[..., 3:4] * trunc)
        finvs.append(fi); locals_.append(pts)
    loss = oov.compute_avg_sdf_difference(sdf[0], sdf[1], mask)
    d_pts = torch.autograd.grad(loss, locals_)
    g1, dO1 = pose_chain(finvs[0], ovlp, target_d, rays_d_cam, d_pts[0])
    g2, dO2 = pose_chain(finvs[1], ovlp, target_d, rays_d_cam, d_pts[1])
    if want_pts_grad:
        return loss.detach(), g1, g2, dO1 + dO2, d_pts
    return loss.detach(), g1, g2, dO1 + dO2


def batched_oracle(models, pair_ids, target_d, rays_d_cam, mask, ovlp, first_poses, trunc):
    """OverlapSDF.pairs restated as a loop over pairs of the composition: losses (P,)."""
    return torch.stack([oov.get_sdf_dif2(models, target_d[p][:, None], rays_d_cam[p], mask[p][:, None], ovlp[p], i1, i2,
                                         first_poses[i1], first_poses[i2], trunc) for p, (i1, i2) in enumerate(pair_ids)])


def _golden():
    fx = np.load(GOLD)
    cfg = H.make_config(int(fx["hash_size"]))
    models = [H.oracle_field(cfg, _state(fx, i)) for i in range(2)]
    return fx, models


class _LinearField:
    """A field whose SDF is linear in the point, sdf(x_i) = G_i . x_i: d sdf_i / d x_i = G_i, any dtype."""

    def __init__(self, G):
        self.G = G

    def run_network(self, pts):
        out = torch.zeros(pts.shape[0], 10, dtype=pts.dtype)
        return torch.cat([out[:, :3], (pts * self.G).sum(-1, keepdim=True), out[:, 4:]], -1)


def _golden_cases(fx):
    t = lambda k: torch.from_numpy(fx[k])
    rays = t("rays")
    return rays, ((t("ovlp"), (rays[:, 6:7] > 0), (0, 1)), (t("pose2"), t("mask2"), (1, 0)))


def test_chain_matches_fp64_autograd_of_infer_pts():
    """points -> dA -> dF, dO restated equals autograd through oracle/overlap.infer_pts in fp64, with the golden fields'
    point gradients as the upstream gradient of each side."""
    fx, models = _golden()
    trunc = float(fx["trunc"])
    rays, cases = _golden_cases(fx)
    d64 = lambda t: t.detach().to(torch.float64)
    for ovlp, mask, (i1, i2) in cases:
        _, _, _, _, d_pts = pair_chain(models, rays[:, 6:7], rays[:, :3], mask, ovlp, i1, i2, torch.from_numpy(fx["first1"]),
                                       torch.from_numpy(fx["first2"]), trunc, want_pts_grad=True)
        for side, F in enumerate((fx["first1"], fx["first2"])):
            F64 = torch.from_numpy(F).to(torch.float64).requires_grad_(True)
            O64 = d64(ovlp).requires_grad_(True)
            _, sdf = oov.infer_pts(F64.inverse() @ O64, _LinearField(d64(d_pts[side])), d64(rays[:, :3]), d64(rays[:, 6:7]), 1.0)
            sdf.sum().backward()
            dF, dO = pose_chain(F64.detach().inverse(), ovlp, rays[:, 6:7], rays[:, :3], d_pts[side])
            assert H.rel_err(dF, F64.grad) < 1e-6, H.rel_err(dF, F64.grad)
            assert H.rel_err(dO, O64.grad) < 1e-6, H.rel_err(dO, O64.grad)


def test_chain_matches_autograd_of_composition():
    """End to end in fp32 against autograd of oracle/overlap.get_sdf_dif2: the loss to 1e-5 (summation order), the gradients to the fp32
    rounding of autograd's own chain (measured 5.5e-5 on this fixture)."""
    fx, models = _golden()
    t = lambda k: torch.from_numpy(fx[k])
    trunc = float(fx["trunc"])
    rays, cases = _golden_cases(fx)
    for ovlp, mask, (i1, i2) in cases:
        f1 = t("first1").requires_grad_(True); f2 = t("first2").requires_grad_(True)
        O = ovlp.clone().requires_grad_(True)
        loss = oov.get_sdf_dif2(models, rays[:, 6:7], rays[:, :3], mask, O, i1, i2, f1, f2, trunc)
        loss.backward()
        l, g1, g2, dO = pair_chain(models, rays[:, 6:7], rays[:, :3], mask, ovlp, i1, i2, t("first1"), t("first2"), trunc)
        assert abs(float(l) - float(loss.detach())) <= 1e-5 * abs(float(loss.detach()))
        for got, ref in ((g1, f1.grad), (g2, f2.grad), (dO, O.grad)):
            assert H.rel_err(got, ref) < 2e-4, H.rel_err(got, ref)


def test_adjugate_inverse_is_the_fp64_inverse_rounded_once():
    fx, _ = _golden()
    for k in ("first1", "first2"):
        F = fx[k]
        ref = np.linalg.inv(F.astype(np.float64))
        assert np.array_equal(inverse_adjugate(F).numpy(), ref.astype(np.float32))
        assert H.rel_err(inverse_adjugate(F), torch.from_numpy(F).inverse()) < 1e-6


def test_batched_oracle_equals_single_pair_calls():
    fx, models = _golden()
    trunc = float(fx["trunc"])
    rays = torch.from_numpy(fx["rays"])
    N = rays.shape[0]
    g = torch.Generator().manual_seed(3)
    pair_ids = [(0, 1), (1, 0), (0, 0), (1, 1)]
    P = len(pair_ids)
    perm = [torch.randperm(N, generator=g) for _ in range(P)]
    target_d = torch.stack([rays[p, 6] for p in perm])
    dirs = torch.stack([rays[p, :3] for p in perm])
    mask = torch.stack([(torch.rand(N, generator=g) > 0.3).float() for _ in range(P)])
    ovlp = torch.from_numpy(fx["ovlp"])[None].repeat(P, 1, 1, 1)
    first = torch.from_numpy(np.stack([fx["first1"], fx["first2"]])).requires_grad_(True)
    losses = batched_oracle(models, pair_ids, target_d, dirs, mask, ovlp, first, trunc)
    losses.sum().backward()
    acc = torch.zeros(2, 4, 4)
    for p, (i1, i2) in enumerate(pair_ids):
        f1 = first.detach()[i1].clone().requires_grad_(True); f2 = first.detach()[i2].clone().requires_grad_(True)
        lp = oov.get_sdf_dif2(models, target_d[p][:, None], dirs[p], mask[p][:, None], ovlp[p], i1, i2, f1, f2, trunc)
        assert float(lp) == float(losses[p])
        lp.backward()
        acc[i1] += f1.grad; acc[i2] += f2.grad
    assert H.rel_err(acc, first.grad) < 1e-6


def test_entry_points_exported():
    """The fused operator's C entry points are declared, bound and exported (the library is built for sm_100a; loading it
    makes no CUDA call)."""
    import ctypes as C
    from mipsfusion_b200 import _lib as L
    dll = C.CDLL(L.LIB_PATH)
    header = open(L.HEADER_PATH).read()
    for name in ("mf_overlap_points", "mf_overlap_loss", "mf_overlap_pose_bwd"):
        assert hasattr(dll, name) and name in L.PROTOTYPES and f"int {name}(" in header
