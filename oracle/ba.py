"""ORACLE (test infrastructure only): the local bundle adjustment loop of the mapping process, MIPSFusion.local_BA
(mipsfusion.py:259-370), in CPU torch with autograd.

Per iteration: a ray batch of the submap's keyframes plus the current frame's rays, rays generated from ``poses_all``
(:320-322), the oracle field's forward and total loss (oracle/scene.py), ``loss.backward(retain_graph=True)``, the map Adam
step and zero_grad every iteration (map_accum_step 1, oracle/adam.py), and every ``pose_accum_step`` iterations one
``torch.optim.Adam`` step on the keyframe poses, after which ``poses_all`` is rebuilt from the parameters.

Restated, not pinned against mipsfusion.py (no checkout of the reference is available offline): the loop structure above is
taken from SURVEY.md 3.1, and the pose parametrisation from the tracking oracle (oracle/tracking.py: the ``matrix_to_quaternion``
shim, ``qt_to_transform_matrix``, Adam with a quaternion group at lr_rot and a translation group at lr_trans, default betas and
eps).  So are: pose 0 (the submap's first keyframe) is fixed (``get_pose_param_optim(poses[1:])``), the last pose (the current
frame) is fixed unless ``optim_cur``, ``poses_all`` is the fixed poses concatenated with the optimised ones, and the pose
gradients of a trailing partial accumulation period are never applied.

The ray batches come from :func:`store_batch`: the keyed Feistel draws of oracle/keyframes.py with the seeds the device loop
uses, gathered by ``sample_rays_in_submap``, so the oracle and the device see the same rays bit for bit."""
import torch

from . import adam as oadam
from . import keyframes as okf
from .shims.pytorch3d.transforms import matrix_to_quaternion
from .tracking import qt_to_transform_matrix


def store_batch(store, first_kf_Id, related_kf_ids, pix_num, seed, cur_rays7=None):
    """store (num_kf, n_rays, 7) -> rays7 (R,7), pose_idx (R,) of one iteration: the draws mf_kf_sample_rays makes with
    segment seeds seed, seed + 1, seed + 2, then the current frame's rays with pose index -1 (the last pose)."""
    related = torch.as_tensor(related_kf_ids, dtype=torch.int64)
    n_rel, nr = int(related.shape[0]), store.shape[1]
    nf, no, nl = okf.split_counts(pix_num, n_rel)
    n_other_kf = n_rel - 2 if n_rel > 2 else n_rel - 1
    draws = dict(idx_first=torch.from_numpy(okf.feistel_sample(nr, nf, seed & 0xffffffff)))
    if no:
        draws["idx_other"] = torch.from_numpy(okf.feistel_sample(n_other_kf * nr, no, (seed + 1) & 0xffffffff))
    if nl:
        draws["idx_last"] = torch.from_numpy(okf.feistel_sample(nr, nl, (seed + 2) & 0xffffffff))
    rays, _, kf_indices = okf.sample_rays_in_submap(store, first_kf_Id, related, pix_num, **draws)
    if cur_rays7 is None:
        return rays, kf_indices
    return torch.cat([rays, cur_rays7], 0), torch.cat([kf_indices, -torch.ones(cur_rays7.shape[0], dtype=torch.int64)])


def pose_parameters(poses_all, optim_cur):
    """get_pose_param_optim (:235-241) on the optimised poses: (rot (n,4), trans (n,3)) Parameters and ``build()`` ->
    poses_all (K,4,4) = first pose | optimised poses | current frame's pose when it is not optimised."""
    K = poses_all.shape[0]
    opt = poses_all[1:] if optim_cur else poses_all[1:K - 1]
    rot = torch.nn.parameter.Parameter(matrix_to_quaternion(opt[:, :3, :3]).clone())
    trans = torch.nn.parameter.Parameter(opt[:, :3, 3].clone())

    def build():
        parts = [poses_all[:1], qt_to_transform_matrix(rot, trans)]
        if not optim_cur:
            parts.append(poses_all[K - 1:])
        return torch.cat(parts, 0)
    return rot, trans, build


def gen_rays(rays7, pose_idx, P):                                  # mipsfusion.py:320-322
    idx = pose_idx.clone()
    idx[idx < 0] += P.shape[0]
    return P[idx, :3, 3], torch.sum(rays7[:, None, :3] * P[idx, :3, :3], -1)


def local_ba(field, batches, poses_all, pose_accum_step, lr_rot, lr_trans, optim_cur, lr_decoder=1e-2, lr_embed=1e-2, u=None,
             EMD_w=0.01):
    """batches: one (rays7 (R,7), pose_idx (R,)) per iteration.  Steps ``field`` in place.
    -> dict: poses (K,4,4) after the loop, losses (n_iters, 4) [rgb, depth, sdf, fs], and per pose step the poses after it
    (``step_poses``) and the accumulated gradient of the optimised poses' (q, t) it applied (``step_grads``, (n, 7))."""
    rot, trans, build = pose_parameters(poses_all, optim_cur)
    pose_opt = torch.optim.Adam([{"params": rot, "lr": lr_rot}, {"params": trans, "lr": lr_trans}])
    map_opt = oadam.make_optimizer(field, lr_decoder, lr_embed)
    P = build()
    losses, step_poses, step_grads = [], [], []
    for i, (rays7, pose_idx) in enumerate(batches):
        rays_o, rays_d = gen_rays(rays7, pose_idx, P)
        ret = field.forward(rays_o, rays_d, rays7[:, 3:6], rays7[:, 6:7], None if u is None else u[i], EMD_w=EMD_w)
        field.total_loss(ret).backward(retain_graph=True)                                       # :327
        losses.append([float(ret[k].detach()) for k in ("rgb_loss", "depth_loss", "sdf_loss", "fs_loss")])
        map_opt.step()                                                                           # :330-335
        map_opt.zero_grad()
        if (i + 1) % pose_accum_step == 0:                                                       # :338-342
            step_grads.append(torch.cat([rot.grad, trans.grad], 1).clone())
            pose_opt.step()
            pose_opt.zero_grad()
            P = build()
            step_poses.append(P.detach().clone())
    return dict(poses=P.detach().clone(), losses=torch.tensor(losses), step_poses=step_poses, step_grads=step_grads)
