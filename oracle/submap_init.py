"""ORACLE (test infrastructure only): submap initialisation of the mapping process, MIPSFusion.first_frame_mapping
(mipsfusion.py:155-194) and initialize_new_localMLP (:198-222), in CPU torch with autograd; and the per-iteration
current-frame draw of the local bundle adjustment (:306-309).

Per iteration of the initialisation: ``random.sample(range(H*W), pix_num)``, the index decoded column-major (h = i % H,
w = i // H, :178,209), direction / rgb / depth of those pixels gathered, rays generated with the frame's pose (:320-322 as
oracle/ba.py's ``gen_rays``), the oracle field's forward and total loss, backward, and the map Adam step with zero_grad
(oracle/adam.py).

Restated, not pinned against mipsfusion.py (no checkout of the reference is available offline; taken from SURVEY.md 3.1 and
Appendix C): the draw and its column-major decode, the identity pose of the frame that opens a submap, one map step per
iteration, and a fresh optimiser per submap.  The draw is the keyed Feistel permutation of oracle/keyframes.py in place of
python's ``random.sample``, so the oracle and the device see the same rays bit for bit."""
import torch

from . import adam as oadam
from . import keyframes as okf
from . import sampling as osamp
from .ba import gen_rays


def frame_batch(frame, pix_num, seed):
    """frame: dict 'direction' (H,W,3), 'rgb' (H,W,3), 'depth' (H,W) -> rays7 (pix_num, 7) of one iteration: pixel
    index i = perm(j) of the seeded permutation of range(H*W), pixel (i % H, i // H)."""
    H, W = frame["depth"].shape[-2:]
    i = torch.from_numpy(okf.feistel_sample(H * W, pix_num, seed & 0xffffffff))
    h, w = i % H, torch.div(i, H, rounding_mode="floor")
    d, c, z = frame["direction"].reshape(H, W, 3), frame["rgb"].reshape(H, W, 3), frame["depth"].reshape(H, W)
    return torch.cat([d[h, w], c[h, w], z[h, w][:, None]], -1)


def cur_frame_rays(frame, n_cur, keys):
    """The current frame's rows of one BA iteration: sample_pixels_mix(H, W, 16, 24, depth, n_cur) on ``keys`` (H*W), then
    [dir | rgb | depth] of those (row, col) pixels."""
    H, W = frame["depth"].shape[-2:]
    rows, cols = osamp.sample_pixels_mix(H, W, 16, 24, frame["depth"].reshape(H, W), n_cur, keys)
    px = rows * W + cols
    return torch.cat([frame["direction"].reshape(-1, 3)[px], frame["rgb"].reshape(-1, 3)[px], frame["depth"].reshape(-1, 1)[px]], -1)


def first_frame_mapping(field, batches, c2w, u=None, EMD_w=0.01, lr_decoder=1e-2, lr_embed=1e-2):
    """batches: one rays7 (R,7) per iteration; c2w (4,4) the frame's pose.  Steps ``field`` in place with a fresh Adam.
    -> losses (n_iters, 4) [rgb, depth, sdf, fs]."""
    opt = oadam.make_optimizer(field, lr_decoder, lr_embed)
    P = torch.as_tensor(c2w, dtype=torch.float32).reshape(1, 4, 4)
    losses = []
    for i, rays7 in enumerate(batches):
        rays_o, rays_d = gen_rays(rays7, -torch.ones(rays7.shape[0], dtype=torch.int64), P)
        ret = field.forward(rays_o, rays_d, rays7[:, 3:6], rays7[:, 6:7], None if u is None else u[i], EMD_w=EMD_w)
        field.total_loss(ret).backward()
        losses.append([float(ret[k].detach()) for k in ("rgb_loss", "depth_loss", "sdf_loss", "fs_loss")])
        opt.step()
        opt.zero_grad()
    return torch.tensor(losses)
