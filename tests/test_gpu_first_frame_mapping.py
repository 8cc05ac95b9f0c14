"""Submap initialisation on the device (FusedMapper.first_frame_mapping, the reference's first_frame_mapping /
initialize_new_localMLP, mipsfusion.py:155-222) and the per-iteration current-frame draw of local_ba (:306-309): the frame
draw kernel against the numpy Feistel restatement and a torch gather, the first iteration against step_host, the loops
against the CPU oracles (oracle/submap_init.py, oracle/ba.py), and the no-sync / no-allocation property."""
import gc
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers as H

pytestmark = pytest.mark.gpu

N_KF = 8
# camera-frame box of the synthetic frame's samples: the submap bound when the frame's pose is the identity
CAM_BOUND = [[-6.5, 6.5], [-5.0, 5.0], [-7.5, 0.5]]


@pytest.fixture(scope="module")
def room():
    """A full-resolution (460 x 620) synthetic frame rendered at pose traj[N_KF], the trajectory, and the frame on the GPU."""
    from mipsfusion_b200 import synth
    traj = synth.trajectory(N_KF + 1)
    fr = synth.render_frame(traj[N_KF], synth.camera_rays(), seed=3)
    frame = {k: fr[k].contiguous() for k in ("direction", "rgb", "depth")}
    return dict(frame=frame, dev={k: v.cuda() for k, v in frame.items()}, traj=traj.to(torch.float32).contiguous())


def _cfg(bound=None):
    cfg = H.make_config(14, n_samples_d=32, n_range_d=11)
    if bound is not None:
        cfg["mapping"]["bound"] = bound
    return cfg


def _gather(frame, i):
    Hh = frame["depth"].shape[0]
    h, w = i % Hh, torch.div(i, Hh, rounding_mode="floor")
    return torch.cat([frame["direction"][h, w], frame["rgb"][h, w], frame["depth"][h, w][:, None]], -1)


def test_kernel_draws_equal_the_feistel_sample_and_the_column_major_gather(room):
    from mipsfusion_b200.keyframe_store import sample_frame_rays
    from oracle import keyframes as okf
    fd = room["dev"]
    Hh, W = fd["depth"].shape
    assert (Hh, W) == (460, 620)
    for n in (1, 1800, 4096):
        seed = 4242 + n
        idx = torch.empty(n, device="cuda", dtype=torch.int64)
        rays = sample_frame_rays(fd, n, "cuda", seed=seed, out_idx=idx)
        ref_i = okf.feistel_sample(Hh * W, n, seed)
        np.testing.assert_array_equal(idx.cpu().numpy(), ref_i)
        assert torch.equal(rays, _gather(fd, torch.from_numpy(ref_i).cuda()))
    g = torch.Generator().manual_seed(1)
    small = {"direction": torch.randn(37, 53, 3, generator=g).cuda(), "rgb": torch.rand(37, 53, 3, generator=g).cuda(),
             "depth": torch.rand(37, 53, generator=g).cuda()}
    idx = torch.empty(37 * 53, device="cuda", dtype=torch.int64)
    rays = sample_frame_rays(small, 37 * 53, "cuda", seed=99, out_idx=idx)
    assert torch.equal(torch.sort(idx).values, torch.arange(37 * 53, device="cuda"))
    assert torch.equal(rays, _gather(small, idx))


def test_kernel_explicit_indices_and_argument_checks(room):
    import mipsfusion_b200 as mf
    from mipsfusion_b200.keyframe_store import sample_frame_rays
    fd = room["dev"]
    n = 1800
    idx = torch.empty(n, device="cuda", dtype=torch.int64)
    drawn = sample_frame_rays(fd, n, "cuda", seed=7, out_idx=idx)
    assert torch.equal(sample_frame_rays(fd, n, "cuda", idx=idx), drawn)
    assert torch.equal(sample_frame_rays(fd, n, "cuda", idx=idx.cpu().tolist()), drawn)        # the reference's random.sample list
    with pytest.raises(mf.MipsFusionB200Error):
        sample_frame_rays(fd, 460 * 620 + 1, "cuda", seed=1)
    with pytest.raises(mf.MipsFusionB200Error, match="outside"):
        sample_frame_rays(fd, 2, "cuda", idx=[0, 460 * 620])
    with pytest.raises(mf.MipsFusionB200Error, match="outside"):
        sample_frame_rays(fd, 2, "cuda", idx=[-1, 5])
    assert sample_frame_rays(fd, 0, "cuda", seed=1).shape == (0, 7)


def test_first_iteration_equals_step_host(room):
    from mipsfusion_b200.mapper import FusedMapper
    from oracle import submap_init as oinit
    cfg = _cfg()
    state = H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5))
    c2w = room["traj"][N_KF]
    R, seed = 1800, 31
    m1 = FusedMapper(H.cuda_model(cfg, state))
    torch.cuda.manual_seed(11)                    # the step's own jitter draw (torch.rand of the reference) on both sides
    la = m1.first_frame_mapping(room["dev"], 1, c2w=c2w.cuda(), pix_num=R, seed=seed)[0].cpu()
    rays7 = oinit.frame_batch(room["frame"], R, seed).contiguous()
    m2 = FusedMapper(H.cuda_model(cfg, state))
    torch.cuda.manual_seed(11)
    lb = m2.step_host(rays7.pin_memory(), None, c2w[None].cuda())
    np.testing.assert_array_equal(la.numpy(), lb.numpy())
    assert float(la[7]) > 0


def _probe(model, field, pts):
    with torch.no_grad():
        return model.run_network(pts.cuda()).cpu(), field.run_network(pts)


def _probe_points(bound, n=600, seed=0):
    b = torch.tensor(bound, dtype=torch.float32)
    return torch.rand(n, 3, generator=torch.Generator().manual_seed(seed)) * (b[:, 1] - b[:, 0]) + b[:, 0]


@pytest.mark.parametrize("pose", ["identity", "traj"])
def test_first_frame_mapping_vs_oracle(room, pose):
    from mipsfusion_b200.mapper import FusedMapper
    from oracle import submap_init as oinit
    bound = CAM_BOUND if pose == "identity" else None
    cfg = _cfg(bound)
    c2w = torch.eye(4) if pose == "identity" else room["traj"][N_KF]
    R, n_iters, seed, S = 1024, 10, 900, 43
    u = torch.rand(n_iters, R, S, generator=torch.Generator().manual_seed(2))
    of = H.oracle_field(cfg, grid_scale=0.3, seed=5)
    model = H.cuda_model(cfg, H.state_of(of))
    pts = _probe_points(cfg["mapping"]["bound"])
    out0, _ = _probe(model, of, pts)
    mapper = FusedMapper(model)
    losses = mapper.first_frame_mapping(room["dev"], n_iters, c2w=None if pose == "identity" else c2w.cuda(), pix_num=R, seed=seed,
                                        u=u.cuda()).cpu().numpy()
    ref = oinit.first_frame_mapping(of, [oinit.frame_batch(room["frame"], R, seed + i) for i in range(n_iters)], c2w, u=u).numpy()
    out1, ref1 = _probe(model, of, pts)
    from mipsfusion_b200 import _lib as L
    assert L.lib().mf_tc_check_error() == 0
    lerr = float(np.max(np.abs(losses[:, :4] - ref) / np.abs(ref)))
    ferr, moved = H.rel_err(out1, ref1), H.rel_err(out1, out0)
    print(f"\n  {pose}: losses max rel diff {lerr:.1e}; field after {n_iters} iterations rel err {ferr:.1e} (moved {moved:.1e})")
    np.testing.assert_allclose(losses[:, :4], ref, rtol=5e-3)
    assert ferr < 5e-3, ferr
    assert moved > 1e-3, moved
    assert np.all(losses[:, 7] > 0.5 * R)


@pytest.mark.parametrize("initial", ["saved", "constructor"])
def test_new_submap_after_recover_initial_param(room, initial):
    """A trained model, ``recover_initial_param()`` and a new FusedMapper follow the oracle run from the initial parameters.
    "saved": ``save_initial_param()`` after loading a state with a visible grid; "constructor": the parameters JointEncoding drew
    at construction (grid U(-1e-4, 1e-4)), where nearly every grid gradient is ~0 and Adam's first steps move each touched
    element by about lr in a direction rounding decides (section 2 of DESIGN.md): the field is held to 1e-2 there."""
    from mipsfusion_b200.mapper import FusedMapper
    from oracle import submap_init as oinit
    cfg = _cfg(CAM_BOUND)
    R, n_iters, seed, S = 1024, 10, 77, 43
    model = H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5)))
    if initial == "saved":
        model.save_initial_param()
    FusedMapper(model).first_frame_mapping(room["dev"], 3, pix_num=R, seed=1)          # the previous submap's training
    model.recover_initial_param()
    init = {k: v.detach().cpu().clone() for k, v in model.initial_dict.items()}
    u = torch.rand(n_iters, R, S, generator=torch.Generator().manual_seed(3))
    losses = FusedMapper(model).first_frame_mapping(room["dev"], n_iters, pix_num=R, seed=seed, u=u.cuda()).cpu().numpy()
    of = H.oracle_field(cfg, state=init)
    ref = oinit.first_frame_mapping(of, [oinit.frame_batch(room["frame"], R, seed + i) for i in range(n_iters)], torch.eye(4), u=u).numpy()
    out1, ref1 = _probe(model, of, _probe_points(CAM_BOUND))
    ferr = H.rel_err(out1, ref1)
    print(f"\n  new submap ({initial}): losses max rel diff {float(np.max(np.abs(losses[:, :4] - ref) / np.abs(ref))):.1e}; "
          f"field rel err {ferr:.1e}")
    np.testing.assert_allclose(losses[:, :4], ref, rtol=5e-3)
    assert ferr < (5e-3 if initial == "saved" else 1e-2), ferr


def _steady_calls(mapper, fd, c2w, u):
    """Two calls after a warm-up: no synchronising torch call, no allocation (as tests/test_gpu_track.py)."""
    for _ in range(2):
        mapper.first_frame_mapping(fd, 5, c2w=c2w, pix_num=1800, u=u)
    gc.collect()
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    n_alloc = torch.cuda.memory_stats()["allocation.all.allocated"]
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(2):
            losses = mapper.first_frame_mapping(fd, 5, c2w=c2w, pix_num=1800, u=u)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert torch.cuda.memory_stats()["allocation.all.allocated"] == n_alloc, (c2w is None, u is None)
    assert torch.cuda.memory_allocated() == before, (c2w is None, u is None)
    assert bool(torch.isfinite(losses).all())


def test_no_sync_no_allocation(room):
    from mipsfusion_b200.mapper import FusedMapper
    cfg = _cfg()
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5))))
    u = torch.rand(5, 1800, 43, device="cuda")
    for c2w, uu in ((None, None), (room["traj"][N_KF].cuda(), u)):
        _steady_calls(mapper, room["dev"], c2w, uu)


def test_edge_cases(room):
    import mipsfusion_b200 as mf
    from mipsfusion_b200.mapper import FusedMapper
    cfg = _cfg()
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5))))
    grid0, mlp0 = mapper.grid.clone(), mapper.mlp.clone()
    with pytest.raises(mf.MipsFusionB200Error, match="sample"):
        mapper.first_frame_mapping(room["dev"], 2)
    with pytest.raises(mf.MipsFusionB200Error, match="n_iters"):
        mapper.first_frame_mapping(room["dev"], -1, pix_num=64)
    mapper.model.config["mapping"]["sample"] = 64
    losses = mapper.first_frame_mapping(room["dev"], 0)
    assert losses.shape == (0, 8)
    assert torch.equal(mapper.grid, grid0) and torch.equal(mapper.mlp, mlp0) and mapper.step_count == 0
    losses = mapper.first_frame_mapping(room["dev"], 2, seed=5)                        # pix_num from config["mapping"]["sample"]
    assert losses.shape == (2, 8) and bool(torch.isfinite(losses).all()) and mapper.step_count == 2
    assert not torch.equal(mapper.grid, grid0)


# ---- local_ba with the current frame drawn every iteration ----------------------------------------------------------------
def _ba_fixture(room, seed=1):
    """A keyframe ray store of N_KF synthetic keyframes (30 x 40 rays each, rendered at the stored lattice), their poses with a
    perturbation, and the full-resolution current frame (room, pose traj[N_KF])."""
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    cfg = _cfg()
    cfg["training"]["perturb"] = 0
    cfg["sampling"] = {"kf_n_rays_h": 30, "kf_n_rays_w": 40}
    dirs = room["frame"]["direction"]
    st = mf.KeyframeRayStore(cfg, dirs.shape[0], dirs.shape[1], N_KF, "cuda")
    lat = dirs[st.row_indices.cpu(), st.col_indices.cpu()].reshape(30, 40, 3).contiguous()
    traj = room["traj"]
    for k in range(N_KF):
        st.rays[k].copy_(synth.frame_rays(synth.render_frame(traj[k], lat, seed=k)))
        st.frame_ids.append(k)
    poses = traj.clone()
    poses[1:, :3, 3] += 0.01 * torch.randn(N_KF, 3, generator=torch.Generator().manual_seed(seed))
    return cfg, st, poses.contiguous()


def test_local_ba_cur_frame_equals_cur_rays7(room):
    from mipsfusion_b200 import sampling_helper as sh
    from mipsfusion_b200.mapper import FusedMapper
    cfg, st, poses = _ba_fixture(room)
    fd = room["dev"]
    Hh, W = fd["depth"].shape
    state = H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5))
    n_cur, pix, related = 600, 512, list(range(N_KF))
    keys = torch.randn(1, Hh * W, generator=torch.Generator().manual_seed(8)).abs().cuda()
    hp = dict(n_iters=1, pose_accum_step=5, lr_rot=1e-3, lr_trans=1e-3, optim_cur=True, seed=55)
    m1 = FusedMapper(H.cuda_model(cfg, state))
    _, la = m1.local_ba(st, 0, related, poses.cuda(), pix, cur_frame=fd, n_cur=n_cur, cur_keys=keys, **hp)
    rows, cols = sh.sample_pixels_mix(Hh, W, 16, 24, fd["depth"], n_cur, keys=keys[0])
    px = rows * W + cols
    cur = torch.cat([fd["direction"].reshape(-1, 3)[px], fd["rgb"].reshape(-1, 3)[px], fd["depth"].reshape(-1, 1)[px]], 1).contiguous()
    m2 = FusedMapper(H.cuda_model(cfg, state))
    _, lb = m2.local_ba(st, 0, related, poses.cuda(), pix, cur_rays7=cur, **hp)
    np.testing.assert_array_equal(la.cpu().numpy(), lb.cpu().numpy())
    assert torch.equal(m1._bufs[("store", pix, n_cur)]["rays7"], m2._bufs[("store", pix, n_cur)]["rays7"])


@pytest.mark.parametrize("impl", ["fp32", "tc"])
def test_local_ba_cur_frame_vs_oracle(room, impl):
    from mipsfusion_b200.mapper import FusedMapper
    from oracle import ba as oba
    from oracle import submap_init as oinit
    cfg, st, poses = _ba_fixture(room, seed=1)
    fd = room["dev"]
    Hh, W = fd["depth"].shape
    n_cur, pix, n_iters, seed, K = 512, 512, 15, 1234, N_KF + 1
    related = list(range(N_KF))
    keys = torch.randn(n_iters, Hh * W, generator=torch.Generator().manual_seed(9)).abs()
    store = st.rays.cpu()
    batches = [oba.store_batch(store, 0, related, pix, seed + 3 * i, oinit.cur_frame_rays(room["frame"], n_cur, keys[i]))
               for i in range(n_iters)]
    of0 = H.oracle_field(cfg, grid_scale=0.3, seed=5)
    ref = oba.local_ba(H.oracle_field(cfg, grid_scale=0.3, seed=5), batches, poses, 5, 1e-3, 1e-3, True)
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(of0)))
    mapper.pose_grad_impl = impl
    p, losses = mapper.local_ba(st, 0, related, poses.cuda(), pix, n_iters=n_iters, pose_accum_step=5, lr_rot=1e-3, lr_trans=1e-3,
                                optim_cur=True, seed=seed, cur_frame=fd, n_cur=n_cur, cur_keys=keys.cuda())
    p, losses = p.cpu(), losses.cpu().numpy()
    from mipsfusion_b200 import _lib as L
    assert L.lib().mf_tc_check_error() == 0
    err = float((p - ref["poses"]).abs().max())
    rel = np.abs(losses[:, :4] - ref["losses"].numpy()) / np.abs(ref["losses"].numpy())
    print(f"\n  cur_frame ({impl}): per term max rel diff (rgb, depth, sdf, fs) {['%.1e' % v for v in rel.max(0)]}, "
          f"per iteration {['%.0e' % v for v in rel.max(1)]}")
    print(f"  cur_frame ({impl}): losses max rel diff {float(np.max(np.abs(losses[:, :4] - ref['losses'].numpy()) / np.abs(ref['losses'].numpy()))):.1e}; "
          f"poses after {n_iters} iterations max abs diff {err:.1e} (oracle moved them by {float((ref['poses'] - poses).abs().max()):.1e})")
    np.testing.assert_allclose(losses[:, :4], ref["losses"].numpy(), rtol=5e-3)
    assert err <= 5e-4, err
    assert torch.equal(p[0], poses[0])


def test_local_ba_cur_frame_arguments_and_device_keys(room):
    import mipsfusion_b200 as mf
    from mipsfusion_b200.mapper import FusedMapper
    cfg, st, poses = _ba_fixture(room)
    fd = room["dev"]
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5))))
    args = (st, 0, list(range(N_KF)), poses.cuda(), 512)
    hp = dict(n_iters=6, pose_accum_step=3, lr_rot=1e-3, lr_trans=1e-3, optim_cur=False)
    with pytest.raises(mf.MipsFusionB200Error, match="n_cur"):
        mapper.local_ba(*args, cur_frame=fd, n_cur=16 * 24 - 1, **hp)
    with pytest.raises(mf.MipsFusionB200Error, match="n_cur"):
        mapper.local_ba(*args, cur_frame=fd, n_cur=16 * 24 + 4097, **hp)
    with pytest.raises(mf.MipsFusionB200Error, match="not both"):
        mapper.local_ba(*args, cur_rays7=st.rays[0, :64].contiguous(), cur_frame=fd, n_cur=512, **hp)
    mapper.local_ba(*args, cur_frame=fd, n_cur=16 * 24 + 4096, seed=1, **hp)                # the largest draw (warm-up)
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        p, losses = mapper.local_ba(*args, cur_frame=fd, n_cur=16 * 24 + 4096, seed=2, **hp)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert bool(torch.isfinite(losses).all()) and bool(torch.isfinite(p).all())
    assert float(losses[:, 7].min()) > 0
