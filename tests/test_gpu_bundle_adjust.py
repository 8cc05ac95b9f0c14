"""Local bundle adjustment on the device (FusedMapper.local_ba, the reference's MIPSFusion.local_BA, mipsfusion.py:259-370):
the two pose kernels against torch autograd + torch.optim.Adam, the store-fed step's pose gradients against the host route,
the whole loop against the CPU oracle (oracle/ba.py), and the data-parallel loop on two GPUs."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers as H

pytestmark = pytest.mark.gpu


def _ulp_ok(a, b, n=1):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(np.all(np.abs(a - b) <= n * np.spacing(np.maximum(np.abs(a), np.abs(b)))))


def test_ba_pose_kernels_vs_torch_adam():
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200 import synth
    from mipsfusion_b200.tracker import matrix_to_quaternion
    from oracle.tracking import qt_to_transform_matrix
    K, lr_rot, lr_trans = 51, 1e-3, 2e-3
    poses = synth.trajectory(K).to(torch.float32).contiguous()
    frozen = torch.zeros(K, dtype=torch.uint8)
    frozen[0] = frozen[50] = 1
    opt_ids = [k for k in range(K) if not frozen[k]]
    dev = torch.device("cuda")
    state, out = torch.full((K, 24), 7.0, device=dev), torch.empty(K, 4, 4, device=dev)
    poses_d, frozen_d = poses.to(dev), frozen.to(dev)
    L.call("mf_ba_pose_init", L.ptr(poses_d), L.ptr(frozen_d), K, L.ptr(state), L.ptr(out), L.stream())
    s = state.cpu()
    q_ref = torch.stack([matrix_to_quaternion(poses[k, :3, :3]) for k in opt_ids])
    assert _ulp_ok(s[opt_ids, :4].numpy(), q_ref.numpy()), np.abs(s[opt_ids, :4].numpy() - q_ref.numpy()).max()
    assert torch.equal(s[opt_ids, 4:7], poses[opt_ids, :3, 3]) and float(s[:, 7:].abs().max()) == 0.0
    rot = torch.nn.Parameter(s[opt_ids, :4].clone()); trans = torch.nn.Parameter(s[opt_ids, 4:7].clone())
    opt = torch.optim.Adam([{"params": rot, "lr": lr_rot}, {"params": trans, "lr": lr_trans}])
    np.testing.assert_array_equal(out.cpu()[frozen.bool()].numpy(), poses[frozen.bool()].numpy())
    assert H.rel_err(out.cpu()[opt_ids], qt_to_transform_matrix(rot, trans).detach()) < 1e-6
    g = torch.Generator().manual_seed(12)
    for it in range(3):
        d = torch.randn(K, 4, 4, generator=g) * (10.0 ** (it - 1))
        d_dev = d.to(dev)
        L.call("mf_ba_pose_update", L.ptr(state), L.ptr(d_dev), L.ptr(frozen_d), K, lr_rot, lr_trans, L.ptr(out), L.stream())
        (qt_to_transform_matrix(rot, trans)[:, :3, :] * d[opt_ids, :3, :]).sum().backward()
        opt.step(); opt.zero_grad()
        s, o = state.cpu(), out.cpu()
        assert float(d_dev.abs().max()) == 0.0
        m = torch.cat([opt.state[rot]["exp_avg"], opt.state[trans]["exp_avg"]], 1)
        v = torch.cat([opt.state[rot]["exp_avg_sq"], opt.state[trans]["exp_avg_sq"]], 1)
        errs = dict(q=H.rel_err(s[opt_ids, :4], rot.detach()), t=H.rel_err(s[opt_ids, 4:7], trans.detach()),
                    m=H.rel_err(s[opt_ids, 7:14], m), v=H.rel_err(s[opt_ids, 14:21], v),
                    poses=H.rel_err(o[opt_ids], qt_to_transform_matrix(rot, trans).detach()))
        print(f"\n  pose update {it + 1}: " + ", ".join(f"{k} {e:.1e}" for k, e in errs.items()))
        assert max(errs.values()) <= 1e-6, errs
        assert np.all(s[opt_ids, 21].numpy() == it + 1)
        np.testing.assert_array_equal(o[frozen.bool()].numpy(), poses[frozen.bool()].numpy())
        assert float(s[frozen.bool()].abs().max()) == 0.0
    assert L.lib().mf_tc_check_error() == 0


def _store_fixture(n_kf, hw=(30, 40), seed=0):
    """A keyframe ray store of ``n_kf`` synthetic frames, their poses + a perturbed current-frame pose, current-frame rays."""
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    cfg = H.make_config(14, n_samples_d=32, n_range_d=11)
    cfg["training"]["perturb"] = 0
    cfg["sampling"] = {"kf_n_rays_h": hw[0], "kf_n_rays_w": hw[1]}
    dirs = synth.camera_rays()
    traj = synth.trajectory(n_kf + 1)
    st = mf.KeyframeRayStore(cfg, dirs.shape[0], dirs.shape[1], n_kf, "cuda")
    for kf in range(n_kf):
        fr = synth.render_frame(traj[kf], dirs, seed=kf)
        st.add_keyframe({"direction": dirs, "rgb": fr["rgb"], "depth": fr["depth"], "frame_id": kf})
    g = torch.Generator().manual_seed(seed)
    poses = traj.to(torch.float32).clone()
    poses[1:, :3, 3] += 0.01 * torch.randn(n_kf, 3, generator=g)           # something for the pose steps to correct
    cur = st.rays[n_kf - 1, ::7][:64].clone()
    return cfg, st, poses.contiguous(), cur


def test_store_fed_pose_gradients_equal_host_route():
    from mipsfusion_b200.mapper import FusedMapper
    cfg, st, poses, cur = _store_fixture(3)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=2)
    related = [0, 1, 2]
    P = poses.cuda()
    m1 = FusedMapper(H.cuda_model(cfg, H.state_of(of)))
    la, da = m1.step_from_store(st, 0, related, P, 256, cur_rays7=cur, seed=77, pose_grad=True)
    la, da = la.cpu().numpy().copy(), da.cpu().numpy().copy()
    rays, _, kidx = st.sample_rays_in_submap(0, related, 256, seed=77)
    rays7 = torch.cat([rays, cur], 0).cpu().contiguous()
    idx = torch.cat([kidx.cpu(), -torch.ones(cur.shape[0], dtype=torch.int64)])
    m2 = FusedMapper(H.cuda_model(cfg, H.state_of(of)))
    lb, db = m2.step_host(rays7.pin_memory(), idx.pin_memory(), P, pose_grad=True)
    np.testing.assert_array_equal(la, lb.numpy())
    err = H.rel_err(da, db.cpu().numpy())
    print(f"\n  store-fed vs host pose gradients: rel err {err:.1e}")
    assert float(np.abs(db.cpu().numpy()).max()) > 0 and err <= 1e-6, err
    from mipsfusion_b200 import _lib as L
    assert L.lib().mf_tc_check_error() == 0


def _qt(P):
    """(K,4,4) -> (K,7) quaternion + translation (the oracle's matrix_to_quaternion)."""
    from oracle.shims.pytorch3d.transforms import matrix_to_quaternion
    P = torch.as_tensor(P, dtype=torch.float32)
    return torch.cat([matrix_to_quaternion(P[:, :3, :3]), P[:, :3, 3]], 1)


def _compare_first_step(dev_pose, ref, opt_ids, label):
    """2e-5 on the (q, t) components whose accumulated oracle gradient exceeds 1e-3 of the largest of its pose."""
    a, b = _qt(dev_pose)[opt_ids], _qt(ref["step_poses"][0])[opt_ids]
    g = ref["step_grads"][0].abs()
    keep = g > 1e-3 * g.max(1, keepdim=True).values
    d = (a - b).abs()
    print(f"\n  {label}: first pose step |dq,dt| max {float(d[keep].max()):.1e} on {int(keep.sum())} components, "
          f"{int((~keep).sum())} below the gradient margin (max {float(d[~keep].max()) if (~keep).any() else 0.0:.1e})")
    assert float(d[keep].max()) <= 2e-5


@pytest.mark.parametrize("impl,optim_cur", [("fp32", False), ("tc", True)])
def test_local_ba_vs_oracle_loop(impl, optim_cur):
    from mipsfusion_b200.mapper import FusedMapper
    from oracle import ba as oba
    cfg, st, poses, cur = _store_fixture(8, seed=1)
    of0 = H.oracle_field(cfg, grid_scale=0.3, seed=5)
    related, K, pix, n_iters, seed = list(range(8)), 9, 1024 - 64, 15, 1234
    hp = dict(pose_accum_step=5, lr_rot=1e-3, lr_trans=1e-3, optim_cur=optim_cur, seed=seed)
    store = st.rays.cpu()
    batches = [oba.store_batch(store, 0, related, pix, seed + 3 * i, cur.cpu()) for i in range(n_iters)]
    of = H.oracle_field(cfg, grid_scale=0.3, seed=5)
    ref = oba.local_ba(of, batches, poses, 5, 1e-3, 1e-3, optim_cur)
    opt_ids = list(range(1, K)) if optim_cur else list(range(1, K - 1))
    # after the first pose step
    m5 = FusedMapper(H.cuda_model(cfg, H.state_of(of0)))
    m5.pose_grad_impl = impl
    p5, _ = m5.local_ba(st, 0, related, poses.cuda(), pix, cur_rays7=cur, n_iters=5, **hp)
    _compare_first_step(p5.cpu(), ref, opt_ids, impl)
    # the whole loop
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(of0)))
    mapper.pose_grad_impl = impl
    p, losses = mapper.local_ba(st, 0, related, poses.cuda(), pix, cur_rays7=cur, n_iters=n_iters, **hp)
    p, losses = p.cpu(), losses.cpu().numpy()
    from mipsfusion_b200 import _lib as L
    assert L.lib().mf_tc_check_error() == 0
    err = float((p - ref["poses"]).abs().max())
    moved = float((ref["poses"] - poses).abs().max())
    print(f"  {impl}: losses max rel diff {float(np.max(np.abs(losses[:, :4] - ref['losses'].numpy()) / np.abs(ref['losses'].numpy()))):.1e}; "
          f"poses after {n_iters} iterations max abs diff {err:.1e} (oracle moved them by {moved:.1e})")
    np.testing.assert_allclose(losses[:, :4], ref["losses"].numpy(), rtol=5e-3)
    assert err <= 5e-4, err
    assert torch.equal(p[0], poses[0])
    assert torch.equal(p[K - 1], poses[K - 1]) != optim_cur


def test_local_ba_hyper_parameters_come_from_config_or_raise():
    from mipsfusion_b200.mapper import FusedMapper
    import mipsfusion_b200 as mf
    cfg, st, poses, cur = _store_fixture(3)
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, seed=1))))
    with pytest.raises(mf.MipsFusionB200Error, match="pose_accum_step"):
        mapper.local_ba(st, 0, [0, 1, 2], poses.cuda(), 128, n_iters=2, lr_rot=1e-3, lr_trans=1e-3, optim_cur=False)
    mapper.model.config["mapping"].update(iters=4, pose_accum_step=2, lr_rot=1e-3, lr_trans=1e-3, optim_cur=False)
    p, losses = mapper.local_ba(st, 0, [0, 1, 2], poses.cuda(), 128, cur_rays7=cur, seed=3)
    n_alloc = len(mapper._bufs)
    p2, losses2 = mapper.local_ba(st, 0, [0, 1, 2], poses.cuda(), 128, cur_rays7=cur, seed=3)
    assert losses.shape == (4, 8) and p2.data_ptr() == p.data_ptr() and len(mapper._bufs) == n_alloc
    assert torch.equal(p2.cpu()[0], poses[0]) and torch.equal(p2.cpu()[3], poses[3])


def _ba_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from mipsfusion_b200.mapper import FusedMapper
    cfg, st, poses, cur = _store_fixture(8, seed=1)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=5)
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(of)), group=dist.group.WORLD)
    p, _ = mapper.local_ba(st, 0, list(range(8)), poses.to(dev), 512 - 64, cur_rays7=cur.to(dev), n_iters=15, pose_accum_step=5,
                           lr_rot=1e-3, lr_trans=1e-3, optim_cur=True, seed=4321)
    torch.cuda.synchronize()
    same = []
    for t in (p, mapper.grid, mapper.mlp):
        t = t.detach().contiguous()
        gathered = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        same.append(all(bool(torch.equal(x, gathered[0])) for x in gathered))
    if rank == 0:
        np.savez(out, poses=p.cpu().numpy(), same=np.array(same), store=st.rays.cpu().numpy(), cur=cur.cpu().numpy(),
                 init=poses.numpy())
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_local_ba_data_parallel_on_two_gpus(tmp_path):
    """Each rank draws its own rays; poses, grid and decoder stay bitwise equal across the ranks, and the result follows the
    oracle loop fed with both ranks' draws concatenated (the batch the two ranks together train on)."""
    import torch.multiprocessing as mp
    from oracle import ba as oba
    out = str(tmp_path / "ba.npz")
    mp.spawn(_ba_worker, args=(2, 29651, out), nprocs=2, join=True)
    r = np.load(out)
    assert r["same"].all(), r["same"]
    store, cur = torch.from_numpy(r["store"]), torch.from_numpy(r["cur"])
    batches = []
    for i in range(15):
        parts = [oba.store_batch(store, 0, list(range(8)), 512 - 64, 4321 + 3 * (i * 2 + k), cur) for k in range(2)]
        batches.append((torch.cat([parts[0][0], parts[1][0]]), torch.cat([parts[0][1], parts[1][1]])))
    cfg = H.make_config(14, n_samples_d=32, n_range_d=11)
    cfg["training"]["perturb"] = 0
    ref = oba.local_ba(H.oracle_field(cfg, grid_scale=0.3, seed=5), batches, torch.from_numpy(r["init"]), 5, 1e-3, 1e-3, True)
    err = float(np.abs(r["poses"] - ref["poses"].numpy()).max())
    print(f"\n  2 GPUs vs oracle on the concatenated draws: poses max abs diff {err:.1e}")
    assert err <= 5e-4, err
