"""Deterministic mode (mipsfusion_b200.set_deterministic): the hash-grid gradient by fixed-point accumulation equals the numpy
restatement (oracle/det_scatter.py) bit for bit and does not depend on the point order; the map step, the pose-gradient step,
tracking and the drop-in autograd route repeat bit for bit; the four-role backward is refused.  Every test restores the switch
state it found."""
import contextlib
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers as H

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def det_mode(on=True, pdl=None):
    from mipsfusion_b200 import _lib as L
    prev, prev_pdl = L.lib().mf_get_deterministic(), L.lib().mf_get_pdl()
    L.call("mf_set_deterministic", 1 if on else 0)
    if pdl is not None:
        L.call("mf_set_pdl", 1 if pdl else 0)
    try:
        yield
    finally:
        L.call("mf_set_deterministic", prev)
        L.call("mf_set_pdl", prev_pdl)


def _bits(t):
    return t.detach().cpu().contiguous().numpy().view(np.uint32)


@pytest.mark.parametrize("T", [19, 12])
def test_hashgrid_bwd_equals_oracle_bitwise_and_order_independent(T):
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200.encodings import grid_meta
    from oracle import det_scatter as ds
    from oracle import hashgrid as hg
    table = hg.level_table(T)
    meta = grid_meta(T, 16, 2, 16, hg.per_level_scale_of())
    rng = np.random.default_rng(T)
    N = 20000
    x = rng.uniform(-0.1, 1.1, size=(N, 3)).astype(np.float32)          # dense, hashed and wrapping cells
    dy = (rng.standard_normal((N, 32)) * np.exp2(rng.integers(-10, 4, size=(N, 32)))).astype(np.float32)
    dy[rng.random((N, 32)) < 0.2] = 0.0
    g0 = (rng.standard_normal(table["n_params"]) * 1e-3).astype(np.float32)
    ref = ds.fixed_point_sum(*ds.contributions(x, dy, table), ds.headroom(N), g0)[0]
    grid = torch.zeros(table["n_params"], device="cuda")

    def run(perm):
        g = torch.from_numpy(g0).cuda()
        xs, ys = torch.from_numpy(x[perm]).cuda(), torch.from_numpy(dy[perm]).cuda()
        L.call("mf_hashgrid_bwd", L.ptr(xs), L.ptr(ys), L.ptr(grid), C.byref(meta), L.ptr(g), None, N, L.stream())
        torch.cuda.synchronize()
        return g.cpu().numpy()

    with det_mode():
        a = run(np.arange(N))
        b = run(rng.permutation(N))
    assert np.array_equal(a.view(np.uint32), ref.view(np.uint32)), int(np.sum(a.view(np.uint32) != ref.view(np.uint32)))
    assert np.array_equal(b.view(np.uint32), a.view(np.uint32))
    assert int(L.lib().mf_det_workspace_bytes()) > 0
    with det_mode(False):                                                # the atomic scatter agrees to fp32 rounding
        c = run(np.arange(N))
    np.testing.assert_allclose(c, a, rtol=1e-5, atol=1e-6 * float(np.abs(a).max()))


def _map_run(cfg, state, batch, steps, det, pdl=None):
    from mipsfusion_b200.mapper import FusedMapper
    with det_mode(det, pdl):
        mapper = FusedMapper(H.cuda_model(cfg, state))
        ro, rd, rgb, d, u = batch
        losses = [mapper.step(ro, rd, rgb, d, u=u).clone() for _ in range(steps)]
        torch.cuda.synchronize()
    out = {"losses": torch.stack(losses).cpu().numpy()}
    for k in ("g_grid", "grid", "g_mlp", "mlp"):
        out[k] = getattr(mapper, k).cpu().numpy().copy()
    return out


def test_map_steps_bitwise_reproducible():
    cfg = H.make_config(16, n_samples_d=32, n_range_d=11)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=7)
    state = H.state_of(of)
    rays_o, rays_d, rgb, d, u = H.synth_batch(2048, 43, seed=11)
    batch = tuple(t.cuda().contiguous() for t in (rays_o, rays_d, rgb, d.reshape(-1), u))
    a = _map_run(cfg, state, batch, 25, True, pdl=True)
    b = _map_run(cfg, state, batch, 25, True, pdl=True)
    c = _map_run(cfg, state, batch, 25, True, pdl=False)
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), k
        assert a[k].tobytes() == c[k].tobytes(), (k, "PDL on / off")
    # one step against the default (atomic) mode: the bars of test_gpu_map_glue
    one_det = _map_run(cfg, state, batch, 1, True)
    one_def = _map_run(cfg, state, batch, 1, False)
    for k in ("losses", "g_mlp", "mlp"):
        assert one_det[k].tobytes() == one_def[k].tobytes(), k
    for k in ("g_grid", "grid"):
        np.testing.assert_allclose(one_det[k], one_def[k], rtol=1e-5, atol=1e-7 * max(1.0, float(np.abs(one_def[k]).max())), err_msg=k)


@pytest.mark.parametrize("impl", ["tc", "fp32"])
def test_pose_gradient_step_bitwise_reproducible(impl):
    from mipsfusion_b200.mapper import FusedMapper
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_gpu_mapper_pose import _multi_pose_batch
    cfg = H.make_config(14, n_samples_d=32, n_range_d=11)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=5)
    rays7, pose_idx, poses, _ = _multi_pose_batch(1024, 6, seed=21)
    outs = []
    with det_mode():
        for _ in range(2):
            mapper = FusedMapper(H.cuda_model(cfg, H.state_of(of)))
            mapper.pose_grad_impl = impl
            torch.manual_seed(17)                                        # step_host draws the sample jitter on the device
            losses, d_poses = mapper.step_host(rays7.pin_memory(), pose_idx.pin_memory(), poses.cuda(), pose_grad=True)
            torch.cuda.synchronize()
            outs.append((_bits(losses), _bits(d_poses), _bits(mapper.grid), _bits(mapper.mlp)))
    for a, b, name in zip(outs[0], outs[1], ("losses", "d_poses", "grid", "mlp")):
        assert np.array_equal(a, b), (impl, name)


def test_tracker_graph_equals_eager_bitwise():
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import synth
    import test_gpu_track as T
    cfg = T._config()
    of = H.oracle_field(cfg, grid_scale=0.3, seed=13)
    model = H.cuda_model(cfg, H.state_of(of))
    dirs = synth.camera_rays()
    c2w = synth.trajectory(4)[1]
    frame = synth.render_frame(c2w, dirs)
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(3)
    fx = type("F", (), {})()
    fx.depth, fx.rgb = frame["depth"].to(dev), frame["rgb"].to(dev)
    init = c2w.clone(); init[:3, 3] += torch.tensor([0.01, -0.008, 0.006]); init = init.to(dev)
    keys = torch.randn(460 * 620, generator=g).abs().to(dev)
    u = torch.rand(T.N_GO, T.N_PX, 75, generator=g).to(dev)
    with det_mode():
        refiner = mf.FusedPoseRefiner(model)
        tracker = mf.FusedTracker(model, T._ro(cfg, dirs, dev), refiner)
        cg, ig = T._track(tracker, fx, init, T.N_RO, T.N_GO, keys, u, graph=True)
        ce, ie = T._track(tracker, fx, init, T.N_RO, T.N_GO, keys, u, graph=False)
        ce2, ie2 = T._track(tracker, fx, init, T.N_RO, T.N_GO, keys, u, graph=False)
        assert "_graph_error" not in tracker.__dict__, tracker.__dict__.get("_graph_error")
    assert torch.equal(ce, ce2) and torch.equal(ie["go_state"], ie2["go_state"])
    assert torch.equal(cg, ce) and torch.equal(ig["go_state"], ie["go_state"])


@pytest.mark.parametrize("rays_grad", [False, True])
def test_autograd_route_bitwise_reproducible(rays_grad):
    """Drop-in route: JointEncoding.forward + loss.backward() (tensor-core backward; with rays.requires_grad the fp32 one)."""
    cfg = H.make_config(16, n_samples_d=32, n_range_d=11)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=9)
    rays_o, rays_d, rgb, d, u = H.synth_batch(1024, 43, seed=3)
    grads = []
    with det_mode():
        for _ in range(2):
            model = H.cuda_model(cfg, H.state_of(of))
            ro, rd = rays_o.cuda(), rays_d.cuda()
            if rays_grad:
                ro.requires_grad_(True); rd.requires_grad_(True)
            ret = model(ro, rd, rgb.cuda(), d.cuda(), u=u.cuda())
            t = cfg["training"]
            (t["rgb_weight"] * ret["rgb_loss"] + t["sdf_weight"] * ret["sdf_loss"] + t["fs_weight"] * ret["fs_loss"]).backward()
            torch.cuda.synchronize()
            gs = [_bits(p.grad) for p in model.parameters() if p.grad is not None]
            if rays_grad:
                gs += [_bits(ro.grad), _bits(rd.grad)]
            grads.append(gs)
    assert len(grads[0]) >= 2
    for a, b in zip(*grads):
        assert np.array_equal(a, b)


def test_four_role_backward_is_refused():
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200.mapper import FusedMapper
    cfg = H.make_config(14, n_samples_d=32, n_range_d=11)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=7)
    rays_o, rays_d, rgb, d, u = H.synth_batch(512, 43, seed=11)
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(of)))
    try:
        L.call("mf_set_bwd_impl", 3)
        with det_mode(), pytest.raises(L.MipsFusionB200Error, match="four-role"):
            mapper.step(rays_o.cuda(), rays_d.cuda(), rgb.cuda(), d.reshape(-1).cuda(), u=u.cuda())
    finally:
        L.call("mf_set_bwd_impl", 0)
    torch.cuda.synchronize()


def test_captured_map_step_replays_equal_to_eager_without_allocation():
    """After an eager warm-up: eager steps neither allocate nor synchronise the host; a captured step replays bitwise equal to
    the eager step.  (The Adam step count is a launch argument, fixed at capture: the replay is compared after ONE replay, as
    the second eager step; a second replay's losses -- computed before its update -- are compared with the third step's.)"""
    from mipsfusion_b200.mapper import FusedMapper
    cfg = H.make_config(16, n_samples_d=32, n_range_d=11)
    of = H.oracle_field(cfg, grid_scale=0.3, seed=7)
    state = H.state_of(of)
    rays_o, rays_d, rgb, d, u = H.synth_batch(2048, 43, seed=11)
    batch = tuple(t.cuda().contiguous() for t in (rays_o, rays_d, rgb, d.reshape(-1), u))
    with det_mode():
        eager = FusedMapper(H.cuda_model(cfg, state))
        le = [eager.step(*batch[:4], u=batch[4]).clone()]
        held = torch.empty(2, 8, device="cuda")
        torch.cuda.synchronize()
        n_alloc = torch.cuda.memory_stats()["allocation.all.allocated"]
        torch.cuda.set_sync_debug_mode("error")
        try:
            held[0].copy_(eager.step(*batch[:4], u=batch[4]))
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert torch.cuda.memory_stats()["allocation.all.allocated"] == n_alloc
        grid2 = _bits(eager.grid).copy()
        held[1].copy_(eager.step(*batch[:4], u=batch[4]))
        torch.cuda.synchronize()
        le += [held[0], held[1]]
        cap = FusedMapper(H.cuda_model(cfg, state))
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            lc = [cap.step(*batch[:4], u=batch[4]).clone()]              # warm-up on the capturing stream
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                out = cap.step(*batch[:4], u=batch[4])
            g.replay()
            lc.append(out.clone())
            s.synchronize()
            grid_cap = _bits(cap.grid).copy()
            g.replay()
            lc.append(out.clone())
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
    for a, b in zip(le, lc):
        assert torch.equal(a, b)
    assert grid2.tobytes() == grid_cap.tobytes()


def _oracle_curve(det, n):
    """n map steps (deterministic mode or the default) and the oracle's loop on the same draws: (device losses, oracle losses)."""
    from mipsfusion_b200.mapper import FusedMapper
    from oracle import adam as oadam
    cfg = H.make_config(12, n_samples_d=32, n_range_d=11)
    of = H.oracle_field(cfg, seed=7)
    R, S = 256, 43
    rays_o, rays_d, rgb, d, _ = H.synth_batch(R, S, seed=11)
    g = torch.Generator().manual_seed(11)
    mapper = FusedMapper(H.cuda_model(cfg, H.state_of(of)))
    opt_o = oadam.make_optimizer(of)
    dargs = [t.cuda().contiguous() for t in (rays_o, rays_d, rgb, d)]
    lo, ld = [], []
    with det_mode(det):
        for _ in range(n):
            u = torch.rand(R, S, generator=g)
            opt_o.zero_grad()
            ret_o = of.forward(rays_o, rays_d, rgb, d, u)
            of.total_loss(ret_o).backward()
            opt_o.step()
            lo.append([float(ret_o[k]) for k in ("rgb_loss", "depth_loss", "sdf_loss", "fs_loss")])
            ld.append(mapper.step(*dargs, u=u.cuda())[:4].cpu().numpy().copy())
    return np.array(ld), np.array(lo)


def test_map_steps_follow_the_oracle():
    """25 deterministic map steps against the oracle's loop on the same draws.  DESIGN §2's loss-curve bar (rtol 5e-3 over the
    first 12 steps, test_gpu_scene) holds; over all 25 steps the drift from the oracle -- fp32 / tensor-core rounding
    compounded by Adam -- is no larger than the default mode's on the same run (within a factor 2 per loss term)."""
    ld, lo = _oracle_curve(True, 25)
    np.testing.assert_allclose(ld[:12], lo[:12], rtol=5e-3)
    ld0, _ = _oracle_curve(False, 25)
    dev_det, dev_def = np.abs(ld - lo).max(0), np.abs(ld0 - lo).max(0)
    print(f"\n  max |device - oracle| over 25 steps per loss term: deterministic {dev_det}, default {dev_def}")
    assert np.all(dev_det <= 2 * dev_def + 1e-7), (dev_det, dev_def)


def _two_runs(fn):
    """fn() twice in deterministic mode, torch's generators seeded identically before each (the steps draw their sample
    jitter on the device when no explicit draw is given)."""
    outs = []
    with det_mode():
        for _ in range(2):
            torch.manual_seed(23)
            outs.append({k: _bits(v) for k, v in fn().items()})
            torch.cuda.synchronize()
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k
    return outs[0]


@pytest.mark.parametrize("impl", ["tc", "fp32"])
def test_local_ba_with_pose_steps_bitwise_reproducible(impl):
    from mipsfusion_b200.mapper import FusedMapper
    from test_gpu_bundle_adjust import _store_fixture
    cfg, st, poses, cur = _store_fixture(8, seed=1)
    state = H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5))
    hp = dict(n_iters=10, pose_accum_step=5, lr_rot=1e-3, lr_trans=1e-3, optim_cur=True, seed=1234)

    def run():
        m = FusedMapper(H.cuda_model(cfg, state))
        m.pose_grad_impl = impl
        p, losses = m.local_ba(st, 0, list(range(8)), poses.cuda(), 1024 - 64, cur_rays7=cur, **hp)
        return {"poses": p, "losses": losses, "grid": m.grid, "mlp": m.mlp}
    out = _two_runs(run)
    assert not np.array_equal(out["poses"], _bits(poses))                  # the pose steps moved the poses


def _room():
    from mipsfusion_b200 import synth
    import test_gpu_first_frame_mapping as F
    traj = synth.trajectory(F.N_KF + 1)
    fr = synth.render_frame(traj[F.N_KF], synth.camera_rays(), seed=3)
    frame = {k: fr[k].contiguous() for k in ("direction", "rgb", "depth")}
    return dict(frame=frame, dev={k: v.cuda() for k, v in frame.items()}, traj=traj.to(torch.float32).contiguous())


def test_local_ba_with_current_frame_draw_and_first_frame_mapping_bitwise_reproducible():
    """local_ba drawing the current frame's pixels on the device (top-k draw, cur_frame) and first_frame_mapping (frame draw)."""
    from mipsfusion_b200.mapper import FusedMapper
    import test_gpu_first_frame_mapping as F
    room = _room()
    cfg, st, poses = F._ba_fixture(room)
    state = H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=5))
    hp = dict(n_iters=10, pose_accum_step=5, lr_rot=1e-3, lr_trans=1e-3, optim_cur=True, seed=55)

    def ba():
        m = FusedMapper(H.cuda_model(cfg, state))
        p, losses = m.local_ba(st, 0, list(range(F.N_KF)), poses.cuda(), 512, cur_frame=room["dev"], n_cur=600, **hp)
        return {"poses": p, "losses": losses, "grid": m.grid, "mlp": m.mlp}
    _two_runs(ba)

    c2w = room["traj"][F.N_KF].cuda()

    def init():
        m = FusedMapper(H.cuda_model(cfg, state))
        losses = m.first_frame_mapping(room["dev"], 10, c2w=c2w, pix_num=1800, seed=31)
        return {"losses": losses, "grid": m.grid, "mlp": m.mlp}
    _two_runs(init)


def test_step_from_store_pose_gradients_bitwise_reproducible():
    from mipsfusion_b200.mapper import FusedMapper
    from test_gpu_bundle_adjust import _store_fixture
    cfg, st, poses, cur = _store_fixture(3)
    state = H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=2))

    def run():
        m = FusedMapper(H.cuda_model(cfg, state))
        losses, d_poses = m.step_from_store(st, 0, [0, 1, 2], poses.cuda(), 256, cur_rays7=cur, seed=77, pose_grad=True)
        return {"losses": losses, "d_poses": d_poses, "grid": m.grid, "mlp": m.mlp}
    _two_runs(run)


def test_pose_refiner_bitwise_reproducible_and_graph_equals_eager():
    import mipsfusion_b200 as mf
    import test_gpu_track as T
    cfg = T._config()
    model = H.cuda_model(cfg, H.state_of(H.oracle_field(cfg, grid_scale=0.3, seed=13)))
    R, n_iter = 500, 10
    rays7, _, poses, g = H.synth_batch_packed(R, seed=31)
    start = poses[0].clone()
    start[:3, 3] += torch.tensor([0.01, -0.008, 0.006])
    u = torch.rand(n_iter, R, 75, generator=g).cuda()
    args = (start.cuda(), rays7[:, :3].cuda().contiguous(), rays7[:, 3:6].cuda().contiguous(), rays7[:, 6].cuda().contiguous(), n_iter)
    outs = []
    with det_mode():
        refiner = mf.FusedPoseRefiner(model)
        for graph in (False, False, True):
            c2w, state = refiner.refine(*args, u=u, graph=graph)
            outs.append((_bits(c2w).copy(), _bits(state).copy()))
    for o in outs[1:]:
        assert np.array_equal(o[0], outs[0][0]) and np.array_equal(o[1], outs[0][1])


def test_workspace_growth_under_capture_is_an_error():
    """A stream that has not run this mode before has no workspace: the first call under capture is refused, not faulted."""
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200.encodings import grid_meta
    from oracle import hashgrid as hg
    table = hg.level_table(12)
    meta = grid_meta(12, 16, 2, 16, hg.per_level_scale_of())
    N = 1000
    x = torch.rand(N, 3, device="cuda")
    dy = torch.randn(N, 32, device="cuda")
    grid = torch.zeros(table["n_params"], device="cuda")
    grad = torch.zeros_like(grid)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with det_mode():
        with torch.cuda.stream(s):
            gr.capture_begin()
            try:
                rc = L.lib().mf_hashgrid_bwd(L.ptr(x), L.ptr(dy), L.ptr(grid), C.byref(meta), L.ptr(grad), None, N, s.cuda_stream)
                msg = L.lib().mf_last_error().decode()
            finally:
                gr.capture_end()
    torch.cuda.synchronize()
    assert rc != 0 and "capture" in msg, (rc, msg)
    with det_mode():                                                     # outside capture the same call grows the workspace and runs
        with torch.cuda.stream(s):
            L.call("mf_hashgrid_bwd", L.ptr(x), L.ptr(dy), L.ptr(grid), C.byref(meta), L.ptr(grad), None, N, s.cuda_stream)
    torch.cuda.synchronize()
    assert float(grad.abs().sum()) > 0
