"""FusedTracker (RandomOptimizer -> hand-off -> pixel draw -> GO loop in one device-resident call) against the composed route
the reference consumes (RandomOptimizer.optimize + sample_pixels_mix + FusedPoseRefiner.refine), at the reference's tracking
shape: 620 x 460 frame, 2000 particles x 16 x 24 lattice, GO 1000 pixels x 75 samples."""
import gc
import math
import os
import types

import numpy as np
import pytest
import torch

import helpers as H

pytestmark = pytest.mark.gpu

N_PX, N_RO, N_GO = 1000, 5, 10


def _config():
    cfg = H.make_config(16, n_samples_d=50, n_range_d=25)
    cfg["tracking"] = {"RO": {"particle_size": 2000, "initial_scaling_factor": 0.02, "rescaling_factor": 0.5, "n_rows": 16, "n_cols": 24},
                       "ignore_edge_W": 20, "ignore_edge_H": 20, "lr_rot": 1e-3, "lr_trans": 1e-3, "wait_iters": 100, "best": True,
                       "iter_RO": N_RO, "iter": N_GO, "sample": N_PX}
    return cfg


def _ro(cfg, dirs, dev, group=None):
    import mipsfusion_b200 as mf
    ds = types.SimpleNamespace(H=460, W=620, fx=320.0, fy=320.0, cx=309.5, cy=229.5, rays_d=dirs)
    g = torch.Generator().manual_seed(5)
    particles = torch.randn(2000, 6, generator=g).clamp(-2, 2)
    particles[0] = 0
    return mf.RandomOptimizer(cfg, types.SimpleNamespace(dataset=ds, device=str(dev)), particles=particles, group=group)


@pytest.fixture(scope="module")
def fx():
    from mipsfusion_b200 import synth
    dev = torch.device("cuda", 0)
    cfg = _config()
    of = H.oracle_field(cfg, grid_scale=0.3, seed=13)
    model = H.cuda_model(cfg, H.state_of(of))
    dirs = synth.camera_rays()
    c2w = synth.trajectory(4)[1]
    frame = synth.render_frame(c2w, dirs)
    d = torch.eye(4)
    d[:3, 3] = torch.tensor([0.01, -0.008, 0.006])
    ang = 0.01
    d[:3, :3] = torch.tensor([[1.0, -ang, 0.0], [ang, 1.0, 0.0], [0.0, 0.0, 1.0]]) / (1 + ang * ang) ** 0.5
    d[2, 2] = 1.0
    g = torch.Generator().manual_seed(3)
    S = 75
    return types.SimpleNamespace(dev=dev, cfg=cfg, model=model, ro=_ro(cfg, dirs, dev), dirs=dirs.to(dev),
                                 depth=frame["depth"].to(dev), rgb=frame["rgb"].to(dev), init=(c2w @ d).to(dev),
                                 keys=torch.randn(460 * 620, generator=g).abs().to(dev), u=torch.rand(N_GO, N_PX, S, generator=g).to(dev),
                                 keys2=torch.randn(460 * 620, generator=g).abs().to(dev), u2=torch.rand(N_GO, N_PX, S, generator=g).to(dev))


def _composed(fx, refiner, init, n_ro, n_go, keys, u):
    """The composed route as bench.py's frame does it: RO pose on the host, pixel draw, GO from that pose."""
    from mipsfusion_b200 import sampling_helper as sh
    pose = fx.ro.optimize(fx.model, fx.depth, init.cpu(), init.cpu(), n_iter=n_ro)
    rows, cols = sh.sample_pixels_mix(460, 620, 16, 24, fx.depth, N_PX, keys=keys)
    c2w, state = refiner.refine(pose.to(fx.dev), fx.dirs[rows, cols], fx.rgb[rows, cols], fx.depth[rows, cols], n_go, u=u[:n_go])
    info = (fx.ro.last_info.clone(), torch.stack(fx.ro.last_better)) if n_ro > 0 else None
    return dict(pose=pose, info=info, rows=rows, cols=cols, c2w=c2w.clone(), state=state.clone())


def _track(tracker, fx, init, n_ro, n_go, keys, u, graph=None):
    c2w, info = tracker.track(fx.depth, fx.rgb, init, n_iter_ro=n_ro, n_iter_go=n_go, keys=keys, u=u[:n_go], graph=graph)
    return c2w.clone(), {k: v.clone() for k, v in info.items()}


def _ulps(a, b):
    """Distance in units in the last place between two float32 arrays (same-sign ordering)."""
    def ordered(x):
        i = np.ascontiguousarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7fffffff), i)
    return np.abs(ordered(a) - ordered(b))


def test_ro_stage_and_pixels_match_composed_route(fx):
    import mipsfusion_b200 as mf
    refiner = mf.FusedPoseRefiner(fx.model)
    tracker = mf.FusedTracker(fx.model, fx.ro, refiner)
    ref = _composed(fx, refiner, fx.init, N_RO, N_GO, fx.keys, fx.u)
    c2w, info = _track(tracker, fx, fx.init, N_RO, N_GO, fx.keys, fx.u)
    torch.cuda.synchronize()
    assert "_graph_error" not in tracker.__dict__, tracker.__dict__.get("_graph_error")
    assert torch.equal(info["ro_pose"].cpu(), ref["pose"])
    assert torch.equal(info["ro_info"], ref["info"][0])
    assert torch.equal(info["ro_better"], ref["info"][1])
    assert int(info["ro_info"][:, 1].sum()) > 0                       # (RO moved the pose at least once)
    assert torch.equal(info["rows"], ref["rows"]) and torch.equal(info["cols"], ref["cols"])
    err = float((c2w - ref["c2w"]).abs().max())
    print(f"\n  track vs composed route after {N_GO} GO iterations: max abs diff {err:.2e}")
    assert err <= 5e-4


def test_handoff_matches_host_init(fx):
    """go_state after the hand-off (n_iter_go = 0) against refine's host set-up of the same RO pose."""
    import mipsfusion_b200 as mf
    refiner = mf.FusedPoseRefiner(fx.model)
    tracker = mf.FusedTracker(fx.model, fx.ro, refiner)
    ref = _composed(fx, refiner, fx.init, N_RO, 0, fx.keys, fx.u)
    _, info = _track(tracker, fx, fx.init, N_RO, 0, fx.keys, fx.u)
    st, host = info["go_state"].cpu(), ref["state"].cpu()
    assert torch.equal(st[4:], host[4:])                              # translation, moments, step count, flags
    assert float(st[22]) == -1.0 and float(st[23]) == 0.0 and float(st[24]) == 0.0
    ul = _ulps(st[:4].numpy(), host[:4].numpy())
    print(f"\n  hand-off quaternion: {int((ul > 0).sum())} of 4 components differ from the host set-up (max {int(ul.max())} ulp)")
    assert ul.max() <= 1


def _rotations():
    """Random rotations, rotations within 1e-6..1e-1 rad of a half turn about random axes, and the exact half turns about the
    coordinate axes: every branch of matrix_to_quaternion's argmax."""
    g = torch.Generator().manual_seed(11)
    q = torch.randn(200, 4, generator=g, dtype=torch.float64)
    ax = torch.randn(150, 3, generator=g, dtype=torch.float64)
    ax = ax / ax.norm(dim=1, keepdim=True)
    ang = math.pi - 10.0 ** (-1 - 5 * torch.rand(150, generator=g, dtype=torch.float64))
    q2 = torch.cat([torch.cos(ang / 2)[:, None], torch.sin(ang / 2)[:, None] * ax], 1)
    q3 = torch.eye(4, dtype=torch.float64)
    q = torch.cat([q, q2, q3])
    q = q / q.norm(dim=1, keepdim=True)
    r, i, j, k = q.unbind(1)
    m = torch.stack([1 - 2 * (j * j + k * k), 2 * (i * j - k * r), 2 * (i * k + j * r),
                     2 * (i * j + k * r), 1 - 2 * (i * i + k * k), 2 * (j * k - i * r),
                     2 * (i * k - j * r), 2 * (j * k + i * r), 1 - 2 * (i * i + j * j)], 1).reshape(-1, 3, 3)
    return m.float()


def test_handoff_kernel_on_random_rotations():
    import mipsfusion_b200  # noqa: F401
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200 import tracker as T
    from mipsfusion_b200.random_optimizer import pose_compose
    rots = _rotations()
    n = rots.shape[0]
    trans = torch.randn(n, 3, generator=torch.Generator().manual_seed(12))
    dev = torch.device("cuda", 0)
    rot_d, trans_d = rots.to(dev), trans.to(dev)
    c2w = torch.full((n, 4, 4), float("nan"), device=dev)
    st = torch.full((n, 32), float("nan"), device=dev)
    for a in range(n):
        L.call("mf_track_handoff", L.ptr(rot_d[a]), L.ptr(trans_d[a]), L.ptr(c2w[a]), L.ptr(st[a]), L.stream())
    c2w, st = c2w.cpu(), st.cpu()
    branches, worst, n_diff = set(), 0, 0
    for a in range(n):
        m = rots[a]
        qa = torch.stack([1.0 + m[0, 0] + m[1, 1] + m[2, 2], 1.0 + m[0, 0] - m[1, 1] - m[2, 2], 1.0 - m[0, 0] + m[1, 1] - m[2, 2],
                          1.0 - m[0, 0] - m[1, 1] + m[2, 2]])
        branches.add(int(torch.argmax(qa.clamp_min(0).sqrt())))
        assert torch.equal(c2w[a], pose_compose(m, trans[a]))
        ul = _ulps(st[a, :4].numpy(), T.matrix_to_quaternion(m).numpy())
        worst, n_diff = max(worst, int(ul.max())), n_diff + int((ul > 0).sum())
        assert torch.equal(st[a, 4:7], trans[a])
        assert float(st[a, 22]) == -1.0 and not st[a, 7:22].any() and not st[a, 23:].any()
    print(f"\n  hand-off on {n} rotations: {n_diff} of {4 * n} quaternion components differ from the host formula, max {worst} ulp")
    assert branches == {0, 1, 2, 3}
    assert worst <= 1


@pytest.mark.parametrize("use_best,wait_iters", [(True, 100), (False, 100), (True, 0), (False, 0)])
def test_final_pose_matches_composed_route(fx, use_best, wait_iters):
    """The GO stage starts from a quaternion within 1 ulp of the host set-up; Adam turns such a start difference into
    the same divergence as two fp32 implementations (DESIGN.md 2): 2e-5 after 3 iterations, 5e-4 after 10."""
    import mipsfusion_b200 as mf
    refiner = mf.FusedPoseRefiner(fx.model, use_best=use_best, wait_iters=wait_iters)
    tracker = mf.FusedTracker(fx.model, fx.ro, refiner)
    for n_go, bar in ((3, 2e-5), (10, 5e-4)):
        ref = _composed(fx, refiner, fx.init, N_RO, n_go, fx.keys, fx.u)
        c2w, info = _track(tracker, fx, fx.init, N_RO, n_go, fx.keys, fx.u)
        err = float((c2w - ref["c2w"]).abs().max())
        st, host = info["go_state"].cpu(), ref["state"].cpu()
        print(f"\n  use_best {use_best}, wait_iters {wait_iters}, {n_go} GO iterations: pose max abs diff {err:.2e}, "
              f"steps {int(st[21])} / {int(host[21])}")
        assert err <= bar, (n_go, err)
        assert float(st[21]) == float(host[21]) and float(st[24]) == float(host[24])


def test_graph_equals_eager(fx):
    """Same explicit draws: the captured sequence and the eager one, and two replays with new draws copied in against two
    eager runs with the same draws.  The RO stage, the hand-off and the pixel draw are bitwise deterministic and asserted
    equal.  The GO stage is not bitwise reproducible even between two eager runs: d loss / d c2w is summed with float atomics
    in no fixed order (mf_gen_rays_bwd), and the tensor-core ray gradients amplify a last-bit pose difference; so the GO
    pose and parameters are held to the 10-iteration bar of DESIGN.md 2 (5e-4), the step count and stop flag exactly, and
    the spread of two eager runs is printed beside the graph / eager difference."""
    import mipsfusion_b200 as mf
    refiner = mf.FusedPoseRefiner(fx.model)
    tracker = mf.FusedTracker(fx.model, fx.ro, refiner)
    for keys, u in ((fx.keys, fx.u), (fx.keys2, fx.u2)):
        cg, ig = _track(tracker, fx, fx.init, N_RO, N_GO, keys, u, graph=True)
        ce, ie = _track(tracker, fx, fx.init, N_RO, N_GO, keys, u, graph=False)
        ce2, ie2 = _track(tracker, fx, fx.init, N_RO, N_GO, keys, u, graph=False)
        assert "_graph_error" not in tracker.__dict__, tracker.__dict__.get("_graph_error")
        for k in ("ro_info", "ro_better", "ro_pose", "rows", "cols"):
            assert torch.equal(ig[k], ie[k]) and torch.equal(ie2[k], ie[k]), k
        d_ge, d_ee = float((cg - ce).abs().max()), float((ce2 - ce).abs().max())
        print(f"\n  graph vs eager: pose bit-equal {torch.equal(cg, ce)} (max diff {d_ge:.1e}), go_state bit-equal "
              f"{torch.equal(ig['go_state'], ie['go_state'])}; two eager runs: pose max diff {d_ee:.1e}, go_state bit-equal "
              f"{torch.equal(ie2['go_state'], ie['go_state'])}")
        assert d_ge <= 5e-4 and float((ig["go_state"][:7] - ie["go_state"][:7]).abs().max()) <= 5e-4
        assert torch.equal(ig["go_state"][21], ie["go_state"][21]) and torch.equal(ig["go_state"][24], ie["go_state"][24])


def _steady_calls(tracker, fx, keys, u, graph):
    """Two calls after a warm-up: no synchronising torch call, no allocation, memory_allocated unchanged.  (A helper, so that
    no result of an earlier tracker -- views of its buffers -- stays referenced and is released inside the measured calls.)"""
    for _ in range(2):
        tracker.track(fx.depth, fx.rgb, fx.init, keys=keys, u=u, graph=graph)
    gc.collect()
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    n_alloc = torch.cuda.memory_stats()["allocation.all.allocated"]
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(2):
            c2w, _ = tracker.track(fx.depth, fx.rgb, fx.init, keys=keys, u=u, graph=graph)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert torch.cuda.memory_stats()["allocation.all.allocated"] == n_alloc, (graph, keys is None)
    assert torch.cuda.memory_allocated() == before, (graph, keys is None)
    assert bool(torch.isfinite(c2w).all())


def test_no_sync_no_allocation(fx):
    import mipsfusion_b200 as mf
    from mipsfusion_b200 import _lib as L
    for graph in (None, False):
        tracker = mf.FusedTracker(fx.model, fx.ro)
        for keys, u in ((None, None), (fx.keys, fx.u)):
            _steady_calls(tracker, fx, keys, u, graph)
        if graph is None:
            assert "_graph_error" not in tracker.__dict__, tracker.__dict__.get("_graph_error")
            assert all("graph" in tb for tb in tracker._bufs.values())
    torch.cuda.synchronize()
    assert L.lib().mf_tc_check_error() == 0


def test_zero_iteration_cases(fx):
    import mipsfusion_b200 as mf
    from mipsfusion_b200.random_optimizer import pose_compose
    refiner = mf.FusedPoseRefiner(fx.model)
    tracker = mf.FusedTracker(fx.model, fx.ro, refiner)
    # n_iter_ro = 0 (the ScanNet configs): the GO stage starts from init_pose
    c2w, info = _track(tracker, fx, fx.init, 0, 3, fx.keys, fx.u)
    assert info["ro_info"].shape == (0, 4) and info["ro_better"].shape[0] == 0
    init = fx.init.cpu()
    assert torch.equal(info["ro_pose"].cpu(), pose_compose(init[:3, :3], init[:3, 3]))
    ref = _composed(fx, refiner, fx.init, 0, 3, fx.keys, fx.u)
    err = float((c2w - ref["c2w"]).abs().max())
    print(f"\n  n_iter_ro = 0: pose after 3 GO iterations vs refine(init_pose): {err:.2e}")
    assert err <= 2e-5
    # n_iter_go = 0: the RO pose, bit for bit
    ref = _composed(fx, refiner, fx.init, N_RO, 0, fx.keys, fx.u)
    c2w, info = _track(tracker, fx, fx.init, N_RO, 0, fx.keys, fx.u)
    assert torch.equal(c2w.cpu(), ref["pose"]) and torch.equal(info["ro_pose"].cpu(), ref["pose"])


def test_missing_config_key_raises(fx):
    import mipsfusion_b200 as mf
    trk = fx.model.config["tracking"]
    tracker = mf.FusedTracker(fx.model, fx.ro)
    for key in ("iter_RO", "iter", "sample"):
        saved = trk.pop(key)
        try:
            with pytest.raises(mf.MipsFusionB200Error, match=key):
                tracker.track(fx.depth, fx.rgb, fx.init)
        finally:
            trk[key] = saved


def _sharded_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import mipsfusion_b200 as mf
        from mipsfusion_b200 import synth
        dev = torch.device("cuda", 0)
        cfg = _config()
        model = H.cuda_model(cfg, H.state_of(H.oracle_field(cfg)))
        ro = _ro(cfg, synth.camera_rays(), dev, group=dist.group.WORLD)
        try:
            mf.FusedTracker(model, ro)
            q.put((rank, "accepted"))
        except mf.MipsFusionB200Error as e:
            q.put((rank, "refused: " + str(e)))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.distributed.is_available() or not torch.distributed.is_gloo_available(),
                    reason="needs a torch.distributed build with gloo")
def test_sharded_random_optimizer_is_refused():
    """A RandomOptimizer sharded over a two-rank group (gloo: both ranks may share one GPU, nothing is launched) is refused."""
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
    out = {}
    while not q.empty():
        r, res = q.get()
        out[r] = res
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    assert sorted(out) == [0, 1] and all(v.startswith("refused") for v in out.values()), out
