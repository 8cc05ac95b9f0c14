"""Gradient pose refinement of tracking -- the "GO" loop of reference MIPSFusion.tracking_render (mipsfusion.py:501-556) --
as a fixed sequence of kernels on persistent buffers: no autograd graph, no allocation, no host synchronisation inside the loop.

Per iteration: pose parameters (quaternion + translation, get_pose_param_optim :235-241) -> c2w (qt_to_transform_matrix,
geometry_helper.py:11-17) -> rays (:531-532) -> z sampling -> fused field forward -> render + losses -> their backward ->
field backward producing ONLY the ray gradients (the reference also back-propagates into the frozen model and discards it,
Appendix C of SURVEY.md) -> ray generation backward -> d loss / d c2w -> quaternion / translation gradient + Adam step, with
the reference's best-loss bookkeeping (:540-552) on the device.  The early exit after ``wait_iters`` non-improving iterations
becomes a device flag that freezes the pose (later iterations are no-ops on the state), so the returned pose is the reference's.

``JointEncoding.forward`` + ``loss.backward()`` + ``torch.optim.Adam`` on the pose parameters stays available as the drop-in
route (the reference loop runs unchanged on it); this class is the fast route."""
import ctypes as C

import torch

from . import _lib as L
from . import dist as D
from .decoder import _Workspace


def matrix_to_quaternion(m):
    """pytorch3d.transforms.matrix_to_quaternion for one (3,3) rotation (the reference's ``matrix_to_tensor``), real part
    first, standardised to a non-negative real part.  Host-side set-up of the pose parameters (published formula)."""
    m = m.detach().to("cpu", torch.float32)
    m00, m01, m02, m10, m11, m12, m20, m21, m22 = [m[i, j] for i in range(3) for j in range(3)]
    q_abs = torch.stack([1.0 + m00 + m11 + m22, 1.0 + m00 - m11 - m22, 1.0 - m00 + m11 - m22, 1.0 - m00 - m11 + m22]).clamp_min(0).sqrt()
    cand = torch.stack([torch.stack([q_abs[0] ** 2, m21 - m12, m02 - m20, m10 - m01]),
                        torch.stack([m21 - m12, q_abs[1] ** 2, m10 + m01, m02 + m20]),
                        torch.stack([m02 - m20, m10 + m01, q_abs[2] ** 2, m12 + m21]),
                        torch.stack([m10 - m01, m20 + m02, m21 + m12, q_abs[3] ** 2])])
    cand = cand / (2.0 * q_abs[:, None].clamp_min(0.1))
    q = cand[int(torch.argmax(q_abs))]
    return -q if q[0] < 0 else q


class FusedPoseRefiner:
    def __init__(self, model, lr_rot=None, lr_trans=None, wait_iters=None, use_best=None, backward="tc"):
        """backward: "tc" -- tensor-core backward that produces only the ray gradients (fast; pose gradients 2.4e-4 against the
        oracle, DESIGN.md 2); "fp32" -- CUDA-core backward (the parity route of the drop-in module: 5e-7)."""
        self.model = model
        self.backward = backward
        cfg = model.config
        self.dev = model._device
        trk = cfg.get("tracking", {})
        self.lr_rot = float(trk.get("lr_rot", 1e-3) if lr_rot is None else lr_rot)
        self.lr_trans = float(trk.get("lr_trans", 1e-3) if lr_trans is None else lr_trans)
        self.wait_iters = int(trk.get("wait_iters", 100) if wait_iters is None else wait_iters)
        self.use_best = bool(trk.get("best", True) if use_best is None else use_best)
        t = cfg["training"]
        self.loss_w = torch.tensor([t["rgb_weight"], t["depth_weight"], t["sdf_weight"], t["fs_weight"]], dtype=torch.float32, device=self.dev)
        self._bufs = {}
        self.launches = 0

    def _buffers(self, R, S):
        b = self._bufs.get((R, S))
        if b is None:
            f32 = dict(device=self.dev, dtype=torch.float32)
            b = dict(state=torch.zeros(32, **f32), c2w=torch.zeros(1, 4, 4, **f32), d_c2w=torch.zeros(1, 4, 4, **f32),
                     best=torch.zeros(4, 4, **f32), o=torch.empty(R, 3, **f32), d=torch.empty(R, 3, **f32),
                     d_o=torch.empty(R, 3, **f32), d_d=torch.empty(R, 3, **f32), z=torch.empty(R, S, **f32),
                     counts=torch.empty(2, device=self.dev, dtype=torch.int64), raw=torch.empty(R, S, L.MF_RAW_DIM, **f32),
                     d_raw=torch.empty(R, S, L.MF_RAW_DIM, **f32), rgb=torch.empty(R, 3, **f32), depth=torch.empty(R, **f32),
                     losses=torch.zeros(8, **f32), scratch=torch.empty(R * 8, **f32), u=torch.empty(R, S, **f32),
                     feat=torch.empty(int(L.lib().mf_feat_cache_size(R * S)), device=self.dev, dtype=torch.uint8))
            self._bufs[(R, S)] = b
        return b

    def refine(self, c2w_init, rays_d_cam, target_rgb, target_d, n_iter, u=None, EMD_w=0.0, graph=None):
        """c2w_init (4,4); rays_d_cam (N,3) camera-frame directions, target_rgb (N,3), target_d (N,) or (N,1): device tensors of
        the pixels sampled once for the whole loop (:512-522).  u: optional (n_iter, N, S) stratified-jitter draws.
        -> (c2w (4,4) device tensor: the best pose if ``use_best`` else the reference's `c2w_est`, state tensor).  No synchronisation.

        graph (default: on when ``u`` is None): the whole loop -- n_iter x 15 launches -- is captured once per (N, S, n_iter,
        weights buffers) as a CUDA graph on static input buffers and replayed; the loop is launch-bound (15 kernels of 5-120 us
        per iteration against ~165 us of host time to issue them)."""
        dev = self.dev
        R = rays_d_cam.shape[0]
        b, cfg, lins, field, fb, S = self._setup(R, EMD_w)
        b["in_dirs"].copy_(rays_d_cam.reshape(R, 3), non_blocking=True)
        b["in_rgb"].copy_(target_rgb.reshape(R, 3), non_blocking=True)
        b["in_d"].copy_(target_d.reshape(R), non_blocking=True)
        c2w0 = torch.as_tensor(c2w_init).detach().to("cpu", torch.float32)
        init = torch.zeros(32)
        init[0:4] = matrix_to_quaternion(c2w0[:3, :3]); init[4:7] = c2w0[:3, 3]; init[22] = -1.0
        b["state"].copy_(init.to(dev, non_blocking=True))
        n_iter = int(n_iter)
        use_graph = (u is None) if graph is None else bool(graph)
        if use_graph and u is None and n_iter > 0 and not self.__dict__.get("_graph_off", False):
            key = self._graph_key(R, S, n_iter, EMD_w, cfg, field, fb)
            g = b.get("graph")
            if g is None or g[0] != key:
                try:
                    self._loop(b, cfg, lins, field, fb, R, S, 1, None)          # eager warm-up: lazy allocations, function attributes
                    b["state"].copy_(init.to(dev, non_blocking=True))
                    torch.cuda.current_stream(dev).synchronize()
                    cg = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(cg):
                        self._loop(b, cfg, lins, field, fb, R, S, n_iter, None)
                    g = b["graph"] = (key, cg, (field._keepalive, fb._keepalive))
                    b["state"].copy_(init.to(dev, non_blocking=True))            # (the capture itself does not run anything)
                except Exception as e:                                            # capture not possible here: stay on the eager loop
                    self.__dict__["_graph_off"] = True
                    self.__dict__["_graph_error"] = repr(e)
                    g = None
                    b.pop("graph", None)
                    b["state"].copy_(init.to(dev, non_blocking=True))
            if g is not None:
                g[1].replay()
                self.launches += 15 * n_iter
                return (b["best"], b["state"]) if self.use_best else (b["c2w"][0], b["state"])
        self._loop(b, cfg, lins, field, fb, R, S, n_iter, u)
        if self.use_best and n_iter > 0:
            return b["best"], b["state"]
        # tracking.best = False: the reference hands back `c2w_est`, the matrix it formed at the START of the last executed
        # iteration (mipsfusion.py:544,562-563) -- the last Adam step is never evaluated.  b["c2w"] holds exactly that matrix.
        if n_iter <= 0:
            L.call("mf_pose_to_c2w", L.ptr(b["state"]), L.ptr(b["c2w"]), L.stream())
        return b["c2w"][0], b["state"]

    def _setup(self, R, EMD_w):
        """Static buffers of an R-pixel loop (input copies included) and the current field descriptors (map steps in between
        are picked up).  -> (buffers, render cfg, linspaces, forward field, backward field, S)."""
        model, dev = self.model, self.dev
        cfg, lins = model._render_cfg(True, EMD_w, dev)
        S = cfg.n_samples_d + cfg.n_range_d
        b = self._buffers(R, S)
        field = model._field()
        if "in_dirs" not in b:
            f32 = dict(device=dev, dtype=torch.float32)
            b["in_dirs"], b["in_rgb"], b["in_d"] = torch.empty(R, 3, **f32), torch.empty(R, 3, **f32), torch.empty(R, **f32)
            b["ws"] = torch.empty(int(L.lib().mf_field_bwd_workspace_size(R * S, 1)), **f32)
        if self.backward == "fp32":                    # the fp32 kernel always forms the parameter gradients: give it a sink
            fb = model._field(impl=1)
            if "sink" not in b:
                b["sink"] = (torch.zeros_like(model.embed_fn.params.data), torch.zeros(L.MF_MLP_PARAMS, device=dev, dtype=torch.float32))
        else:
            fb = field
        return b, cfg, lins, field, fb, S

    def _graph_key(self, R, S, n_iter, EMD_w, cfg, field, fb):
        """What a captured loop depends on beyond its static buffers."""
        return (R, S, n_iter, float(EMD_w), self.backward, field.grid, field.mlp_prep, fb.mlp_prep, int(cfg.perturb))

    def _loop(self, b, cfg, lins, field, fb, R, S, n_iter, u):
        """n_iter iterations of the 15-launch sequence on the static buffers of ``b`` (current stream: also the capture stream)."""
        dev = self.dev
        st = L.stream()
        rays_d_cam, target_rgb, target_d, ws = b["in_dirs"], b["in_rgb"], b["in_d"], b["ws"]
        if self.backward == "fp32":
            gg, gm, feat_b = b["sink"][0], b["sink"][1], None
        else:
            gg, gm, feat_b = None, None, b["feat"]
        for it in range(int(n_iter)):
            L.call("mf_pose_to_c2w", L.ptr(b["state"]), L.ptr(b["c2w"]), st)
            L.call("mf_gen_rays", L.ptr(rays_d_cam), L.ptr(b["c2w"]), None, L.ptr(b["o"]), L.ptr(b["d"]), R, 1, st)
            uu = None
            if cfg.perturb:
                uu = b["u"].uniform_() if u is None else L.f32c(u[it], dev)
            L.call("mf_sample_z", L.ptr(target_d), L.ptr(uu), L.ptr(lins[0]), L.ptr(lins[1]), L.ptr(lins[2]), C.byref(cfg),
                   L.ptr(b["z"]), L.ptr(b["counts"]), R, st)
            L.call("mf_field_query_rays", L.ptr(b["o"]), L.ptr(b["d"]), L.ptr(b["z"]), C.byref(field), L.ptr(b["raw"]), L.ptr(b["feat"]), R, S, st)
            L.call("mf_render_loss_fwd", L.ptr(b["raw"]), L.ptr(b["z"]), L.ptr(target_rgb), L.ptr(target_d), L.ptr(b["counts"]),
                   C.byref(cfg), L.ptr(b["rgb"]), L.ptr(b["depth"]), None, None, None, L.ptr(b["losses"]), L.ptr(b["scratch"]), R, S, st)
            L.call("mf_render_loss_bwd", L.ptr(b["raw"]), L.ptr(b["z"]), L.ptr(target_rgb), L.ptr(target_d), L.ptr(b["counts"]),
                   L.ptr(b["losses"]), C.byref(cfg), L.ptr(self.loss_w), None, None, L.ptr(b["d_raw"]), R, S, st)
            L.call("mf_field_query_rays_bwd", L.ptr(b["o"]), L.ptr(b["d"]), L.ptr(b["z"]), C.byref(fb), L.ptr(b["d_raw"]),
                   L.ptr(feat_b), L.ptr(gg), L.ptr(gm), L.ptr(b["d_o"]), L.ptr(b["d_d"]), L.ptr(ws), R, S, st)
            b["d_c2w"].zero_()
            L.call("mf_gen_rays_bwd", L.ptr(rays_d_cam), None, L.ptr(b["d_o"]), L.ptr(b["d_d"]), L.ptr(b["d_c2w"]), R, 1, st)
            L.call("mf_pose_refine_update", L.ptr(b["state"]), L.ptr(b["c2w"]), L.ptr(b["d_c2w"]), L.ptr(b["losses"]), L.ptr(self.loss_w),
                   self.lr_rot, self.lr_trans, self.wait_iters, L.ptr(b["best"]), st)
            self.launches += 15


class FusedTracker:
    """The reference's per-frame tracking (MIPSFusion.tracking_render, mipsfusion.py:470-576, after the pose prediction) as one
    device-resident call: RandomOptimizer iterations from the predicted pose (:483-485), the hand-off of its pose to the gradient
    stage (:501-503, ``mf_track_handoff``), the GO pixel draw (uniform lattice + random valid pixels, :512-522) and the GO loop
    (:501-556).  No host synchronisation: the caller's ``c2w.cpu()`` is the frame's only sync.

    ro: a single-rank :class:`RandomOptimizer` (its sharded exchange passes a host-side sequence number per iteration, which a
    captured graph would freeze; use ``ro.optimize`` for sharded RO).  refiner: the GO stage, ``FusedPoseRefiner(model)`` by
    default (its ``use_best``, learning rates, patience and backward apply)."""
    LATTICE = (16, 24)                 # the GO draw's uniform lattice (mipsfusion.py:512-515)

    def __init__(self, model, ro, refiner=None):
        if D.world(ro.group)[0] > 1:
            raise L.MipsFusionB200Error("FusedTracker: the RandomOptimizer is sharded over a process group; tracking runs on one "
                                        "rank (use RandomOptimizer.optimize for sharded RO)")
        self.model, self.ro = model, ro
        self.refiner = FusedPoseRefiner(model) if refiner is None else refiner
        self.dev = model._device
        self._bufs = {}

    def _hp(self, v, key):
        if v is not None:
            return v
        trk = self.model.config.get("tracking", {})
        if key not in trk:
            raise L.MipsFusionB200Error("FusedTracker: %s not given and config['tracking'] has no '%s'" % (key, key))
        return trk[key]

    def _buffers(self, H, W, n_ro, R, S, n_go):
        key = (H, W, n_ro, R, S, n_go)
        tb = self._bufs.get(key)
        if tb is None:
            dev, ro = self.dev, self.ro
            f32 = dict(device=dev, dtype=torch.float32)
            i64 = dict(device=dev, dtype=torch.int64)
            lh, lw = self.LATTICE
            P = ro.row_indices.shape[0]
            lat = [ro._lattice(off) for off in range(min(n_ro, 5))]
            tb = self._bufs[key] = dict(
                depth=torch.empty(H, W, **f32), rgb=torch.empty(H, W, 3, **f32), init=torch.empty(4, 4, **f32),
                rot=torch.empty(3, 3, **f32), trans=torch.empty(3, **f32), search=torch.empty(6, **f32),
                lat=[(ih * W + iw).contiguous() for ih, iw, _ in lat], lat_dirs=[d for _, _, d in lat], target_d=torch.empty(P, **f32),
                ro_info=torch.zeros(n_ro, 4, device=dev, dtype=torch.int32),
                ro_better=torch.zeros(n_ro, ro.pre_sampled_particle.shape[0], device=dev, dtype=torch.uint8),
                ro_pose=torch.empty(4, 4, **f32), keys=torch.empty(H * W, **f32),
                topk_ws=torch.empty(int(L.lib().mf_topk_workspace_size(H * W)), device=dev, dtype=torch.uint8),
                idx=torch.empty(max(R - lh * lw, 0), **i64), rows=torch.empty(R, **i64), cols=torch.empty(R, **i64),
                flat=torch.empty(R, **i64), u=torch.empty(n_go, R, S, **f32))
        return tb

    def _sequence(self, tb, b, cfg, lins, field, fb, R, S, n_ro, n_go, draw_keys, draw_u):
        """Steps 2-7 of :meth:`track` on the static buffers (current stream: also the capture stream)."""
        ro, model, rf = self.ro, self.model, self.refiner
        st = L.stream()
        H, W = tb["depth"].shape
        tb["rot"].copy_(tb["init"][:3, :3])
        tb["trans"].copy_(tb["init"][:3, 3])
        tb["search"].fill_(float(ro.scaling_coefficient1))
        depth_flat = tb["depth"].view(-1)
        for i in range(n_ro):                                        # RandomOptimizer.optimize's loop, lattice shift i % 5
            torch.index_select(depth_flat, 0, tb["lat"][i % 5], out=tb["target_d"])
            ro.iterate(model, tb["rot"], tb["trans"], tb["search"], tb["target_d"], tb["lat_dirs"][i % 5],
                       better=tb["ro_better"][i], info=tb["ro_info"][i])
        L.call("mf_track_handoff", L.ptr(tb["rot"]), L.ptr(tb["trans"]), L.ptr(tb["ro_pose"]), L.ptr(b["state"]), st)
        if n_go <= 0:
            return
        if draw_keys:
            tb["keys"].normal_().abs_()
        lh, lw = self.LATTICE
        L.call("mf_sample_pixels_topk", L.ptr(tb["depth"]), L.ptr(tb["keys"]), H, W, lh, lw, R, L.ptr(tb["idx"]), L.ptr(tb["rows"]),
               L.ptr(tb["cols"]), L.ptr(tb["topk_ws"]), st)
        torch.mul(tb["rows"], W, out=tb["flat"]).add_(tb["cols"])
        torch.index_select(ro.rays_dir.view(-1, 3), 0, tb["flat"], out=b["in_dirs"])
        torch.index_select(tb["rgb"].view(-1, 3), 0, tb["flat"], out=b["in_rgb"])
        torch.index_select(depth_flat, 0, tb["flat"], out=b["in_d"])
        rf._loop(b, cfg, lins, field, fb, R, S, n_go, None if draw_u else tb["u"])

    @torch.no_grad()
    def track(self, depth, rgb, init_pose, n_iter_ro=None, n_iter_go=None, keys=None, u=None, graph=None):
        """depth (H,W), rgb (H,W,3), init_pose (4,4): device tensors; init_pose is the predicted pose handed to RO.
        n_iter_ro / n_iter_go: ``config["tracking"]`` keys iter_RO / iter unless given; the GO pixel count is
        ``config["tracking"]["sample"]`` (on the 16 x 24 lattice).  keys (H*W): optional pixel-draw keys (abs(randn) drawn on the
        device when None); u (n_iter_go, N, S): optional stratified-jitter draws (uniform on the device when None).
        graph (default on): the whole sequence is captured once per key as a CUDA graph and replayed; explicit draws are copied
        into its static buffers first.  graph=False runs the same sequence eagerly.

        -> (c2w (4,4), info) device tensors, overwritten by the next call of the same shape: c2w is the refiner's result
        (best pose if ``use_best``, else the pose the last GO iteration started from), the RO pose when n_iter_go == 0; info:
        ro_info (n_iter_ro, 4) and ro_better (n_iter_ro, C) as RandomOptimizer.last_info / last_better, ro_pose (4,4),
        go_state (32), rows / cols (N) int64: the GO pixels (not drawn when n_iter_go == 0).  With n_iter_ro == 0 the GO stage
        starts from init_pose.  No host synchronisation; no allocation after the first call for a key."""
        n_ro, n_go = int(self._hp(n_iter_ro, "iter_RO")), int(self._hp(n_iter_go, "iter"))
        R = int(self._hp(None, "sample"))
        if n_ro < 0 or n_go < 0:
            raise L.MipsFusionB200Error("FusedTracker: iteration counts must be >= 0")
        rf = self.refiner
        H, W = depth.shape
        b, cfg, lins, field, fb, S = rf._setup(R, 0.0)
        tb = self._buffers(H, W, n_ro, R, S, n_go)
        tb["depth"].copy_(depth)
        tb["rgb"].copy_(rgb)
        tb["init"].copy_(init_pose)
        if keys is not None:
            tb["keys"].copy_(keys.reshape(-1))
        if u is not None:
            tb["u"].copy_(u)
        draw_keys, draw_u = keys is None, u is None
        args = (tb, b, cfg, lins, field, fb, R, S, n_ro, n_go, draw_keys, draw_u)
        if (True if graph is None else bool(graph)) and not self.__dict__.get("_graph_off", False):
            ro = self.ro
            key = (rf._graph_key(R, S, n_go, 0.0, cfg, field, fb), H, W, n_ro, draw_keys, draw_u, ro.pre_sampled_particle.data_ptr(),
                   float(ro.scaling_coefficient1), float(ro.scaling_coefficient2), float(ro.trunc_value), ro.rays_dir.data_ptr(),
                   rf.lr_rot, rf.lr_trans, rf.wait_iters)
            g = tb.get("graph")
            if g is None or g[0] != key:
                g = None
                tb.pop("graph", None)
                try:
                    self._sequence(*args)                              # eager warm-up: lazy allocations of every stage
                    torch.cuda.current_stream(self.dev).synchronize()
                    cg = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(cg):
                        self._sequence(*args)
                    g = tb["graph"] = (key, cg, (field._keepalive, fb._keepalive))
                except Exception as e:                                  # capture not possible here: stay on the eager sequence
                    self.__dict__["_graph_off"] = True
                    self.__dict__["_graph_error"] = repr(e)
            if g is not None:
                g[1].replay()
                return self._result(tb, b, n_go)
        self._sequence(*args)
        return self._result(tb, b, n_go)

    def _result(self, tb, b, n_go):
        info = dict(ro_info=tb["ro_info"], ro_better=tb["ro_better"], ro_pose=tb["ro_pose"], go_state=b["state"], rows=tb["rows"],
                    cols=tb["cols"])
        if n_go <= 0:
            return tb["ro_pose"], info
        return (b["best"] if self.refiner.use_best else b["c2w"][0]), info
