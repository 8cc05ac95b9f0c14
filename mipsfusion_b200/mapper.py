"""Fused mapping step: the body of the reference's BA loops (mipsfusion.py:293-335, first_frame_mapping
:176-193, InactiveMap.local_BA :250-260) -- forward, loss, backward, Adam, zero_grad -- issued as a fixed
sequence of kernels on persistent buffers, with no autograd graph, no allocation and no host sync.

``JointEncoding.forward`` + ``loss.backward()`` + ``optimizer.step()`` stays available as the drop-in
route; this class is the fast route the online system uses once the model lives on the GPU.  With a
process group it becomes data parallel over ray batches: the global mask counts are all-reduced before
the loss (helper_functions/utils.py:43-47 uses batch-global counts) and the gradients after the backward.
"""
import ctypes as C

import torch

from . import _lib as L
from . import dist as D
from .decoder import _Workspace
from .keyframe_store import _new_seed, frame_tensors


class FusedMapper:
    def __init__(self, model, lr_decoder=None, lr_embed=None, group=None, peer_memory="auto", multicast="auto"):
        self.model = model
        cfg = model.config
        self.dev = model._device
        if self.dev.type != "cuda":
            raise L.MipsFusionB200Error("FusedMapper needs the model on a CUDA device")
        self.lr_decoder = cfg["mapping"]["lr_decoder"] if lr_decoder is None else lr_decoder
        self.lr_embed = cfg["mapping"]["lr_embed"] if lr_embed is None else lr_embed
        self.group = group
        self.world = D.world(group)[0]
        t = cfg["training"]
        # d(total loss)/d(rgb, depth, sdf, fs loss): the weights of get_loss_from_ret (mipsfusion.py:142-152)
        self.loss_w = torch.tensor([t["rgb_weight"], t["depth_weight"], t["sdf_weight"], t["fs_weight"]], dtype=torch.float32,
                                   device=self.dev)
        self.grid = model.embed_fn.params.data
        # master copy of the decoder blob while stepping, zero-padded to a multiple of 4 floats (one vectorised Adam launch)
        nm = L.MF_MLP_PARAMS
        self._mlp_pad = torch.zeros((nm + 3) // 4 * 4, device=self.dev, dtype=torch.float32)
        self._mlp_pad[:nm].copy_(model.decoder.flat_weights())
        self.mlp = self._mlp_pad[:nm]
        self.prep = torch.empty(int(L.lib().mf_mlp_prep_size()), device=self.dev, dtype=torch.float32)
        self.g_grid = torch.zeros_like(self.grid); self.m_grid = torch.zeros_like(self.grid); self.v_grid = torch.zeros_like(self.grid)
        self._g_mlp_pad = torch.zeros_like(self._mlp_pad); self.g_mlp = self._g_mlp_pad[:nm]
        self.m_mlp = torch.zeros_like(self._mlp_pad); self.v_mlp = torch.zeros_like(self._mlp_pad)
        # Data parallel with NVLink peer memory: parameters and (double-buffered) gradients live in a symmetric arena and
        # the gradient all-reduce + Adam + parameter broadcast become one sharded kernel (mf_adam_step_sharded).
        # peer_memory: True (require), False (NCCL all-reduce + replicated Adam), "auto" (try, fall back to NCCL).
        self.arena = None
        self.multicast = multicast                                   # "auto": from 4 GPUs on; True / False: force
        if self.world > 1 and peer_memory:
            try:
                self._init_peer_arena()
            except Exception as e:                                   # no P2P / symmetric memory on this box
                if peer_memory is True:
                    raise
                import warnings
                warnings.warn("FusedMapper: peer memory unavailable (%s); using NCCL all-reduce" % (e,))
                self.arena = None
        if self.world > 1 and self.dev.type == "cuda":
            L.call("mf_set_sm_reserve", 1)                           # room for the count all-reduce beside the forward (step())
        self.step_count = 0
        self.pose_grad_impl = "tc"       # "tc": tensor-core backward (pose gradients 2.4e-4 vs the oracle), "fp32": CUDA cores (5e-7)
        self._bufs = {}
        self.timing = None            # optional dict name -> (start_event, end_event) lists
        self.launches = 0
        with torch.cuda.device(self.dev):
            L.call("mf_mlp_prepare", L.ptr(self.mlp), L.ptr(self.prep), L.stream())
        self._bind_module()

    def _bind_module(self):
        """The module's ten decoder nn.Parameters become views of the flat master copy the Adam kernel steps, and
        ``decoder.prepared()`` hands out this mapper's kernel-layout image: after every mapping step RandomOptimizer.score,
        JointSubmapQuery, JointEncoding.forward and state_dict() all see the stepped grid AND the stepped decoder."""
        dec, o = self.model.decoder, 0
        ps = dec.ordered_params()
        with torch.no_grad():
            for p in ps:
                n = p.numel()
                p.data = self.mlp[o:o + n].view(p.shape)
                o += n
        self._seen_versions = tuple(p._version for p in ps)
        dec.__dict__.pop("_prep_cache", None)
        dec.__dict__["_ext_prep"] = (tuple(p.data_ptr() for p in ps), self)

    def _init_peer_arena(self):
        ng, nm = self.grid.numel(), self.mlp.numel()
        arena = D.PeerArena({"p_grid": ng, "g_grid0": ng, "g_grid1": ng, "p_mlp": nm, "g_mlp0": nm, "g_mlp1": nm}, self.dev, self.group)
        arena.view("p_grid", ng).copy_(self.grid)
        arena.view("p_mlp", nm).copy_(self.mlp)
        self.grid = arena.view("p_grid", ng)
        self.model.embed_fn.params.data = self.grid                 # the module now reads the arena copy
        self.mlp = arena.view("p_mlp", nm)
        self._g_grid = [arena.view("g_grid0", ng), arena.view("g_grid1", ng)]
        self._g_mlp = [arena.view("g_mlp0", nm), arena.view("g_mlp1", nm)]
        self.g_grid, self.g_mlp = self._g_grid[0], self._g_mlp[0]
        nm4 = arena.sizes["p_mlp"]
        self.m_mlp = torch.zeros(nm4, device=self.dev); self.v_mlp = torch.zeros(nm4, device=self.dev)
        self.arena = arena
        torch.cuda.current_stream(self.dev).synchronize()
        arena.barrier()

    def _buffers(self, R, S):
        key = (R, S)
        b = self._bufs.get(key)
        if b is None:
            d = self.dev
            f32 = dict(device=d, dtype=torch.float32)
            b = dict(z=torch.empty(R, S, **f32), counts=torch.empty(2, device=d, dtype=torch.int64),
                     raw=torch.empty(R, S, L.MF_RAW_DIM, **f32), d_raw=torch.empty(R, S, L.MF_RAW_DIM, **f32),
                     rgb=torch.empty(R, 3, **f32), depth=torch.empty(R, **f32), losses=torch.zeros(8, **f32),
                     scratch=torch.empty(R * 8, **f32), u=torch.empty(R, S, **f32),
                     feat=torch.empty(int(L.lib().mf_feat_cache_size(R * S)), device=d, dtype=torch.uint8))
            self._bufs[key] = b
        return b

    def _field(self):
        f = self.model._field(keep=(self.grid, self.prep))
        return f

    def step(self, rays_o, rays_d, target_rgb, target_d, u=None, EMD_w=0.01, update=True, ray_grads=None):
        """One mapping iteration on device tensors (rays_o/rays_d (R,3), target_rgb (R,3), target_d (R,) or (R,1)).
        Returns the (8,) device tensor [rgb_loss, depth_loss, sdf_loss, fs_loss, psnr, fs_w, sdf_w, n_valid].
        ray_grads: optional pair of (R,3) device tensors that receive d loss / d rays_o and d loss / d rays_d (the pose-gradient
        leg of the reference's BA loop, mipsfusion.py:275-282,338-342).  ``self.pose_grad_impl`` selects the backward that
        produces them: "fp32" (CUDA-core decoder, 1e-6 against the oracle per ray) or "tc" (tensor cores, see DESIGN.md)."""
        model = self.model
        R = rays_o.shape[0]
        cfg, lins = model._render_cfg(True, EMD_w, self.dev)
        S = cfg.n_samples_d + cfg.n_range_d
        b = self._buffers(R, S)
        st = L.stream()
        field = self._field()
        target_d = target_d.reshape(R)
        if cfg.perturb:
            if u is None:
                u = b["u"].uniform_()                  # the reference's torch.rand(z_vals.shape), drawn on the device
        else:
            u = None
        tm = self.timing
        def ev():
            if tm is None:
                return None
            e = torch.cuda.Event(enable_timing=True); e.record(); return e
        e0 = ev()
        L.call("mf_sample_z", L.ptr(target_d), L.ptr(u), L.ptr(lins[0]), L.ptr(lins[1]), L.ptr(lins[2]), C.byref(cfg),
               L.ptr(b["z"]), L.ptr(b["counts"]), R, st)
        # batch-global mask counts (utils.py:43-47): only the loss kernels need them, so the 16-byte all-reduce runs on the
        # collective library's stream BESIDE the field forward (which leaves one SM free for it, mf_set_sm_reserve)
        work = D.allreduce_sum_async_(b["counts"], self.group)
        e1 = ev()
        L.call("mf_field_query_rays", L.ptr(rays_o), L.ptr(rays_d), L.ptr(b["z"]), C.byref(field), L.ptr(b["raw"]), L.ptr(b["feat"]),
               R, S, st)
        if work is not None:
            work.wait()
        e2 = ev()
        L.call("mf_render_loss_fwd", L.ptr(b["raw"]), L.ptr(b["z"]), L.ptr(target_rgb), L.ptr(target_d), L.ptr(b["counts"]),
               C.byref(cfg), L.ptr(b["rgb"]), L.ptr(b["depth"]), None, None, None, L.ptr(b["losses"]), L.ptr(b["scratch"]), R, S, st)
        L.call("mf_render_loss_bwd", L.ptr(b["raw"]), L.ptr(b["z"]), L.ptr(target_rgb), L.ptr(target_d), L.ptr(b["counts"]),
               L.ptr(b["losses"]), C.byref(cfg), L.ptr(self.loss_w), None, None, L.ptr(b["d_raw"]), R, S, st)
        e3 = ev()
        if ray_grads is None:
            L.call("mf_field_query_rays_bwd", L.ptr(rays_o), L.ptr(rays_d), L.ptr(b["z"]), C.byref(field), L.ptr(b["d_raw"]),
                   L.ptr(b["feat"]), L.ptr(self.g_grid), L.ptr(self.g_mlp), None, None, L.ptr(_Workspace.get(self.dev, field_points=R * S)), R, S, st)
        else:
            fb = field if self.pose_grad_impl == "tc" else self.model._field(keep=(self.grid, self.prep), impl=1)
            L.call("mf_field_query_rays_bwd", L.ptr(rays_o), L.ptr(rays_d), L.ptr(b["z"]), C.byref(fb), L.ptr(b["d_raw"]),
                   L.ptr(b["feat"]) if self.pose_grad_impl == "tc" else None, L.ptr(self.g_grid), L.ptr(self.g_mlp), L.ptr(ray_grads[0]), L.ptr(ray_grads[1]),
                   L.ptr(_Workspace.get(self.dev, field_points=R * S, want_ray_grads=True)), R, S, st)
            self.launches += 2            # zero-fill of the per-point gradients, reduction over the samples of a ray
        e4 = ev()
        self.launches += 9            # sample_z, field fwd, render+loss fwd (2), render+loss bwd, compaction (2), field bwd, partial reduce
        if update:
            if self.arena is not None:
                self.apply_gradients_sharded()
            else:
                D.average_gradients_([self.g_grid, self.g_mlp], self.group)
                self.apply_gradients()
        e5 = ev()
        if tm is not None:
            for name, a, c in (("sample_z", e0, e1), ("field_fwd", e1, e2), ("render_loss", e2, e3), ("field_bwd", e3, e4),
                               ("adam", e4, e5)):
                tm.setdefault(name, []).append((a, c))
        return b["losses"]

    def step_host(self, rays7, pose_idx, poses, EMD_w=0.01, pose_grad=False):
        """One mapping iteration from the HOST batch of the reference's BA loop (mipsfusion.py:289-322):
        ``rays7`` (R,7) float32 host tensor [dir_cam | rgb | depth] (pinned memory makes the copy asynchronous),
        ``pose_idx`` (R,) int64 host tensor (keyframe slot of each ray, -1 = current frame = last pose) or None,
        ``poses`` (K,4,4) camera-to-submap poses on the device.  Copies the batch to the device, generates the rays,
        runs :meth:`step` and returns the 8 loss terms as a host tensor (one synchronisation).
        pose_grad=True additionally returns d loss / d poses as a (K,4,4) device tensor (rows 0-2 filled: rotation block and
        translation column; the ray gradients are pushed through the ray generation by mf_gen_rays_packed_bwd).  The
        reference's loop feeds it to its pose parameters with ``poses_all.backward(d_poses)`` before ``pose_optimizer.step()``
        (mipsfusion.py:327,338-342)."""
        R = rays7.shape[0]
        hb = self._bufs.get(("host", R))
        if hb is None:
            f32 = dict(device=self.dev, dtype=torch.float32)
            hb = dict(rays7=torch.empty(R, 7, **f32), idx=torch.empty(R, device=self.dev, dtype=torch.int64),
                      o=torch.empty(R, 3, **f32), d=torch.empty(R, 3, **f32), rgb=torch.empty(R, 3, **f32),
                      depth=torch.empty(R, **f32), out=torch.empty(8, dtype=torch.float32).pin_memory())
            self._bufs[("host", R)] = hb
        hb["rays7"].copy_(rays7, non_blocking=True)
        if pose_idx is not None:
            hb["idx"].copy_(pose_idx, non_blocking=True)
        res = self._step_packed(hb, hb["idx"] if pose_idx is not None else None, poses, EMD_w, pose_grad)
        losses = res[0] if pose_grad else res
        hb["out"].copy_(losses, non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()
        return (hb["out"], res[1]) if pose_grad else hb["out"]

    def _step_packed(self, b, pose_idx, poses, EMD_w, pose_grad, u=None, d_poses=None):
        """The mapping iteration on a packed batch already on the device (``b["rays7"]`` (R,7), ``pose_idx`` (R,) or None):
        ray generation with ``poses`` (K,4,4), :meth:`step`, and with ``pose_grad`` the pose-gradient leg.  Returns the device
        losses, with ``pose_grad`` (losses, d_poses): ``d_poses`` (K,4,4) is ADDED to when given (the BA loop's accumulation
        across iterations), else a fresh zeroed tensor that is averaged over the ranks before it is returned."""
        R = b["rays7"].shape[0]
        poses = poses if (poses.is_cuda and poses.dtype == torch.float32 and poses.is_contiguous()) \
            else poses.to(self.dev, torch.float32).contiguous()
        K = poses.shape[0]
        L.call("mf_gen_rays_packed", L.ptr(b["rays7"]), L.ptr(poses), L.ptr(pose_idx), L.ptr(b["o"]), L.ptr(b["d"]), L.ptr(b["rgb"]),
               L.ptr(b["depth"]), R, K, L.stream())
        self.launches += 1
        if not pose_grad:
            return self.step(b["o"], b["d"], b["rgb"], b["depth"], u=u, EMD_w=EMD_w)
        if "d_o" not in b:
            b["d_o"], b["d_d"] = torch.empty_like(b["o"]), torch.empty_like(b["d"])
        losses = self.step(b["o"], b["d"], b["rgb"], b["depth"], u=u, EMD_w=EMD_w, ray_grads=(b["d_o"], b["d_d"]))
        average = d_poses is None
        if average:
            d_poses = torch.zeros(K, 4, 4, device=self.dev, dtype=torch.float32)
            self.launches += 1
        L.call("mf_gen_rays_packed_bwd", L.ptr(b["rays7"]), L.ptr(pose_idx), L.ptr(b["d_o"]), L.ptr(b["d_d"]), L.ptr(d_poses), R, K,
               L.stream())
        self.launches += 1
        if average:
            self._average_pose_grads(d_poses)
        return losses, d_poses

    def _average_pose_grads(self, d_poses):
        if self.world > 1:                                           # every rank holds the same poses: average the gradients
            D.allreduce_sum_(d_poses, self.group)
            d_poses.mul_(1.0 / self.world)

    def _store_batch(self, store, first_kf_Id, related_kf_ids, pix_num, cur_rays7, cur=None, **draws):
        """Packed batch buffers of (pix_num, n_cur) filled from the keyframe ray store: ``pix_num`` rays of the submap's
        keyframes (:meth:`KeyframeRayStore.sample_rays_in_submap`, pose index = slot in ``related_kf_ids``), then the current
        frame's rays (pose index -1 = last pose): ``cur_rays7``, or with ``cur`` = (frame tensors, n_cur, keys) ``n_cur`` pixels
        of the full-resolution frame drawn as ``sample_pixels_mix(H, W, 16, 24, depth, n_cur)`` (:meth:`_draw_cur`)."""
        n_cur = int(cur[1]) if cur is not None else 0 if cur_rays7 is None else int(cur_rays7.shape[0])
        pix_num = int(pix_num)
        R = pix_num + n_cur
        sb = self._bufs.get(("store", pix_num, n_cur))             # (keyed by the split: the tail of `idx` must stay -1)
        if sb is None:
            f32 = dict(device=self.dev, dtype=torch.float32)
            sb = dict(rays7=torch.empty(R, 7, **f32), idx=torch.full((R,), -1, device=self.dev, dtype=torch.int64),
                      kf_ids=torch.empty(pix_num, device=self.dev, dtype=torch.int64),
                      o=torch.empty(R, 3, **f32), d=torch.empty(R, 3, **f32), rgb=torch.empty(R, 3, **f32), depth=torch.empty(R, **f32))
            self._bufs[("store", pix_num, n_cur)] = sb
        if any(draws.get(k) is not None for k in ("idx_first", "idx_other", "idx_last")):
            rays, _, kf_indices = store.sample_rays_in_submap(first_kf_Id, related_kf_ids, pix_num, **draws)[:3]
            sb["rays7"][:pix_num].copy_(rays)                       # explicit draws: gathered into a fresh tensor
            sb["idx"][:pix_num].copy_(kf_indices)
        else:                                                       # device draws: the gather writes straight into the batch
            store.sample_rays_in_submap(first_kf_Id, related_kf_ids, pix_num, out=sb["rays7"],
                                        out_ids=(sb["kf_ids"], sb["idx"][:pix_num]), **draws)
        if cur is not None:
            self._draw_cur(cur, sb["rays7"][pix_num:])
        elif n_cur:
            sb["rays7"][pix_num:].copy_(cur_rays7)
        self.launches += 1
        return sb

    def _draw_cur(self, cur, out):
        """The current frame's pixels of one BA iteration (mipsfusion.py:306-309): the 16 x 24 lattice, then the top
        ``n_cur - 384`` of abs(randn) keys over the valid off-lattice pixels (``keys`` (H*W,), drawn here when None), gathered
        into ``out`` (n_cur, 7).  Three steps on buffers that persist per (H, W, n_cur): keys, mf_sample_pixels_topk,
        mf_kf_store."""
        (d, c, z, H, W), n_cur, keys = cur
        key = ("cur", H, W, n_cur)
        cb = self._bufs.get(key)
        if cb is None:
            cb = self._bufs[key] = dict(keys=torch.empty(H * W, device=self.dev, dtype=torch.float32),
                                        rows=torch.empty(n_cur, device=self.dev, dtype=torch.int64),
                                        cols=torch.empty(n_cur, device=self.dev, dtype=torch.int64),
                                        ws=torch.empty(int(L.lib().mf_topk_workspace_size(H * W)), device=self.dev, dtype=torch.uint8))
        if keys is None:
            keys = cb["keys"].normal_().abs_()                       # torch.randn_like(depth).abs() (sampling_helper.py:60)
            self.launches += 2
        st = L.stream()
        L.call("mf_sample_pixels_topk", L.ptr(z), L.ptr(keys), H, W, 16, 24, n_cur, None, L.ptr(cb["rows"]), L.ptr(cb["cols"]),
               L.ptr(cb["ws"]), st)
        L.call("mf_kf_store", L.ptr(d), L.ptr(c), L.ptr(z), L.ptr(cb["rows"]), L.ptr(cb["cols"]), W, n_cur, L.ptr(out), st)
        self.launches += 11                                          # lattice, top-k init, 6 radix passes, compaction, sort; gather

    def step_from_store(self, store, first_kf_Id, related_kf_ids, poses_all, pix_num, cur_rays7=None, EMD_w=0.01, pose_grad=False,
                        **draws):
        """One mapping iteration fed from the device-resident keyframe ray store (steps 3.1-3.4 of the reference's BA
        loop, mipsfusion.py:293-335, without any host data): sample ``pix_num`` rays of the submap's keyframes
        (:class:`KeyframeRayStore.sample_rays_in_submap`), append the current frame's rays ``cur_rays7`` (n,7; pose index
        -1 = last pose), generate the rays with ``poses_all`` (K,4,4) and run :meth:`step`.  Returns the device losses;
        pose_grad=True returns (losses, d_poses) with d_poses as :meth:`step_host` returns it (rank average included)."""
        sb = self._store_batch(store, first_kf_Id, related_kf_ids, pix_num, cur_rays7, **draws)
        return self._step_packed(sb, sb["idx"], poses_all, EMD_w, pose_grad)

    def first_frame_mapping(self, batch, n_iters, c2w=None, pix_num=None, seed=None, u=None, EMD_w=0.01):
        """Submap initialisation (the reference's first_frame_mapping, mipsfusion.py:155-194, and initialize_new_localMLP,
        :198-222) on the device: ``n_iters`` map steps on one full-resolution frame, each on ``pix_num`` rays drawn afresh
        (``mf_frame_sample_rays``: random.sample(range(H*W), pix_num) decoded column-major, gathered into the packed batch)
        and generated with the frame's pose ``c2w`` (4,4) in the submap's frame (identity when None: the frame that opens a
        submap defines its frame).  Map Adam runs every iteration, zero_grad fused in.

        batch: as :meth:`KeyframeRayStore.add_keyframe` takes it.  pix_num: ``config["mapping"]["sample"]`` unless given.
        seed: base of the draws (rank r, iteration i draws with seed + i world + r); from torch's CPU generator when None.
        u: optional (n_iters, pix_num, S) stratified jitter.  A new submap is a fresh model (or ``model.recover_initial_param()``)
        and a new FusedMapper, whose Adam state starts at zero as the reference's create_optimizer's does.  With a process
        group the step's data-parallel exchange applies and every rank draws its own rays.

        -> losses (n_iters, 8) device tensor, overwritten by the next call of the same shape; the model is stepped in place.
        No host synchronisation; no allocation after the first call for an (H, W, pix_num, n_iters) when the inputs are
        float32, contiguous and on the device."""
        n_iters = int(n_iters)
        if n_iters < 0:
            raise L.MipsFusionB200Error("first_frame_mapping: n_iters must be >= 0, got %d" % n_iters)
        if pix_num is None:
            mc = self.model.config.get("mapping", {})
            if "sample" not in mc:
                raise L.MipsFusionB200Error("first_frame_mapping: pix_num not given and config['mapping'] has no 'sample'")
            pix_num = mc["sample"]
        R = int(pix_num)
        d, c, z, H, W = frame_tensors(batch, self.dev)
        if not 0 < R <= H * W:
            raise L.MipsFusionB200Error("first_frame_mapping: pix_num must lie in [1, H*W = %d], got %d" % (H * W, R))
        losses = self._bufs.get(("init_losses", R, n_iters))
        if losses is None:
            losses = self._bufs[("init_losses", R, n_iters)] = torch.zeros(n_iters, 8, device=self.dev, dtype=torch.float32)
        if n_iters == 0:
            return losses
        sb = self._bufs.get(("frame", R))
        if sb is None:
            f32 = dict(device=self.dev, dtype=torch.float32)
            sb = self._bufs[("frame", R)] = dict(rays7=torch.empty(R, 7, **f32), o=torch.empty(R, 3, **f32), d=torch.empty(R, 3, **f32),
                                                 rgb=torch.empty(R, 3, **f32), depth=torch.empty(R, **f32))
        if c2w is None:
            P = self._bufs.get("eye")
            if P is None:
                P = self._bufs["eye"] = torch.eye(4, device=self.dev, dtype=torch.float32)[None]
        else:
            P = torch.as_tensor(c2w).reshape(1, 4, 4)
            if not (P.is_cuda and P.dtype == torch.float32 and P.is_contiguous()):
                P = P.to(self.dev, torch.float32).contiguous()      # once, not per iteration
        if u is not None:
            u = L.f32c(u, self.dev)
        self.model.decoder.prepared()                                # adopt external writes to the decoder's parameters
        seed = _new_seed() if seed is None else int(seed)
        world, rank = D.world(self.group)
        st = L.stream()
        for i in range(n_iters):
            L.call("mf_frame_sample_rays", L.ptr(d), L.ptr(c), L.ptr(z), H, W, R, (seed + i * world + rank) & 0xffffffff, None,
                   L.ptr(sb["rays7"]), None, st)
            li = self._step_packed(sb, None, P, EMD_w, False, u=None if u is None else u[i])
            losses[i].copy_(li)
            self.launches += 2
        return losses

    def local_ba(self, store, first_kf_Id, related_kf_ids, poses_all, pix_num, cur_rays7=None, n_iters=None, pose_accum_step=None,
                 lr_rot=None, lr_trans=None, optim_cur=None, seed=None, u=None, EMD_w=0.01, cur_frame=None, n_cur=None, cur_keys=None):
        """The reference's local bundle adjustment (MIPSFusion.local_BA, mipsfusion.py:259-370; the same body runs in
        InactiveMap.local_BA, local_BA_switch and initialize_new_localMLP) on the device: ``n_iters`` mapping iterations fed from
        the keyframe ray store (as :meth:`step_from_store`) that also accumulate d loss / d poses, and every ``pose_accum_step``
        iterations one Adam step on the keyframe poses (quaternion + translation, get_pose_param_optim :235-241,280-282,
        step :338-342).  Gradients of a trailing partial period are dropped, as in the reference.

        poses_all (K,4,4): the related keyframes' poses in the order of ``related_kf_ids``, then the current frame's.  Pose 0
        (the submap's first keyframe) is never optimised, the last one only with ``optim_cur``; both come back bit for bit.
        n_iters, pose_accum_step, lr_rot, lr_trans, optim_cur: ``config["mapping"]`` keys iters, pose_accum_step, lr_rot,
        lr_trans, optim_cur unless given.  seed: base of the ray draws (rank r, iteration i draw with seed + 3 (i world + r),
        the three segment seeds of mf_kf_sample_rays); from torch's CPU generator when None.  u: optional (n_iters, R, S)
        stratified jitter.  With a process group every rank draws its own rays and the pose gradients are averaged over the
        ranks once per pose step, so all ranks hold the same poses.

        The current frame's rays: ``cur_rays7`` (n,7), the same rows in every iteration; or ``cur_frame`` (a batch dict as
        :meth:`KeyframeRayStore.add_keyframe` takes it) with ``n_cur``: every iteration draws ``n_cur`` pixels of it afresh as
        the reference's ``sample_pixels_mix(H, W, 16, 24, depth, n_cur)`` does (mipsfusion.py:306-309), on abs(randn) keys
        drawn on the device or from ``cur_keys[i]`` (cur_keys (n_iters, H*W)).  384 <= n_cur <= 384 + 4096.

        -> (poses (K,4,4), losses (n_iters, 8)) device tensors, overwritten by the next call of the same shape.  No host
        synchronisation; no allocation after the first call for a (K, pix_num, n_cur, n_iters) (and frame size)."""
        mc = self.model.config.get("mapping", {})

        def hp(v, key):
            if v is not None:
                return v
            if key not in mc:
                raise L.MipsFusionB200Error("local_ba: %s not given and config['mapping'] has no '%s'" % (key, key))
            return mc[key]
        n_iters, accum = int(hp(n_iters, "iters")), int(hp(pose_accum_step, "pose_accum_step"))
        lr_rot, lr_trans, optim_cur = float(hp(lr_rot, "lr_rot")), float(hp(lr_trans, "lr_trans")), bool(hp(optim_cur, "optim_cur"))
        if accum < 1:
            raise L.MipsFusionB200Error("local_ba: pose_accum_step must be >= 1")
        cur = None
        if cur_frame is None and (n_cur is not None or cur_keys is not None):
            raise L.MipsFusionB200Error("local_ba: n_cur / cur_keys are for the cur_frame draw; cur_frame is missing")
        if cur_frame is not None:
            if cur_rays7 is not None:
                raise L.MipsFusionB200Error("local_ba: pass cur_rays7 or cur_frame, not both")
            if n_cur is None:
                raise L.MipsFusionB200Error("local_ba: cur_frame needs n_cur")
            n_cur = int(n_cur)
            if n_cur < 16 * 24 or n_cur - 16 * 24 > 4096:
                raise L.MipsFusionB200Error("local_ba: n_cur must lie in [384, 4480] (the 16 x 24 lattice plus at most 4096 "
                                            "random pixels), got %d" % n_cur)
            frame = frame_tensors(cur_frame, self.dev)
            if cur_keys is not None:
                cur_keys = L.f32c(cur_keys, self.dev)
                if tuple(cur_keys.shape) != (n_iters, frame[3] * frame[4]):
                    raise L.MipsFusionB200Error("local_ba: cur_keys must be (n_iters, H*W) = (%d, %d)" % (n_iters, frame[3] * frame[4]))
            cur = (frame, n_cur, cur_keys)
        self.model.decoder.prepared()                                # adopt external writes to the decoder's parameters
        K = int(poses_all.shape[0])
        n_cur = int(n_cur) if cur is not None else 0 if cur_rays7 is None else int(cur_rays7.shape[0])
        key = ("ba", K, int(pix_num), n_cur)
        bb = self._bufs.get(key)
        if bb is None:
            f32 = dict(device=self.dev, dtype=torch.float32)
            bb = self._bufs[key] = dict(state=torch.zeros(K, 24, **f32), poses=torch.empty(K, 4, 4, **f32),
                                        d_poses=torch.zeros(K, 4, 4, **f32), frozen={}, losses={})
        frozen = bb["frozen"].get(optim_cur)
        if frozen is None:
            f = torch.zeros(K, dtype=torch.uint8)
            f[0] = 1                                                 # get_pose_param_optim(poses[1:])
            if not optim_cur:
                f[-1] = 1
            frozen = bb["frozen"][optim_cur] = f.to(self.dev)
        losses = bb["losses"].get(n_iters)
        if losses is None:
            losses = bb["losses"][n_iters] = torch.zeros(n_iters, 8, device=self.dev, dtype=torch.float32)
        poses_in = poses_all if (poses_all.is_cuda and poses_all.dtype == torch.float32 and poses_all.is_contiguous()) \
            else poses_all.to(self.dev, torch.float32).contiguous()
        st = L.stream()
        L.call("mf_ba_pose_init", L.ptr(poses_in), L.ptr(frozen), K, L.ptr(bb["state"]), L.ptr(bb["poses"]), st)
        bb["d_poses"].zero_()
        self.launches += 2
        seed = _new_seed() if seed is None else int(seed)
        world, rank = D.world(self.group)
        for i in range(n_iters):
            ci = None if cur is None else (cur[0], cur[1], None if cur[2] is None else cur[2][i])
            sb = self._store_batch(store, first_kf_Id, related_kf_ids, pix_num, cur_rays7, cur=ci,
                                   seed=(seed + 3 * (i * world + rank)) & 0xffffffff)
            li, _ = self._step_packed(sb, sb["idx"], bb["poses"], EMD_w, True, u=None if u is None else L.f32c(u[i], self.dev),
                                      d_poses=bb["d_poses"])
            losses[i].copy_(li)
            self.launches += 1
            if (i + 1) % accum == 0:
                self._average_pose_grads(bb["d_poses"])
                L.call("mf_ba_pose_update", L.ptr(bb["state"]), L.ptr(bb["d_poses"]), L.ptr(frozen), K, lr_rot, lr_trans,
                       L.ptr(bb["poses"]), st)
                self.launches += 1
        return bb["poses"], losses

    def apply_gradients(self):
        """Adam on (grid, decoder) with the reference's groups (mipsfusion.py:580-584), zero_grad fused in."""
        self.step_count += 1
        st = L.stream()
        if self.grid.numel() % 4 == 0 and self.grid.data_ptr() % 16 == 0:
            L.call("mf_adam_step_pair", L.ptr(self.grid), L.ptr(self.g_grid), L.ptr(self.m_grid), L.ptr(self.v_grid), self.grid.numel(),
                   float(self.lr_embed), 1e-15, 0.0, L.ptr(self._mlp_pad), L.ptr(self._g_mlp_pad), L.ptr(self.m_mlp), L.ptr(self.v_mlp),
                   self._mlp_pad.numel(), float(self.lr_decoder), 1e-8, 1e-6, 0.9, 0.99, self.step_count, st)
            self.launches += 1
        else:
            L.call("mf_adam_step", L.ptr(self.grid), L.ptr(self.g_grid), L.ptr(self.m_grid), L.ptr(self.v_grid), self.grid.numel(),
                   float(self.lr_embed), 0.9, 0.99, 1e-15, 0.0, self.step_count, 1, st)
            L.call("mf_adam_step", L.ptr(self._mlp_pad), L.ptr(self._g_mlp_pad), L.ptr(self.m_mlp), L.ptr(self.v_mlp), self._mlp_pad.numel(),
                   float(self.lr_decoder), 0.9, 0.99, 1e-8, 1e-6, self.step_count, 1, st)
            self.launches += 2
        L.call("mf_mlp_prepare", L.ptr(self.mlp), L.ptr(self.prep), st)
        self.launches += 1

    def apply_gradients_sharded(self):
        """Data-parallel update over peer memory: barrier, one sharded reduce + Adam + broadcast kernel per tensor,
        barrier.  The gradient buffers alternate between steps; the kernel clears the one the next backward uses."""
        self.step_count += 1
        a, st = self.arena, L.stream()
        cur, nxt = (self.step_count - 1) & 1, self.step_count & 1
        bases = (C.c_uint64 * a.world)(*a.peer_bases)
        # in-switch reduction / multicast store (NVLS) pays from 4 GPUs on (measured on 8 x B200: 74 vs 115 us at 8 GPUs,
        # 85 vs 88 us at 4, 99 vs 61 us at 2 for the 9.0 M-parameter grid); below that plain peer loads / stores
        mc = a.multicast_base if (self.multicast is True or (self.multicast == "auto" and a.world >= 4)) else 0
        a.barrier()                                                  # every rank's gradients are complete
        L.call("mf_adam_step_sharded", bases, a.world, a.rank, a.offsets["p_grid"], a.offsets["g_grid%d" % cur],
               a.offsets["g_grid%d" % nxt], L.ptr(self.m_grid), L.ptr(self.v_grid), a.sizes["p_grid"],
               float(self.lr_embed), 0.9, 0.99, 1e-15, 0.0, self.step_count, mc, st)
        L.call("mf_adam_step_sharded", bases, a.world, a.rank, a.offsets["p_mlp"], a.offsets["g_mlp%d" % cur],
               a.offsets["g_mlp%d" % nxt], L.ptr(self.m_mlp), L.ptr(self.v_mlp), a.sizes["p_mlp"],
               float(self.lr_decoder), 0.9, 0.99, 1e-8, 1e-6, self.step_count, mc, st)
        a.barrier()                                                  # every slab has reached every replica
        self.g_grid, self.g_mlp = self._g_grid[nxt], self._g_mlp[nxt]
        L.call("mf_mlp_prepare", L.ptr(self.mlp), L.ptr(self.prep), st)
        self.launches += 3            # two sharded updates + weight prepare (the barriers are torch's kernels)

    def sync_to_module(self):
        """Kept for callers of the first version: the module's parameters ARE the stepped weights (views of the flat master,
        see :meth:`_bind_module`), so there is nothing to copy; re-binds if the module's parameters were re-assigned."""
        ps = self.model.decoder.ordered_params()
        ext = self.model.decoder.__dict__.get("_ext_prep")
        if ext is None or ext[1] is not self or tuple(p.data_ptr() for p in ps) != ext[0]:
            o = 0
            with torch.no_grad():
                for p in ps:                                   # adopt whatever the module holds now, then bind again
                    n = p.numel()
                    self.mlp[o:o + n].copy_(p.detach().reshape(-1))
                    o += n
            L.call("mf_mlp_prepare", L.ptr(self.mlp), L.ptr(self.prep), L.stream())
            self._bind_module()
