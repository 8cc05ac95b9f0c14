"""Overlap-region SDF consistency of the inactive-map global BA (InactiveMap.get_SDF_dif / get_SDF_dif2, InactiveMap.py:128-192;
loss helper_functions/geometry_helper.py:225-229) as one fused operator over many submap pairs.

    ov = OverlapSDF(model_list)                      # the submaps' JointEncoding modules, one device
    loss = ov.get_SDF_dif(rays, ovlp_kf_pose, id1, id2, first_kf_pose1, first_kf_pose2, trunc_value)
    loss = ov.get_SDF_dif2(target_d, rays_d_cam, mask, ovlp_kf_pose, id1, id2, first_kf_pose1, first_kf_pose2, trunc_value)
    losses = ov.pairs(pair_ids, target_d, rays_d_cam, mask, ovlp_kf_pose, first_kf_poses, trunc_value)     # (P,)

A call is three kernels of overlap_kernels.cu around one fp32 field query per distinct submap (mf_field_query); the backward
is one point-gradient field backward per distinct submap and the pose backward.  Every sum has a fixed order (no atomics),
so the losses and the pose gradients are bitwise reproducible, and ``pairs`` equals the single-pair calls bit for bit.
"""
import ctypes as C

import torch

from . import _lib as L
from .decoder import _Workspace


class _Plan:
    """Persistent buffers of one call shape: (pair list, N, per-ray overlap poses, number of first-keyframe poses)."""

    def __init__(self, dev, pairs, N, per_ray, n_first):
        P = len(pairs)
        self.P, self.N, self.per_ray, self.n_first = P, N, per_ray, n_first
        # rows grouped by submap (first appearance order), (pair, side) order inside a submap: one field launch per submap
        order, rows = [], {}
        for p, ids in enumerate(pairs):
            for s in range(2):
                if ids[s] not in rows:
                    rows[ids[s]] = []
                    order.append(ids[s])
                rows[ids[s]].append((p, s))
        tab = [[0, 0, 0, 0] for _ in range(P)]
        self.segments, row = [], 0
        for m in order:
            self.segments.append((m, row * N, len(rows[m]) * N))
            for p, s in rows[m]:
                tab[p][2 + s] = row * N
                row += 1
        for p, ids in enumerate(pairs):
            tab[p][0], tab[p][1] = (0, 1) if n_first == 0 else (ids[0], ids[1])
        n_poses = 2 if n_first == 0 else n_first
        f32 = dict(device=dev, dtype=torch.float32)
        self.tab = torch.tensor(tab, dtype=torch.int32).to(dev)
        self.pts = torch.empty(2 * P * N, 3, **f32)
        self.raw = torch.empty(2 * P * N, L.MF_RAW_DIM, **f32)
        self.d_raw = torch.empty(2 * P * N, L.MF_RAW_DIM, **f32)
        self.d_pts = torch.empty(2 * P * N, 3, **f32)
        self.loss = torch.empty(P, **f32)
        self.finv = torch.empty(P, 2, 16, **f32)
        self.dF_pair = torch.empty(P, 2, 16, **f32)
        self.first = torch.empty(n_poses, 4, 4, **f32)            # staging copy of the poses when they are not fp32 contiguous
        self.d_first = torch.empty(n_poses, 4, 4, **f32)
        self.ovlp = torch.empty(P, N if per_ray else 1, 4, 4, **f32)
        self.d_ovlp = torch.empty_like(self.ovlp)
        # the gradients handed to autograd are these views; holding them here keeps autograd from adopting a view of a buffer
        # that the next call overwrites as a parameter's .grad (it accumulates into an existing .grad or copies instead)
        self.g_first = [self.d_first[0], self.d_first[1]] if n_first == 0 else [self.d_first]
        self.g_ovlp = {}
        self.n_ws = max(n for _, _, n in self.segments)
        self.generation = 0


def _rows(t, R, w, what, dev):
    """(view, row stride in elements) of t as R rows of w fp32 elements with unit column stride: row-strided views (the
    columns of the reference's (N,7) ray tensor) are read in place."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda or t.device != dev:
        raise L.MipsFusionB200Error(f"OverlapSDF: {what} must be a CUDA tensor on {dev} (no CPU fallback)")
    if t.numel() != R * w:
        raise L.MipsFusionB200Error(f"OverlapSDF: {what} has shape {tuple(t.shape)}, expected {R} x {w} elements")
    if t.dtype != torch.float32:
        t = t.float()
    try:
        v = t.view(R, w)
    except RuntimeError:
        v = t.contiguous().view(R, w)
    if w > 1 and v.stride(1) != 1:
        v = v.contiguous()
    return v, int(v.stride(0)) if R > 1 else w


class _OverlapFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, op, plan, io, trunc, ovlp, *firsts):
        st = L.stream()
        P, N = plan.P, plan.N
        if len(firsts) == 2:                                       # single pair: the two poses side by side
            plan.first[0].copy_(firsts[0]); plan.first[1].copy_(firsts[1])
            first = plan.first
        else:
            first = firsts[0]
            if first.dtype != torch.float32 or not first.is_contiguous():
                first = plan.first.copy_(first)
        ovlp_shape = tuple(ovlp.shape)
        if ovlp.dtype != torch.float32 or not ovlp.is_contiguous():
            ovlp = plan.ovlp.copy_(ovlp.reshape(plan.ovlp.shape))
        (td, ld_d), (dirs, ld_dir), (mask, kind, ld_m) = io
        L.call("mf_overlap_points", L.ptr(first), L.ptr(plan.tab), P, N, L.ptr(ovlp), int(plan.per_ray), td.data_ptr(), ld_d,
               dirs.data_ptr(), ld_dir, L.ptr(plan.finv), L.ptr(plan.pts), st)
        keep = []
        for m, r0, n in plan.segments:
            model = op.models[m]
            field = model._field(impl=1)
            keep.append(field._keepalive)
            L.call("mf_field_query", plan.pts[r0:].data_ptr(), C.byref(field), op.normalize[m], plan.raw[r0:].data_ptr(), n, st)
        L.call("mf_overlap_loss", L.ptr(plan.raw), L.ptr(plan.tab), P, N, td.data_ptr(), ld_d,
               None if mask is None else mask.data_ptr(), kind, ld_m, float(trunc), L.ptr(plan.loss), L.ptr(plan.d_raw), st)
        plan.generation += 1
        ctx.op, ctx.plan, ctx.io, ctx.keep, ctx.gen = op, plan, io, keep, plan.generation
        ctx.ovlp, ctx.ovlp_shape = ovlp, ovlp_shape
        return plan.loss.view(()) if len(firsts) == 2 else plan.loss.view(P)

    @staticmethod
    def backward(ctx, g):
        op, plan = ctx.op, ctx.plan
        if plan.generation != ctx.gen:
            raise L.MipsFusionB200Error("OverlapSDF: a later call of the same shape has reused this call's buffers; "
                                        "run backward before the next call (or batch the pairs into one pairs() call)")
        st = L.stream()
        P, N = plan.P, plan.N
        dev = plan.loss.device
        ws = _Workspace.get(dev, field_points=plan.n_ws)
        for (m, r0, n), keep in zip(plan.segments, ctx.keep):
            field = op.models[m]._field(keep, impl=1)
            L.call("mf_field_query_bwd", plan.pts[r0:].data_ptr(), C.byref(field), op.normalize[m], plan.d_raw[r0:].data_ptr(),
                   None, None, plan.d_pts[r0:].data_ptr(), L.ptr(ws), n, st)
        if g.dtype != torch.float32 or g.device != dev:
            g = g.to(dev, torch.float32)
        ld_g = int(g.stride(0)) if g.dim() == 1 else 0
        want_ovlp = ctx.needs_input_grad[4]
        (td, ld_d), (dirs, ld_dir), _ = ctx.io
        L.call("mf_overlap_pose_bwd", L.ptr(plan.finv), L.ptr(plan.tab), P, N, L.ptr(ctx.ovlp), int(plan.per_ray), td.data_ptr(),
               ld_d, dirs.data_ptr(), ld_dir, L.ptr(plan.d_pts), g.data_ptr(), ld_g, plan.first.shape[0], L.ptr(plan.dF_pair),
               L.ptr(plan.d_first), L.ptr(plan.d_ovlp) if want_ovlp else None, st)
        d_ovlp = None
        if want_ovlp:
            shape = ctx.ovlp_shape
            d_ovlp = plan.g_ovlp.get(shape)
            if d_ovlp is None:
                d_ovlp = plan.g_ovlp[shape] = plan.d_ovlp.view(shape)
        firsts = [gf if need else None for gf, need in zip(plan.g_first, ctx.needs_input_grad[5:])]
        return (None, None, None, None, d_ovlp, *firsts)


class OverlapSDF:
    """Fused InactiveMap.get_SDF_dif / get_SDF_dif2 over the submaps' fields ``model_list`` (JointEncoding modules on one CUDA
    device).  The field weights are read through each model's fp32 descriptor on every call (``_field(impl=1)``, the decoder
    ``_FieldQueryFn`` uses for point gradients), so weights stepped by a mapper are seen without a copy.

    Semantics (tests/golden/overlap.npz pins them to the reference's own methods): for pair (id1, id2) and side s, the local
    pose A = first_kf_pose_s^-1 @ ovlp_kf_pose (the inverse in fp64 through the adjugate, rounded once to fp32), the point
    x = A[:3,3] + (sum_k d_cam[k] A[:3,k]) depth, sdf_s = run_network(x)[3] * trunc_value of submap id_s (fp32 decoder), and
    loss = sum (sdf1 m - sdf2 m)^2 / (count_nonzero(m) + 0.001) with m = (depth > 0) (get_SDF_dif) or the caller's mask
    (get_SDF_dif2).  The reference adds ``0. * compute_avg_rgb_difference(...)``; its value and gradient are 0 for finite
    fields, so it is not computed.

    Gradients: ``backward`` fills d loss / d first-keyframe poses (summed over the pairs that use a submap, in pair order) and
    d loss / d overlap poses when they require grad.  It produces NO hash-grid or decoder gradients: callers that want
    parameter gradients use the composition (oracle/overlap.py over the models' run_network).

    No host synchronisation, and no allocation after the first call of a shape (pairs, N, overlap-pose layout).  The returned
    loss is a view of that shape's buffer: the next call of the same shape overwrites it, and a backward after such a call
    raises.  Gradients of the pose tensors accumulate into an existing ``.grad`` in place."""

    def __init__(self, model_list):
        self.models = list(model_list)
        if not self.models:
            raise L.MipsFusionB200Error("OverlapSDF: empty model list")
        devs = {m.embed_fn.params.device for m in self.models}
        if len(devs) != 1:
            raise L.MipsFusionB200Error(f"OverlapSDF: the models live on different devices {sorted(map(str, devs))}")
        self.device = devs.pop()
        if self.device.type != "cuda":
            raise L.MipsFusionB200Error("OverlapSDF: the models must live on a CUDA device (no CPU fallback)")
        self.normalize = [int(bool(m.config["grid"]["tcnn_encoding"])) for m in self.models]
        self._plans = {}

    # ---- InactiveMap.get_SDF_dif (InactiveMap.py:149-165) --------------------------------------------------------
    def get_SDF_dif(self, rays, ovlp_kf_pose, id1, id2, first_kf_pose1, first_kf_pose2, trunc_value):
        """rays (N,7) = [d_cam | rgb | depth]; mask = (depth > 0).  -> 0-dim loss."""
        if rays.dim() != 2 or rays.shape[1] < 7:
            raise L.MipsFusionB200Error(f"OverlapSDF.get_SDF_dif: rays must be (N,7), got {tuple(rays.shape)}")
        N = rays.shape[0]
        io = (_rows(rays[:, 6], N, 1, "target depth", self.device), _rows(rays[:, :3], N, 3, "ray directions", self.device),
              (None, 0, 0))
        return self._single(io, N, ovlp_kf_pose, id1, id2, first_kf_pose1, first_kf_pose2, trunc_value)

    # ---- InactiveMap.get_SDF_dif2 (InactiveMap.py:177-192) -------------------------------------------------------
    def get_SDF_dif2(self, target_d, rays_d_cam, mask, ovlp_kf_pose, id1, id2, first_kf_pose1, first_kf_pose2, trunc_value):
        """target_d (N,1), rays_d_cam (N,3), mask (N,1) (bool, uint8 or float).  -> 0-dim loss."""
        N = target_d.shape[0] if target_d.dim() > 0 else 0
        if target_d.dim() != 2 or tuple(target_d.shape) != (N, 1) or tuple(rays_d_cam.shape) != (N, 3) or mask.numel() != N:
            raise L.MipsFusionB200Error("OverlapSDF.get_SDF_dif2: need target_d (N,1), rays_d_cam (N,3), mask (N,1); got "
                                        f"{tuple(target_d.shape)}, {tuple(rays_d_cam.shape)}, {tuple(mask.shape)}")
        io = (_rows(target_d, N, 1, "target_d", self.device), _rows(rays_d_cam, N, 3, "rays_d_cam", self.device),
              self._mask(mask, N))
        return self._single(io, N, ovlp_kf_pose, id1, id2, first_kf_pose1, first_kf_pose2, trunc_value)

    # ---- many pairs --------------------------------------------------------------------------------------------
    def pairs(self, pair_ids, target_d, rays_d_cam, mask, ovlp_kf_pose, first_kf_poses, trunc_value):
        """get_SDF_dif2 of P pairs in one call.  pair_ids (P,2) on the host (list, numpy or CPU tensor: the point layout is
        planned from it without a device round trip); target_d (P,N), rays_d_cam (P,N,3), mask (P,N), ovlp_kf_pose (P,N,4,4)
        or (P,1,4,4), first_kf_poses (M,4,4) with M = len(model_list).  -> (P,) device tensor of losses."""
        if isinstance(pair_ids, torch.Tensor):
            if pair_ids.is_cuda:
                raise L.MipsFusionB200Error("OverlapSDF.pairs: pair_ids must be on the host (a device copy would synchronise)")
            pair_ids = pair_ids.tolist()
        pairs = [tuple(int(i) for i in ids) for ids in (pair_ids.tolist() if hasattr(pair_ids, "tolist") else pair_ids)]
        if not pairs or any(len(ids) != 2 for ids in pairs):
            raise L.MipsFusionB200Error("OverlapSDF.pairs: pair_ids must be a non-empty (P,2) list of submap ids")
        P = len(pairs)
        if target_d.dim() != 2 or target_d.shape[0] != P:
            raise L.MipsFusionB200Error(f"OverlapSDF.pairs: target_d must be (P,N) with P = {P}, got {tuple(target_d.shape)}")
        N = target_d.shape[1]
        if tuple(rays_d_cam.shape) != (P, N, 3) or tuple(mask.shape) not in ((P, N), (P, N, 1)):
            raise L.MipsFusionB200Error(f"OverlapSDF.pairs: need rays_d_cam (P,N,3) and mask (P,N) for P={P}, N={N}; got "
                                        f"{tuple(rays_d_cam.shape)}, {tuple(mask.shape)}")
        M = len(self.models)
        self._tensor(first_kf_poses, "first_kf_poses")
        if tuple(first_kf_poses.shape) != (M, 4, 4):
            raise L.MipsFusionB200Error(f"OverlapSDF.pairs: first_kf_poses must be ({M},4,4), got {tuple(first_kf_poses.shape)}")
        self._ids(pairs)
        per_ray = self._ovlp(ovlp_kf_pose, (P, N, 4, 4), (P, 1, 4, 4))
        io = (_rows(target_d, P * N, 1, "target_d", self.device), _rows(rays_d_cam, P * N, 3, "rays_d_cam", self.device),
              self._mask(mask, P * N))
        plan = self._plan(pairs, N, per_ray, M)
        return _OverlapFn.apply(self, plan, io, float(trunc_value), ovlp_kf_pose, first_kf_poses)

    # ---- helpers -----------------------------------------------------------------------------------------------
    def _single(self, io, N, ovlp, id1, id2, f1, f2, trunc):
        if N < 1:
            raise L.MipsFusionB200Error("OverlapSDF: no rays")
        for t, what in ((f1, "first_kf_pose1"), (f2, "first_kf_pose2")):
            self._tensor(t, what)
            if tuple(t.shape) != (4, 4):
                raise L.MipsFusionB200Error(f"OverlapSDF: {what} must be (4,4), got {tuple(t.shape)}")
        pair = (int(id1), int(id2))
        self._ids([pair])
        per_ray = self._ovlp(ovlp, (N, 4, 4), (1, 4, 4))
        plan = self._plan([pair], N, per_ray, 0)
        return _OverlapFn.apply(self, plan, io, float(trunc), ovlp, f1, f2)

    def _tensor(self, t, what):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.device != self.device:
            raise L.MipsFusionB200Error(f"OverlapSDF: {what} must be a CUDA tensor on {self.device} (no CPU fallback)")

    def _ids(self, pairs):
        M = len(self.models)
        for ids in pairs:
            if not all(0 <= i < M for i in ids):
                raise L.MipsFusionB200Error(f"OverlapSDF: submap ids {ids} outside [0, {M})")

    def _ovlp(self, ovlp, per_ray_shape, shared_shape):
        self._tensor(ovlp, "ovlp_kf_pose")
        shape = tuple(ovlp.shape)
        if shape not in (per_ray_shape, shared_shape):
            raise L.MipsFusionB200Error(f"OverlapSDF: ovlp_kf_pose must be {per_ray_shape} or {shared_shape}, got {shape}")
        return shape == per_ray_shape and per_ray_shape != shared_shape

    def _mask(self, mask, R):
        self._tensor(mask, "mask")
        if mask.numel() != R:
            raise L.MipsFusionB200Error(f"OverlapSDF: mask has {mask.numel()} elements, expected {R}")
        if mask.dtype in (torch.bool, torch.uint8):
            kind, m = 2, mask.view(torch.uint8) if mask.dtype == torch.bool else mask
            m = m.reshape(R) if m.is_contiguous() else m.contiguous().reshape(R)
            return (m, kind, 1)
        m, ld = _rows(mask, R, 1, "mask", self.device)
        return (m, 1, ld)

    def _plan(self, pairs, N, per_ray, n_first):
        key = (tuple(pairs), N, per_ray, n_first)
        plan = self._plans.get(key)
        if plan is None:
            if len(self._plans) >= 64:
                self._plans.clear()
            plan = self._plans[key] = _Plan(self.device, pairs, N, per_ray, n_first)
        return plan
