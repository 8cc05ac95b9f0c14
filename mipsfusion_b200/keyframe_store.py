"""Device-resident keyframe ray store: the ray part of the reference's KeyframeSet (model/keyframeSet.py:20-25,
76-79,170-175,386-455), the step directly before the mapping hot path ("next" row N1 of SURVEY.md section 8).

The reference keeps ``rays (num_kf, 150*200, 7)`` on the CPU, draws pixel indices with python ``random.sample`` and copies the
sampled batch to the GPU every mapping iteration.  Here the store lives in HBM (50 keyframes x 840 KB), the draws are
explicit device index tensors (``sample_without_replacement``: top-k of uniform keys, drawn on the device when no keys
are given) and the gather is one kernel, so a mapping iteration needs no host data at all.  Same method names, argument
meaning and return values (sampled rays, kf_ids, kf_indices) as the reference; integer outputs are bit-exact for the
same index draws (tests/golden/keyframes.npz)."""
import torch

from . import _lib as L
from . import sampling_helper as sh


def _new_seed():
    return int(torch.randint(0, 2 ** 31 - 1, (1,)))            # torch's CPU generator: torch.manual_seed makes runs repeatable


def sample_without_replacement(n, k, device, keys=None, seed=None):
    """k distinct indices of range(n) in random order (python ``random.sample(range(n), k)``).

    Default: element j is perm(j) for a keyed pseudo-random permutation of range(n) (``mf_sample_distinct``: Feistel
    network + cycle walking, O(k), seeded from torch's CPU generator unless ``seed`` is given).  With explicit ``keys``
    (n floats): the indices of the k largest keys (ties: lower index first) through the radix top-k kernel."""
    if k < 0 or k > n:
        raise ValueError("sample larger than population or is negative")          # python random.sample's own error
    if k == 0:
        return torch.empty(0, device=device, dtype=torch.int64)
    if keys is None:
        out = torch.empty(k, device=device, dtype=torch.int64)
        with torch.cuda.device(device):
            L.call("mf_sample_distinct", n, k, (_new_seed() if seed is None else int(seed)) & 0xffffffff, L.ptr(out), L.stream())
        return out
    if k > 4096:                                  # beyond the selection kernel's single-CTA sort (never reached by the shipped configs)
        return torch.argsort(keys.to(device), descending=True, stable=True)[:k]
    ones = torch.ones(1, n, device=device, dtype=torch.float32)
    return sh._topk(ones, k, (0, 0), keys)[0]


def frame_tensors(batch, device):
    """batch 'direction' (1,H,W,3) | (H,W,3), 'rgb' same, 'depth' (1,H,W) | (H,W) -> (dirs (H*W,3), rgb (H*W,3), depth (H*W),
    H, W): fp32 contiguous on ``device`` (no copy when already so)."""
    H, W = (int(s) for s in batch["depth"].shape[-2:])
    d = L.f32c(batch["direction"].reshape(-1, 3), device); c = L.f32c(batch["rgb"].reshape(-1, 3), device)
    z = L.f32c(batch["depth"].reshape(-1), device)
    if d.shape[0] != H * W or c.shape[0] != H * W or z.shape[0] != H * W:
        raise L.MipsFusionB200Error("frame: direction, rgb and depth are not all %d x %d" % (H, W))
    return d, c, z, H, W


def sample_frame_rays(batch, n, device, seed=None, idx=None, out=None, out_idx=None):
    """The mapping batch of submap initialisation (mipsfusion.py:176-180,207-211): ``n`` rays (n,7) [dir | rgb | depth] of
    distinct pixels of a full-resolution frame (``batch`` as :meth:`KeyframeRayStore.add_keyframe` takes it), the pixel
    index i decoded column-major (h = i % H, w = i // H) as the reference does.  The draw ``random.sample(range(H*W), n)``
    is made inside the gather (``mf_frame_sample_rays``; ``seed`` fixes it, torch's CPU generator when None); ``idx`` gives
    the draws instead: a host sequence is checked against [0, H*W) before it is copied, a device tensor is taken as it is.
    ``out`` (>= n, 7) / ``out_idx`` (n,) int64: optional device buffers for the rays / the drawn indices."""
    dev = torch.device(device)
    d, c, z, H, W = frame_tensors(batch, dev)
    n = int(n)
    if idx is not None:
        if not (isinstance(idx, torch.Tensor) and idx.is_cuda):
            idx = torch.as_tensor(idx, dtype=torch.int64).reshape(-1)
            if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= H * W):
                raise L.MipsFusionB200Error("sample_frame_rays: pixel indices outside [0, %d)" % (H * W))
        idx = idx.to(dev, torch.int64).contiguous()
        if idx.shape[0] != n:
            raise L.MipsFusionB200Error("sample_frame_rays: %d indices for %d rays" % (idx.shape[0], n))
    rays = torch.empty(n, 7, device=dev, dtype=torch.float32) if out is None else out[:n]
    with torch.cuda.device(dev):
        L.call("mf_frame_sample_rays", L.ptr(d), L.ptr(c), L.ptr(z), H, W, n, (_new_seed() if seed is None else int(seed)) & 0xffffffff,
               L.ptr(idx), L.ptr(rays), L.ptr(out_idx), L.stream())
    return rays


class KeyframeRayStore:
    def __init__(self, config, H, W, num_kf, device):
        self.config, self.H, self.W = config, int(H), int(W)
        self.device = torch.device(device)
        self.n_rays_h = int(config["sampling"]["kf_n_rays_h"])
        self.n_rays_w = int(config["sampling"]["kf_n_rays_w"])
        self.num_rays_to_save = self.n_rays_h * self.n_rays_w
        self.row_indices, self.col_indices = sh.sample_pixels_uniformly(self.H, self.W, self.n_rays_h, self.n_rays_w, device=self.device)
        self.rays = torch.zeros(num_kf, self.num_rays_to_save, 7, device=self.device, dtype=torch.float32)
        self.frame_ids = []

    def __len__(self):
        return len(self.frame_ids)

    get_length = __len__

    def add_keyframe(self, batch):
        """batch: 'direction' (1,H,W,3) | (H,W,3), 'rgb' same, 'depth' (1,H,W) | (H,W), 'frame_id' (keyframeSet.py:170-175)."""
        dev = self.device
        d = L.f32c(batch["direction"].reshape(-1, 3), dev); c = L.f32c(batch["rgb"].reshape(-1, 3), dev)
        z = L.f32c(batch["depth"].reshape(-1), dev)
        if d.shape[0] != self.H * self.W:
            raise L.MipsFusionB200Error("add_keyframe: frame is not %d x %d" % (self.H, self.W))
        slot = len(self.frame_ids)
        if slot >= self.rays.shape[0]:
            raise L.MipsFusionB200Error("keyframe ray store is full (%d keyframes)" % self.rays.shape[0])
        with torch.cuda.device(dev):
            L.call("mf_kf_store", L.ptr(d), L.ptr(c), L.ptr(z), L.ptr(self.row_indices), L.ptr(self.col_indices), self.W,
                   self.num_rays_to_save, L.ptr(self.rays[slot]), L.stream())
        self.frame_ids.append(int(batch["frame_id"]))

    @staticmethod
    def split_counts(pix_num, related_kf_num):
        """(first, other, last) ray counts of sample_rays_in_submap (keyframeSet.py:392-415)."""
        first = max(pix_num // related_kf_num, pix_num // 10)
        if related_kf_num == 1:
            return first, 0, 0
        if related_kf_num == 2:
            return first, pix_num - first, 0
        last = max(pix_num // related_kf_num, pix_num // 5)
        return first, pix_num - first - last, last

    def sample_rays_in_submap(self, first_kf_Id, related_kf_ids, pix_num, idx_first=None, idx_other=None, idx_last=None,
                              seed=None, out=None, return_draws=False, out_ids=None):
        """-> sampled_rays (n,7), kf_ids (n,), kf_indices (n,) on the device, in the reference's order (first keyframe,
        other related keyframes, latest keyframe).  idx_* : explicit index draws (int64); without them the draws are
        made inside the gather kernel (one launch; ``seed`` fixes them, ``return_draws`` also returns the indices).
        ``out``: optional (>= n, 7) device buffer that receives the rays; ``out_ids``: optional pair of (n,) int64 device
        buffers that receive kf_ids and kf_indices (device draws only)."""
        dev = self.device
        related = torch.as_tensor(related_kf_ids, dtype=torch.int64).reshape(-1)
        n_rel = int(related.shape[0])
        n_first, n_other, n_last = self.split_counts(int(pix_num), n_rel)
        nr = self.num_rays_to_save
        other_ids = related[1:-1] if n_rel > 2 else related[1:]
        if idx_first is None and idx_other is None and idx_last is None:
            n = n_first + n_other + n_last
            rays = torch.empty(n, 7, device=dev, dtype=torch.float32) if out is None else out[:n]
            if out_ids is None:
                kf_ids = torch.empty(n, device=dev, dtype=torch.int64); kf_indices = torch.empty_like(kf_ids)
            else:
                kf_ids, kf_indices = out_ids
            draws = torch.empty(n, device=dev, dtype=torch.int64) if return_draws else None
            key = tuple(int(v) for v in other_ids)
            cache = self.__dict__.setdefault("_ids_cache", {})
            other_d = cache.get(key)
            if other_d is None:
                other_d = cache[key] = other_ids.to(dev).contiguous()
            with torch.cuda.device(dev):
                L.call("mf_kf_sample_rays", L.ptr(self.rays), nr, int(first_kf_Id), L.ptr(other_d) if n_other else None,
                       int(other_ids.shape[0]), int(related[-1]), n_rel, n_first, n_other, n_last,
                       (_new_seed() if seed is None else int(seed)) & 0xffffffff, L.ptr(rays), L.ptr(kf_ids), L.ptr(kf_indices),
                       L.ptr(draws), L.stream())
            return (rays, kf_ids, kf_indices, draws) if return_draws else (rays, kf_ids, kf_indices)
        if idx_first is None:
            idx_first = sample_without_replacement(nr, n_first, dev)
        if n_other and idx_other is None:
            idx_other = sample_without_replacement(int(other_ids.shape[0]) * nr, n_other, dev)
        if n_last and idx_last is None:
            idx_last = sample_without_replacement(nr, n_last, dev)
        i64 = lambda t: None if t is None else torch.as_tensor(t, dtype=torch.int64).to(dev).contiguous()
        idx_first, idx_other, idx_last = i64(idx_first), i64(idx_other) if n_other else None, i64(idx_last) if n_last else None
        other_d = other_ids.to(dev).contiguous() if n_other else None
        n = n_first + n_other + n_last
        rays = torch.empty(n, 7, device=dev, dtype=torch.float32)
        kf_ids = torch.empty(n, device=dev, dtype=torch.int64); kf_indices = torch.empty_like(kf_ids)
        with torch.cuda.device(dev):
            L.call("mf_kf_gather_rays", L.ptr(self.rays), nr, int(first_kf_Id), L.ptr(other_d), int(related[-1]), n_rel,
                   L.ptr(idx_first), n_first, L.ptr(idx_other), n_other, L.ptr(idx_last), n_last,
                   L.ptr(rays), L.ptr(kf_ids), L.ptr(kf_indices), L.stream())
        return rays, kf_ids, kf_indices

    def sample_rays_in_given_kf(self, given_kf_ids, pix_num, idx=None):
        """keyframeSet.py:446-455: rays from the given keyframes only -> sampled_rays, kf_ids, kf_indices."""
        dev = self.device
        given = torch.as_tensor(given_kf_ids, dtype=torch.int64).reshape(-1)
        nr = self.num_rays_to_save
        if idx is None:
            idx = sample_without_replacement(int(given.shape[0]) * nr, int(pix_num), dev)
        idx = torch.as_tensor(idx, dtype=torch.int64).to(dev).contiguous()
        n = int(idx.shape[0])
        rays = torch.empty(n, 7, device=dev, dtype=torch.float32)
        kf_ids = torch.empty(n, device=dev, dtype=torch.int64); kf_indices = torch.empty_like(kf_ids)
        given_d = given.to(dev).contiguous()
        with torch.cuda.device(dev):
            # "other" segment only, with the given keyframes as the id table: kf_index = idx // n_rays (+1 removed below)
            L.call("mf_kf_gather_rays", L.ptr(self.rays), nr, 0, L.ptr(given_d), 0, int(given.shape[0]) + 1,
                   None, 0, L.ptr(idx), n, None, 0, L.ptr(rays), L.ptr(kf_ids), L.ptr(kf_indices), L.stream())
        return rays, kf_ids, kf_indices - 1
