"""CPU checks of the submap-initialisation oracle (oracle/submap_init.py): the per-iteration frame draw and its column-major
decode, and the current-frame rows of a BA iteration, each against a plain numpy restatement."""
import numpy as np
import torch

from oracle import keyframes as okf
from oracle import submap_init as oinit


def _frame(H, W, seed=0):
    g = torch.Generator().manual_seed(seed)
    depth = torch.rand(H, W, generator=g) * 4
    depth[torch.rand(H, W, generator=g) < 0.1] = 0.0
    return {"direction": torch.randn(H, W, 3, generator=g), "rgb": torch.rand(H, W, 3, generator=g), "depth": depth}


def test_frame_batch_is_the_column_major_gather_of_the_feistel_draw():
    H, W = 37, 53
    fr = _frame(H, W)
    for n, seed in ((1, 0), (700, 12345), (H * W, 0xfffffffe)):
        rays = oinit.frame_batch(fr, n, seed).numpy()
        i = okf.feistel_sample(H * W, n, seed)
        h, w = i % H, i // H
        ref = np.concatenate([fr["direction"].numpy()[h, w], fr["rgb"].numpy()[h, w], fr["depth"].numpy()[h, w][:, None]], 1)
        assert rays.shape == (n, 7)
        np.testing.assert_array_equal(rays, ref)
    assert np.array_equal(np.sort(okf.feistel_sample(H * W, H * W, 5)), np.arange(H * W))


def test_cur_frame_rays_are_the_lattice_then_the_top_keys():
    H, W, n_cur = 60, 80, 16 * 24 + 50
    fr = _frame(H, W, seed=3)
    keys = torch.rand(H * W, generator=torch.Generator().manual_seed(4))
    rays = oinit.cur_frame_rays(fr, n_cur, keys).numpy()
    # numpy: the 16 x 24 lattice (sampling_helper.py:38-48), then the valid off-lattice pixels by descending key
    ih, iw = (H - 16) // 17, (W - 24) // 25
    rl = np.arange(16) * (ih + 1) + ih + ((H - 16) % 17) // 2
    cl = np.arange(24) * (iw + 1) + iw + ((W - 24) % 25) // 2
    lat = (rl[:, None] * W + cl[None, :]).reshape(-1)
    v = (fr["depth"].numpy().reshape(-1) > 0) * keys.numpy()
    v[lat] = 0
    rest = np.argsort(-v, kind="stable")[:n_cur - lat.size]
    px = np.concatenate([lat, rest])
    flat = torch.cat([fr["direction"].reshape(-1, 3), fr["rgb"].reshape(-1, 3), fr["depth"].reshape(-1, 1)], 1).numpy()
    np.testing.assert_array_equal(rays, flat[px])
