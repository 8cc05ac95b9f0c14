"""N2 (marching cubes): the oracle restatement against the reference binary and the golden vectors it generated (CPU), and the
CUDA path through the C-ABI against the oracle / the golden vectors (GPU), bit for bit: vertices, their order, faces."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mc_volumes                                   # noqa: E402
from oracle import marching_cubes as omc            # noqa: E402


def _ensure_oracle():
    if not os.path.exists(os.path.join(os.path.dirname(omc.__file__), "libmcubes_oracle.so")):
        import subprocess
        subprocess.check_call(["make", "-C", os.path.dirname(omc.__file__), "-s"])


def _golden_cases(golden):
    g = golden("mcubes")
    names = sorted(k[:-len("_volume")] for k in g if k.endswith("_volume"))
    return [(n, g[n + "_volume"], float(g[n + "_args"][0]), float(g[n + "_args"][1]), g[n + "_verts"], g[n + "_faces"]) for n in names]


def _same(a, b):
    return a[0].shape == b[0].shape and a[1].shape == b[1].shape and np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_oracle_matches_reference_golden(golden):
    """oracle/mcubes_oracle.cpp == the reference's compiled marching_cubes.cpp on every fixture, bit for bit."""
    _ensure_oracle()
    cases = _golden_cases(golden)
    assert len(cases) >= 10
    for name, vol, iso, trunc, gv, gf in cases:
        v, f = omc.marching_cubes(vol, iso, trunc)
        assert v.dtype == np.float64 and f.dtype == np.uint64 and v.shape[1:] == (3,) and f.shape[1:] == (3,)
        assert _same((v, f), (gv.astype(np.float64), gf.astype(np.uint64))), name


def test_golden_volumes_are_the_seeded_ones(golden):
    """The committed fixtures are the volumes of tests/mc_volumes.py (so the generator script is reproducible)."""
    g = golden("mcubes")
    for name, (vol, iso, trunc) in mc_volumes.cases().items():
        assert np.array_equal(g[name + "_volume"], vol, equal_nan=True), name


def test_oracle_matches_stored_outputs_on_fresh_volumes(golden):
    """Fresh seeds, larger shapes (mc_volumes.fresh_cases()): the restatement against the stored outputs of
    tests/golden/mcubes_fresh.npz, and against the reference's own routine as well where oracle/_ref has been built."""
    import hashlib
    _ensure_oracle()
    g = golden("mcubes_fresh")
    cases = mc_volumes.fresh_cases()
    assert len(cases) == 8
    for name, (vol, iso, trunc) in cases.items():
        assert hashlib.sha256(np.ascontiguousarray(vol).tobytes()).hexdigest() == str(g[name + "_sha256"]), name
        assert np.array_equal(g[name + "_args"], [iso, trunc]), name
        a = omc.marching_cubes(vol, iso, trunc)
        assert _same(a, (g[name + "_verts"].astype(np.float64), g[name + "_faces"].astype(np.uint64))), name
        if omc.have_reference():
            assert _same(a, omc.reference_marching_cubes(vol, iso, trunc)), name


def test_oracle_input_dtypes_and_errors():
    _ensure_oracle()
    vol = mc_volumes.sphere((12, 12, 12), (5.5, 5.2, 5.9), 3.0)
    a = omc.marching_cubes(vol, 0.0, 3.0)
    b = omc.marching_cubes(vol.astype(np.float64), 0.0, 3.0)
    assert _same(a, b) and a[0].shape[0] > 0
    with pytest.raises(RuntimeError):
        omc.marching_cubes(vol[0], 0.0, 3.0)


# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cuda_matches_golden(golden):
    import mipsfusion_b200 as mf
    for name, vol, iso, trunc, gv, gf in _golden_cases(golden):
        v, f = mf.marching_cubes.marching_cubes(vol, iso, trunc)
        assert v.dtype == np.float64 and f.dtype == np.uint64
        assert _same((v, f), (gv.astype(np.float64), gf.astype(np.uint64))), name


@pytest.mark.gpu
def test_cuda_matches_oracle_medium_volumes():
    """Shapes the oracle does in seconds; includes odd sizes, a tensor input already on the device and a non-zero level."""
    import torch
    import mipsfusion_b200 as mf
    _ensure_oracle()
    rng = np.random.default_rng(5)
    vols = [(mc_volumes.room(160, seed=21), 0.0, 3.0),
            (mc_volumes.sphere((97, 130, 71), (48.2, 64.9, 35.1), 30.0, noise=0.4, seed=22), 0.0, 3.0),
            (rng.standard_normal((40, 41, 42)).astype(np.float32), 0.1, 3.0),
            (mc_volumes.sphere((64, 64, 64), (31.7, 32.2, 31.9), 25.0, noise=0.05, seed=23, scale=0.0007), 0.0, 3.0),
            (mc_volumes.sphere((48, 48, 48), (23.7, 24.2, 23.9), 14.0, noise=0.3, seed=24, scale=6.0), 0.0, 50.0)]
    for i, (vol, iso, trunc) in enumerate(vols):
        ov, of_, soup = omc.marching_cubes(vol, iso, trunc, return_soup_count=True)
        dv, df, info = mf.marching_cubes_device(torch.from_numpy(vol).cuda(), iso, trunc, return_info=True)
        assert info["soup_triangles"] == soup, (i, info, soup)
        assert dv.dtype == torch.float32 and df.dtype == torch.int64
        assert np.array_equal(dv.cpu().numpy().astype(np.float64), ov), i
        assert np.array_equal(df.cpu().numpy().astype(np.uint64), of_), i


@pytest.mark.gpu
def test_cuda_edge_cases():
    import torch
    import mipsfusion_b200 as mf
    for shape in [(1, 1, 1), (2, 2, 2), (3, 3, 3), (2, 30, 30), (5, 3, 4)]:
        vol = mc_volumes.sphere(shape, [s / 2 for s in shape], 1.2)
        v, f = mf.marching_cubes.marching_cubes(vol, 0.0, 3.0)
        ov, of_ = omc.marching_cubes(vol, 0.0, 3.0)
        assert _same((v, f), (ov, of_)), shape
    v, f = mf.marching_cubes.marching_cubes(np.full((16, 16, 16), -np.inf, np.float32), 0.0, 3.0)
    assert v.shape == (0, 3) and f.shape == (0, 3)
    with pytest.raises(RuntimeError):
        mf.marching_cubes.marching_cubes(np.zeros((4, 4), np.float32), 0.0, 3.0)
    with pytest.raises(mf.MipsFusionB200Error):
        mf.marching_cubes.marching_cubes(np.zeros((4, 4, 4), np.float32), 0.0, float("inf"))
    # float64 input goes through the reference's double -> float narrowing
    vol = mc_volumes.sphere((20, 20, 20), (9.4, 9.9, 10.3), 6.0, noise=0.2, seed=3).astype(np.float64) + 1e-12
    assert _same(mf.marching_cubes.marching_cubes(vol, 0.0, 3.0), omc.marching_cubes(vol, 0.0, 3.0))
    assert _same(mf.marching_cubes.marching_cubes(torch.from_numpy(vol), 0.0, 3.0), omc.marching_cubes(vol, 0.0, 3.0))


@pytest.mark.gpu
def test_cuda_full_size_properties():
    """512^3 (BASELINE C5 grid): no oracle run at this size -- size-independent properties instead: determinism (two runs agree
    bit for bit), vertices on the level set, closedness of the sphere mesh (edges shared by exactly two faces, up to the
    reference's own near-duplicate vertices), and bit-exact agreement with the oracle on a 96-voxel-thick slab cut out of the
    same volume."""
    import torch
    import mipsfusion_b200 as mf
    n = 512
    ax = torch.arange(n, device="cuda", dtype=torch.float32)
    vol = torch.sqrt((ax[:, None, None] - 255.3) ** 2 + (ax[None, :, None] - 250.9) ** 2 + (ax[None, None, :] - 260.2) ** 2) - 200.0
    vol = torch.tanh(vol * 0.05)
    v1, f1, info = mf.marching_cubes_device(vol, 0.0, 3.0, return_info=True)
    v2, f2 = mf.marching_cubes_device(vol, 0.0, 3.0)
    assert torch.equal(v1, v2) and torch.equal(f1, f2)
    assert f1.shape[0] > 1_000_000 and int(f1.max()) == v1.shape[0] - 1
    # vertices lie on the sphere to interpolation accuracy
    r = torch.sqrt((v1[:, 0] - 255.3) ** 2 + (v1[:, 1] - 250.9) ** 2 + (v1[:, 2] - 260.2) ** 2)
    assert float((r - 200.0).abs().max()) < 0.05
    # closed 2-manifold up to the reference's own near-duplicate vertices: count edges by (min,max) pair
    e = torch.cat([f1[:, [0, 1]], f1[:, [1, 2]], f1[:, [2, 0]]])
    key = e.min(1).values * v1.shape[0] + e.max(1).values
    _, cnt = torch.unique(key, return_counts=True)
    frac_two = float((cnt == 2).float().mean())
    assert frac_two > 0.95, frac_two
    # slab parity against the oracle: rows [200, 296) of the volume, same columns
    slab = vol[200:296].contiguous()
    sv, sf = mf.marching_cubes_device(slab, 0.0, 3.0)
    ov, of_ = omc.marching_cubes(slab.cpu().numpy(), 0.0, 3.0)
    assert np.array_equal(sv.cpu().numpy().astype(np.float64), ov) and np.array_equal(sf.cpu().numpy().astype(np.uint64), of_)


@pytest.mark.gpu
def test_joint_query_extract_mesh_on_device():
    """JointSubmapQuery.extract_mesh (query -> volume -> marching cubes -> vertex colours, all on the device): the mesh equals the
    oracle's marching cubes run on the very volume the device produced (bit for bit), masked grid points carry -inf, the world
    coordinates follow Mesher.py:535-543, and the colours equal a separate colour query at the vertices."""
    import torch
    import mipsfusion_b200 as mf
    import helpers as H
    from test_gpu_tracking_query import _submaps
    cfg = H.make_config(12)
    cfg["grid"]["use_bound_normalize"] = False
    fields, models, poses, amin, amax, cents = _submaps(3, cfg)
    axes = mf.get_grid_uniform(np.array([-0.2, 1.0, -0.6]), np.array([2.4, 4.8, 1.6]), voxel_size=0.09)
    jq = mf.JointSubmapQuery(models, poses, amin, amax, cents)
    out = jq.extract_mesh(axes)
    vol = out["sdf_volume"].cpu().numpy()
    assert vol.shape == tuple(len(a) for a in axes)
    ref = jq.query(axes=axes)
    nx, ny, nz = vol.shape
    mask = ref["mask"].reshape(ny, nx, nz).transpose(0, 1).cpu().numpy()
    assert np.all(np.isneginf(vol[~mask])) and np.all(np.isfinite(vol[mask])) and (~mask).any() and mask.any()
    assert np.array_equal(vol[mask], ref["sdf"].reshape(ny, nx, nz).transpose(0, 1).cpu().numpy()[mask])
    ov, of_ = omc.marching_cubes(vol, 0.0, 3.0)
    assert of_.shape[0] > 100
    assert np.array_equal(out["faces"].cpu().numpy().astype(np.uint64), of_)
    origin = np.array([a[0] for a in axes]); spacing = np.array([a[2] - a[1] for a in axes])
    assert np.allclose(out["vertices"].cpu().numpy(), (ov * spacing + origin).astype(np.float32), rtol=0, atol=1e-6)
    col = jq.query(points=(ov * spacing + origin), color=True)["rgb"]
    assert torch.equal(col, out["colors"]) and out["colors"].shape == (ov.shape[0], 3)


@pytest.mark.gpu
def test_cuda_greedy_clustering_chains():
    """The order-dependent part of the reference's vertex clustering: volumes whose vertices fall into ADJACENT 1e-5 lattice cells
    (see mc_volumes.cases()['lattice_chains']), at sizes where thousands of such chains exist.  The device resolves them as a
    fixed point (possibly several rounds); the result must still be the sequential one, bit for bit."""
    import torch
    import mipsfusion_b200 as mf
    _ensure_oracle()
    rounds, chains = [], []
    for seed, shape, step in [(31, (64, 60, 62), 1.0), (32, (80, 80, 80), 1.0), (33, (48, 50, 52), 0.5)]:
        vol = np.random.default_rng(seed).integers(-2, 3, size=shape).astype(np.float32) * np.float32(step)
        iso = float(np.float32(step) - np.float32(1.2e-5))
        ov, of_ = omc.marching_cubes(vol, iso, 3.0)
        dv, df, info = mf.marching_cubes_device(torch.from_numpy(vol).cuda(), iso, 3.0, return_info=True)
        rounds.append(info["rounds"])
        assert np.array_equal(dv.cpu().numpy().astype(np.float64), ov), (seed, info)
        assert np.array_equal(df.cpu().numpy().astype(np.uint64), of_), (seed, info)
        # the fixture does what it is meant to: representatives two lattice steps apart exist (chains through a merged cell)
        k = (ov.astype(np.float32) / np.float32(1e-5) + np.float32(0.5) * np.sign(ov.astype(np.float32))).astype(np.int64)
        keys = set(map(tuple, k[:30000]))
        chains.append(sum((a + d[0], b + d[1], c + d[2]) in keys for (a, b, c) in keys
                          for d in ((2, 0, 0), (0, 2, 0), (0, 0, 2), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, -1, 0), (1, 0, -1), (0, 1, -1))))
    print("clustering rounds:", rounds, "representative pairs <= 2 lattice steps apart:", chains)
    assert sum(chains) > 100, chains


@pytest.mark.gpu
def test_extract_mesh2_on_device(tmp_path):
    """extract_mesh2 (utils/utils.py:121-207, the caller of the in-tree marching cubes): the SDF volume against the oracle field
    evaluated by the reference's composition on the CPU (1e-3), the mesh against the oracle's marching cubes on the device's own
    volume pushed through the reference's vertex arithmetic (bit for bit), the colours against the oracle (1e-3), and the PLY."""
    import torch
    import mipsfusion_b200 as mf
    import helpers as H
    _ensure_oracle()
    cfg = H.make_config(12)
    cfg["data"]["translation"] = 0
    of = H.oracle_field(cfg, grid_scale=0.5, seed=3)
    model = H.cuda_model(cfg, H.state_of(of), train=False)
    bb = torch.tensor(cfg["mapping"]["bound"], dtype=torch.float64)
    c2w = torch.eye(4)
    c2w[:3, :3] = torch.tensor([[0.9950042, -0.0998334, 0.0], [0.0998334, 0.9950042, 0.0], [0.0, 0.0, 1.0]])
    c2w[:3, 3] = torch.tensor([0.05, -0.1, 0.02])
    path = str(tmp_path / "mesh" / "submap.ply")
    out = mf.extract_mesh2(model.query_sdf, c2w.cuda(), cfg, bb.cuda(), color_func=model.query_color, resolution=28, mesh_savepath=path,
                           slab_points=5000)                                     # several slabs
    tx, ty, tz = mf.getVoxels(bb[0, 1], bb[0, 0], bb[1, 1], bb[1, 0], bb[2, 1], bb[2, 0], None, 28)
    q = torch.stack(torch.meshgrid(tx, ty, tz, indexing='ij'), -1).to(torch.float32)
    w2l = c2w.inverse()
    flat = (w2l[:3, :3] @ q.reshape(-1, 3).to(bb[:, 0]).to(w2l).T + w2l[:3, 3:]).T
    flat = (flat - bb[:, 0]) / (bb[:, 1] - bb[:, 0])
    with torch.no_grad():
        vol_o = of.query_sdf(flat[:, None, :]).reshape(28, 28, 28).numpy()
    vol = out["sdf_volume"].cpu().numpy()
    assert H.rel_err(vol, vol_o) < 1e-3
    ov, of_ = omc.marching_cubes(vol, 0.0, 3.0)
    assert of_.shape[0] > 50 and np.array_equal(out["triangles"], of_)
    v = ov.copy()
    v /= np.array([[27, 27, 27]])
    scale = np.array([tx.numpy()[-1] - tx.numpy()[0], ty.numpy()[-1] - ty.numpy()[0], tz.numpy()[-1] - tz.numpy()[0]])
    v = scale[np.newaxis, :] * v + np.array([tx.numpy()[0], ty.numpy()[0], tz.numpy()[0]])
    v = v / cfg["data"]["sc_factor"] - cfg["data"]["translation"]
    assert np.array_equal(out["vertices"], v)
    vl = (w2l[:3, :3] @ torch.from_numpy(v).to(bb).to(w2l).T + w2l[:3, 3:]).T
    with torch.no_grad():
        col_o = of.query_color(vl[:, None, :]).reshape(-1, 3).numpy()
    assert H.rel_err(out["colors"], col_o) < 1e-3
    raw = open(path, "rb").read()
    head = raw[:raw.index(b"end_header\n") + 11].decode()
    assert f"element vertex {v.shape[0]}" in head and f"element face {of_.shape[0]}" in head
    assert len(raw) == len(head) + v.shape[0] * 16 + of_.shape[0] * 13
