"""Seeded SDF-like volumes for the marching-cubes tests (shared by tests/golden/make_mcubes_golden.py, the CPU and the GPU tests)."""
import numpy as np


def sphere(shape, centre, radius, noise=0.0, seed=0, scale=1.0):
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.arange(s, dtype=np.float32) for s in shape], indexing="ij"))
    c = np.asarray(centre, np.float32).reshape(3, 1, 1, 1)
    v = np.sqrt(((g - c) ** 2).sum(0)) - np.float32(radius)
    if noise:
        v = v + noise * rng.standard_normal(shape)
    return (v * scale).astype(np.float32)


def room(n, seed=0):
    """Two walls, a floor and a ball in a box: several sheets, tanh-compressed like a decoder's SDF in (-1, 1)."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float32)] * 3, indexing="ij")) / np.float32(n)
    d = np.minimum.reduce([g[0] - 0.12, 0.9 - g[1], g[2] - 0.2, np.sqrt(((g - 0.55) ** 2).sum(0)) - 0.17])
    d = d + 0.002 * rng.standard_normal(d.shape).astype(np.float32)
    return np.tanh(d * 12.0).astype(np.float32)


def cases():
    """name -> (volume, isovalue, truncation): small shapes that cover every branch of the reference routine."""
    rng = np.random.default_rng(7)
    out = {}
    out["sphere"] = (sphere((20, 22, 18), (9.3, 10.1, 8.6), 6.2), 0.0, 3.0)
    out["noisy_sphere"] = (sphere((24, 24, 24), (11.3, 12.2, 10.9), 7.5, noise=0.8, seed=1), 0.0, 3.0)          # truncation bites
    out["noise"] = (rng.standard_normal((14, 17, 12)).astype(np.float32), 0.0, 3.0)                                 # every case index
    v = sphere((26, 24, 22), (12.1, 11.4, 10.2), 8.0, noise=0.3, seed=2)
    v[5:9, 3:14, :] = -np.inf
    v[16:18] = np.nan
    v[:, :, 19:] = np.inf
    v[20:, 10:, :] = 5.0
    out["holes"] = (v, 0.0, 3.0)                                                                                    # -inf / nan / +inf / truncated
    out["scaled"] = (sphere((28, 28, 28), (13.7, 13.2, 14.4), 10.0, noise=0.2, seed=3, scale=0.01), 0.0, 3.0)      # near-equal corner values
    out["iso_shift"] = (sphere((20, 20, 20), (9.6, 9.9, 10.3), 5.0, noise=0.1, seed=4), 0.37, 3.0)
    out["integers"] = (np.round(sphere((18, 18, 18), (8.5, 8.5, 8.5), 5.0)).astype(np.float32), 0.0, 3.0)           # corners exactly on the level
    big = sphere((16, 16, 16), (7.7, 7.4, 8.1), 4.0, noise=0.2, seed=5, scale=7.0)
    out["thresh"] = (big, 0.0, 100.0)                                                                               # the thresh = 10 tests fire
    out["flat"] = (np.full((9, 9, 9), 0.5, np.float32), 0.0, 3.0)                                                   # no surface
    out["thin"] = (sphere((2, 12, 12), (0.5, 6, 6), 3.0), 0.0, 3.0)                                                 # no interior cell
    out["room"] = (room(32, seed=6), 0.0, 3.0)
    # vertices 1e-5 .. 1e-4 away from cell corners: integer voxels give nodes on multiples of 1/8; with the level 1.2e-5 below
    # 1.0 every node equal to 1.0 interpolates to mu = 1.2e-5 / (j / 8), i.e. 1-10 lattice steps from the corner along each of
    # its edges -> ADJACENT lattice cells, chains of them, and representatives two steps apart (the order-dependent part of the
    # reference's greedy clustering, marching_cubes.cpp:292-314,346-363)
    ints = np.random.default_rng(8).integers(-2, 3, size=(22, 20, 21)).astype(np.float32)
    out["lattice_chains"] = (ints, float(np.float32(1.0) - np.float32(1.2e-5)), 3.0)
    out["lattice_chains_eighths"] = (np.random.default_rng(9).integers(-2, 3, size=(18, 18, 18)).astype(np.float32) * 0.125,
                                     float(np.float32(0.125) - np.float32(1.1e-5)), 3.0)
    return out


def fresh_cases():
    """name -> (volume, isovalue, truncation): larger volumes than cases(), each at two levels (tests/golden/mcubes_fresh.npz)."""
    rng = np.random.default_rng(123)
    vols = {"sphere48": sphere((48, 40, 44), (23.1, 19.4, 22.2), 15.0, noise=0.3, seed=11),
            "room56": room(56, seed=12),
            "noise20": rng.standard_normal((20, 20, 20)).astype(np.float32) * 2.0,
            "sphere40_scaled": sphere((40, 40, 40), (19.7, 20.2, 19.9), 14.0, noise=0.1, seed=13, scale=0.001)}
    return {f"{name}_iso{k}": (vol, iso, 3.0) for name, vol in vols.items() for k, iso in enumerate((0.0, -0.21))}
