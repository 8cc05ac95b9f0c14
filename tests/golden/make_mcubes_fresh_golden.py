"""Generates tests/golden/mcubes_fresh.npz: marching cubes of the volumes of tests/mc_volumes.py:fresh_cases().
The outputs come from the reference's own routine (oracle/_ref/_mcubes_ref.so, recipe: oracle/Makefile) when it has been built,
and otherwise from the C++ restatement oracle/mcubes_oracle.cpp, which matches that routine bit for bit on every fixture of
tests/golden/mcubes.npz.  The file records which one in `source`.
    make -C oracle && python tests/golden/make_mcubes_fresh_golden.py
Per case: the SHA-256 of the volume's bytes (the volumes are regenerated from their seeds, not stored), vertices as float32
(the routine's values are floats widened to double) and faces as uint32."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import marching_cubes as omc          # noqa: E402
import mc_volumes                                  # noqa: E402

source = "reference" if omc.have_reference() else "oracle"
run = omc.reference_marching_cubes if source == "reference" else omc.marching_cubes
out = {"source": np.array(source)}
for name, (vol, iso, trunc) in mc_volumes.fresh_cases().items():
    v, f = run(vol, iso, trunc)
    assert np.array_equal(v.astype(np.float32).astype(np.float64), v)
    out[name + "_sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(vol).tobytes()).hexdigest())
    out[name + "_args"] = np.array([iso, trunc], np.float64)
    out[name + "_verts"] = v.astype(np.float32)
    out[name + "_faces"] = f.astype(np.uint32)
    print(name, vol.shape, iso, v.shape, f.shape)
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "mcubes_fresh.npz"), **out)
print("source:", source)
