"""Per-array differences between two `bench.py --dump-outputs` directories (two runs of one build, or two builds).
    python scripts/compare_dumps.py DIR_A DIR_B"""
import os
import sys

import numpy as np

a_dir, b_dir = sys.argv[1], sys.argv[2]
for f in sorted(os.listdir(a_dir)):
    a, b = np.load(os.path.join(a_dir, f)), np.load(os.path.join(b_dir, f))
    if a.shape != b.shape:
        print(f"{f}: shapes differ {a.shape} vs {b.shape}")
        continue
    d = np.abs(a.astype(np.float64) - b.astype(np.float64))
    rel = np.linalg.norm(d) / max(np.linalg.norm(a.astype(np.float64)), 1e-30)
    print(f"{f}: {a.dtype} {a.shape}, max |a| {np.abs(a).max():.3e}, max abs diff {d.max():.3e}, relative L2 diff {rel:.3e}, "
          f"elements differing {int((d > 0).sum())}, > 1e-6 {int((d > 1e-6).sum())}, > 1e-4 {int((d > 1e-4).sum())}, "
          f"> 1e-2 {int((d > 1e-2).sum())}")
