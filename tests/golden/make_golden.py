"""Generates the golden vectors of the reference's own bruteForceSearchORB (src/features.cpp:163-182 of the reference tree,
compiled into oracle/_ref by oracle/Makefile, which reads the tree from REF):
  brute_force_orb.npz         hand-shaped cases (ties, a best match in the last train row, a single train row, ...)
  brute_force_orb_random.npz  the uniformly random cases of tests/test_oracle.py::test_brute_force_orb_matches_reference_binary
Run where the reference tree is present; the .npz files are committed, so the tests need neither the tree nor oracle/_ref."""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
from oracle import oracle  # noqa: E402

oracle.build(force=True)
assert oracle.ref_lib() is not None, "reference tree missing: cannot regenerate golden vectors"
rng = np.random.default_rng(20260922)
cases = {}
for name, nq, nt in [("a", 64, 200), ("b", 33, 2), ("c", 17, 1), ("d", 100, 129), ("ties", 40, 60)]:
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    if name == "ties":  # duplicated train rows -> equal distances, lowest index must win
        t[30:] = t[:30]
        q[:10] = t[5:15]
    if name == "a":  # near-duplicates so that some hd < 128 and the LAST train row would be the best
        q[:20] = t[-20:] ^ rng.integers(0, 2, (20, 32), dtype=np.uint8)
    hd, idx = oracle.ref_brute_force_orb(q, t)
    cases[f"{name}_q"], cases[f"{name}_t"], cases[f"{name}_hd"], cases[f"{name}_idx"] = q, t, hd, idx
np.savez_compressed(Path(__file__).parent / "brute_force_orb.npz", **cases)
print("wrote", Path(__file__).parent / "brute_force_orb.npz", {k: v.shape for k, v in cases.items()})

rng = np.random.default_rng(5)
cases = {}
for i, (nq, nt) in enumerate([(50, 300), (7, 2), (3, 1), (128, 1000)]):
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    hd, idx = oracle.ref_brute_force_orb(q, t)
    cases[f"r{i}_q"], cases[f"r{i}_t"], cases[f"r{i}_hd"], cases[f"r{i}_idx"] = q, t, hd, idx
np.savez_compressed(Path(__file__).parent / "brute_force_orb_random.npz", **cases)
print("wrote", Path(__file__).parent / "brute_force_orb_random.npz", {k: v.shape for k, v in cases.items()})
