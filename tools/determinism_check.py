"""Repeat fit / predict on identical inputs and compare bits (race detector of last resort: compute-sanitizer is
closed on this pool).  Usage: python tools/determinism_check.py [N] [reps]"""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "nngp-src_b200"):
    sys.path.insert(0, str(p))
from nngp_b200 import _lib, synth  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 12
xtr, ytr, xte, _ = synth.make_problem(n, 4096, 128)
ytr = np.ones_like(ytr)
ref_alpha = ref_mean = ref_var = None
bad = 0
handles = [_lib.Handle() for _ in range(3)]
for r in range(reps):
    h = handles[r % 3]
    h.fit(xtr, ytr)
    a = h.get_state(x=False, l=False)["alpha"]
    m, v = h.predict(xte)
    if ref_alpha is None:
        ref_alpha, ref_mean, ref_var = a, m, v
        continue
    da, dm, dv = np.max(np.abs(a - ref_alpha)) / np.max(np.abs(ref_alpha)), np.max(np.abs(m - ref_mean)), np.max(np.abs(v - ref_var)) / np.max(ref_var)
    same = np.array_equal(a, ref_alpha) and np.array_equal(m, ref_mean) and np.array_equal(v, ref_var)
    if not same:
        bad += 1
        print(f"rep {r}: MISMATCH alpha rel {da:.3e} mean abs {dm:.3e} var rel {dv:.3e}", flush=True)
print(f"N={n} reps={reps} lookahead={os.environ.get('NNGP_CHOL_LOOKAHEAD', '1')} mismatches={bad}")
