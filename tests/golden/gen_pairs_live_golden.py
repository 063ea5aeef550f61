"""Generates tests/golden/pairs_live_golden.npz by EXECUTING the reference's own codegen (oracle/_ref/libref_pairs.so, see
gen_pairs_golden.py) on a fixed sample of the seeded random stencils of test_pair_derivatives_vs_reference_codegen_live: every 8th of its
200 draws of default_rng(7).standard_normal((4, 3)), so that the comparison runs where the reference sources are absent.
Run: python tests/golden/gen_pairs_live_golden.py"""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import refpairs as R

rng = np.random.default_rng(7)
X = np.stack([rng.standard_normal((4, 3)) for _ in range(200)])[::8]
out = {"X": X}
for name, f in [("g_PE", lambda x: R.g_PE(x[:3])), ("H_PE", lambda x: R.H_PE(x[:3])), ("g_PT", R.g_PT), ("H_PT", R.H_PT), ("g_EE", R.g_EE),
                ("H_EE", R.H_EE), ("cross_g", R.EEcross_g), ("cross_H", R.EEcross_H)]:
    out[name] = np.stack([f(x) for x in X])
p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pairs_live_golden.npz")
np.savez_compressed(p, **out)
print("wrote", p)
