"""Writes tests/golden/ref_eth_general.npz: outputs of the REFERENCE's PolynomialOptimization<N> templates for N = 6, 8, 12
(oracle/_ref/libref_eth_n{N}.so, compiled by oracle/Makefile from a checkout of the reference) on the inputs of
tests/test_general_shape.py::reference_cases.  Run: TG_REFERENCE_DIR=<checkout> python tests/golden/gen_golden_general.py"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib as O  # noqa: E402
import test_general_shape as T  # noqa: E402

O.build_oracle(ref=True)
out = {}
for n in (6, 8, 12):
    lib = C.CDLL(os.path.join(T.ROOT, "oracle", "_ref", f"libref_eth_n{n}.so"))
    for i, case in enumerate(T.reference_cases(n)):
        coef, cost = T.ref_outputs(lib, n, case)
        out[f"n{n}_coef_{i}"] = coef
        out[f"n{n}_cost_{i}"] = np.float64(cost)
np.savez_compressed(T.GOLDEN, **out)
print("wrote", T.GOLDEN, len(out), "arrays")
