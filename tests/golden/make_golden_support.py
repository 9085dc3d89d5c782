#!/usr/bin/env python3
"""Generate tests/golden/support_reference.npz from the reference's own support helpers.

  * chi2: the reference's shipped chi2_lookup_table.npy interpolated the way rednose/helpers/chi2_lookup.py does
    (np.interp over arange(.01, .99, .01)) at a few probabilities, for every dimension of the table;
  * rotations: euler_rotate, quat_rotate, quat_matrix_r and quat_matrix_l of rednose/helpers/sympy_helpers.py
    evaluated at fixed points.

The reference checkout is taken from $REDNOSE_REFERENCE (see oracle/build_ref.py).

  python tests/golden/make_golden_support.py
"""
import importlib.util
import os
import sys

import numpy as np
import sympy as sp

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
PROBS = np.array([0.5, 0.9, 0.95, 0.975, 0.123])


def main():
  sys.path.insert(0, REPO)
  from oracle.build_ref import REF
  t, grid = np.load(os.path.join(REF, "rednose", "helpers", "chi2_lookup_table.npy")), np.arange(.01, .99, .01)
  out = {"chi2_probs": PROBS, "chi2_dims": np.arange(1, t.shape[0]),
         "chi2_values": np.array([[np.interp(p, grid, t[d]) for p in PROBS] for d in range(1, t.shape[0])])}
  spec = importlib.util.spec_from_file_location("ref_sympy_helpers", os.path.join(REF, "rednose", "helpers", "sympy_helpers.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  rng = np.random.default_rng(0)
  e = sp.symbols("r p y")
  q = sp.symbols("q0:4")
  for name, syms, wrap in (("euler_rotate", e, False), ("quat_rotate", q, False), ("quat_matrix_r", q, True), ("quat_matrix_l", q, True)):
    pts = rng.uniform(-1.2, 1.2, (3, len(syms)))
    fn = getattr(mod, name)
    expr = sp.Matrix(fn(list(syms)) if wrap else fn(*syms))
    out[f"{name}_points"] = pts
    out[f"{name}_values"] = np.array([np.array(expr.subs(dict(zip(syms, p)))).astype(float) for p in pts])
  np.savez_compressed(os.path.join(HERE, "support_reference.npz"), **out)


if __name__ == "__main__":
  main()
