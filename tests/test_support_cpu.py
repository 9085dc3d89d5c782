"""Support helpers the filter definitions and the gating thresholds rely on: chi-square quantiles
(rednose/helpers/chi2_lookup.py:15-18) and the rotation helpers (rednose/helpers/sympy_helpers.py)."""
import os

import numpy as np
import pytest
import sympy as sp

from rednose_b200 import geometry as geo
from rednose_b200.chi2 import chi2_ppf

# np.interp(0.95, arange(.01, .99, .01), chi2_lookup_table.npy[dim]) of the reference's shipped table
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "support_reference.npz")
REF_95 = {1: 3.8414588206941227, 2: 5.991464547107981, 3: 7.814727903251177, 6: 12.591587243743978, 17: 27.587111638275328,
          20: 31.410432844230925}


def test_chi2_quantiles_equal_the_reference_lookup():
  for dim, want in REF_95.items():
    assert abs(chi2_ppf(0.95, dim) - want) < 1e-12 * want
  g = np.load(GOLDEN)                                         # the whole table (tests/golden/make_golden_support.py)
  for dim, want in zip(g["chi2_dims"], g["chi2_values"]):
    for p, w in zip(g["chi2_probs"], want):
      assert abs(chi2_ppf(p, int(dim)) - w) < 1e-12 * w


def test_generated_gate_threshold_uses_that_quantile(gen_dir):
  """MAHA_THRESH baked into generated kinds = chi2_ppf(0.95, ZDIM): the generated-C path of the reference uses the
  dimension BEFORE the null-space projection (ekf_sym.py:144 `int(h_sym.shape[0])`, consumed at ekf_c.c:91), unlike
  its Python path (ekf_sym.py:604, y after projection); the CUDA backend follows the C path."""
  import re
  src = open(os.path.join(gen_dir, "msckf.cu"), encoding="utf-8").read() if os.path.exists(os.path.join(gen_dir, "msckf.cu")) else ""
  if not src:
    pytest.skip("msckf not generated")
  m = re.search(r"struct msckf_kind_17 \{.*?ZDIM = (\d+), YDIM = (\d+).*?MAHA = (\w+).*?MAHA_THRESH = ([0-9.e+-]+)", src, re.S)
  assert m and m.group(3) == "true" and int(m.group(1)) == 20 and int(m.group(2)) == 17
  assert abs(float(m.group(4)) - chi2_ppf(0.95, int(m.group(1)))) < 1e-9


def test_numeric_rotations_are_consistent():
  rng = np.random.default_rng(0)
  e = rng.uniform(-1.2, 1.2, (50, 3))
  q = geo.euler2quat(e)
  assert np.allclose(np.linalg.norm(q, axis=1), 1.0) and (q[:, 0] >= 0).all()
  R = geo.quat2rot(q)
  assert np.allclose(R @ np.transpose(R, (0, 2, 1)), np.eye(3), atol=1e-13) and np.allclose(np.linalg.det(R), 1.0)
  for k in range(5):
    assert np.allclose(R[k], geo.rot_matrix(*e[k]), atol=1e-13)          # R = Rz(yaw) Ry(pitch) Rx(roll)
    assert np.allclose(geo.euler2rot(e[k]), R[k], atol=1e-13)


def test_symbolic_helpers_match_the_numeric_ones_and_the_reference():
  r, p, y = sp.symbols("r p y")
  q = sp.symbols("q0:4")
  e = (0.3, -0.7, 1.1)
  Rs = np.array(geo.euler_rotate(r, p, y).subs(dict(zip((r, p, y), e)))).astype(float)
  assert np.allclose(Rs, geo.rot_matrix(*e), atol=1e-14)
  qn = geo.euler2quat(np.array(e))
  Rq = np.array(geo.quat_rotate(*q).subs(dict(zip(q, qn)))).astype(float)
  assert np.allclose(Rq, geo.quat2rot(qn), atol=1e-14)                    # symbolic and numeric quaternion -> rotation agree
  v = sp.Matrix(sp.symbols("a b c"))
  assert geo.cross(v) * v == sp.zeros(3, 1)
  g = np.load(GOLDEN)                                                     # the reference's helpers at fixed points
  for name, syms, args in (("euler_rotate", (r, p, y), (r, p, y)), ("quat_rotate", q, q), ("quat_matrix_r", q, (q,)), ("quat_matrix_l", q, (q,))):
    expr = sp.Matrix(getattr(geo, name)(*args))
    for pt, want in zip(g[f"{name}_points"], g[f"{name}_values"]):
      assert np.allclose(np.array(expr.subs(dict(zip(syms, pt)))).astype(float), want, rtol=0, atol=1e-14), name
