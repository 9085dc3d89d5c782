"""CPU tests of the drop-in surface: the reference's UNMODIFIED example files (read from the reference checkout,
skipped where it is not available) import `rednose.helpers.*`, which this repository provides as a shim over
rednose_b200.  Generation goes through this package's gen_code; running goes through this package's
EKF_sym_pyx (native driver) -- pointed at the oracle's CPU build of the same C-ABI, since there is no GPU here."""
import importlib.util
import os
import re
import runpy
import sys

import numpy as np
import pytest

from oracle.build_ref import REF

REF_EXAMPLES = os.path.join(REF, "examples")
pytestmark = pytest.mark.skipif(not os.path.exists(REF_EXAMPLES), reason="the reference checkout ($REDNOSE_REFERENCE) is not available")


def _load(path, modname):
  spec = importlib.util.spec_from_file_location(modname, path)
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  return mod


def _protos(path):
  with open(path, encoding="utf-8") as f:
    return sorted(re.sub(r"\s+", " ", ln) for ln in f.read().split("\n") if ln.startswith("void "))


@pytest.mark.parametrize("script,name", [("kinematic_kf.py", "kinematic"), ("live_kf.py", "live")])
def test_reference_generator_scripts_run_unchanged(tmp_path, monkeypatch, gen_dir, script, name):
  """`python <filter>.py <target> <output_dir>` (site_scons/site_tools/rednose_filter.py:13) through this package."""
  import rednose
  assert "rednose_b200" in open(os.path.join(os.path.dirname(rednose.__file__), "helpers", "ekf_sym.py")).read()
  monkeypatch.setenv("REDNOSE_B200_NO_COMPILE", "1")
  monkeypatch.setattr(sys, "argv", [script, name, str(tmp_path)])
  runpy.run_path(os.path.join(REF_EXAMPLES, script), run_name="__main__")
  assert os.path.exists(tmp_path / f"{name}.cu") and os.path.exists(tmp_path / f"{name}.h")
  # same C-ABI as the library built from this repository's own definition of the model
  assert _protos(tmp_path / f"{name}.h") == _protos(os.path.join(gen_dir, f"{name}.h"))
  # same structure: the sparsity signature of F / H_err survives (33 F slots, per-kind non-zeros)
  sig = lambda p: re.findall(r"static constexpr int (?:NF|KIND) = [^;]*;", open(p).read())
  assert sig(tmp_path / f"{name}.cu") == sig(os.path.join(gen_dir, f"{name}.cu"))


def test_reference_kinematic_example_on_the_dropin_driver(oracle_dir):
  """examples/test_kinematic_kf.py:10-55 with the reference's own KinematicKalman class."""
  from tests.test_oracle_cpu import GOLDEN
  mod = _load(os.path.join(REF_EXAMPLES, "kinematic_kf.py"), "ref_kinematic_kf")
  np.random.seed(0)
  kf = mod.KinematicKalman(oracle_dir)
  assert type(kf.filter).__module__ == "rednose_b200.ekf_sym_pyx"
  dt = 0.01
  ts = np.arange(0, 5, step=dt)
  x = 0.0
  for t, v in zip(ts, np.sin(ts * 5)):
    kf.predict_and_observe(t, mod.ObservationKind.POSITION, [np.random.normal(x, 0.1)])
    x += v * dt
  got = (kf.x[0], np.sqrt(kf.P[0, 0]), kf.x[1], np.sqrt(kf.P[1, 1]))
  for g, want in zip(got, GOLDEN):
    assert abs(g - want) < 5e-8


def test_reference_live_example_on_the_dropin_driver(oracle_dir):
  """examples/live_kf.py's LiveKalman: uses .x as a live (DIM,1) view, .filter_time, rts_smooth (live_kf.py:269-306)."""
  mod = _load(os.path.join(REF_EXAMPLES, "live_kf.py"), "ref_live_kf")
  K = mod.ObservationKind
  kf = mod.LiveKalman(oracle_dir)
  rng = np.random.default_rng(0)
  estimates = []
  t = 0.0
  for k in range(30):
    t += 0.01
    if k % 10 == 0:
      r = kf.predict_and_observe(t, K.ECEF_POS, [kf.x[:3] + rng.normal(0, 1.0, 3)])
    elif k % 10 == 5:
      r = kf.predict_and_observe(t, K.CAMERA_ODO_TRANSLATION, [np.concatenate([rng.normal(0, 0.1, 3), [0.1, 0.1, 0.1]])])
    elif k % 10 == 7:
      r = kf.predict_and_observe(t, K.ODOMETRIC_SPEED, [[0.0]])
    else:
      r = kf.predict_and_observe(t, K.PHONE_GYRO, [rng.normal(0, 0.01, 3)])
    assert r is not None
    estimates.append(r)
    assert abs(np.linalg.norm(kf.x[3:7]) - 1.0) < 1e-12   # the example's own normalisation wrote through .x
    assert abs(kf.t - t) < 1e-12
  xs, Ps = kf.rts_smooth(estimates)
  assert xs.shape == (30, 23) and Ps.shape == (30, 22, 22) and np.isfinite(xs).all() and np.isfinite(Ps).all()
  assert Ps[10, 0, 0] <= estimates[10][3][0, 0] * (1 + 1e-9)
