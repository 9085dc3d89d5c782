#!/usr/bin/env python3
"""Benchmark of the hot path: fused EKF predict+update steps/s over a batch of independent filters.

  python bench.py --gpus N --steps K --warmup W            # this engine on N B200s (torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's C path on the host cores

One "step" = one launch of <name>_batch_step_<kind> over the whole per-GPU batch: for every filter
one predict(dt) + one update_<kind> (rednose/templates/ekf_c.c:8-33 + :37-121).  Workloads
(BASELINE.json configs / north_star):

  live_1m       1,048,576 live_kf filters (DIM 23 / EDIM 22) per GPU, IMU stream alternating
                PHONE_GYRO (4) / PHONE_ACCEL (10) at 100 Hz plus an ECEF_POS fix (12) every 100 steps
  live_100k     same with 100,000 filters            kinematic_1m   1,048,576 kinematic filters, kind 1

Prints ONE JSON line (rank 0).  `value` is the device-resident throughput; `e2e` goes through the public
BatchedEKF.predict_and_update_batch call with observations in pinned HOST memory and the state estimate
copied back every step; `roofline` is the dominant kernel against the measured HBM peak; `cpu_baseline`
is the oracle's reference-equivalent C path on the host cores (bounded sample).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOADS = {
  # BASELINE.json configs -> named workloads, each with its own JSON line (roofline of ITS dominant kernel)
  "live_1m": dict(filter="live", batch=1 << 20, steps=200, warmup=5),           # the metric's headline config
  "live_100k": dict(filter="live", batch=100_000, steps=200, warmup=5),         # config 3
  "kinematic_1m": dict(filter="kinematic", batch=1 << 20, steps=200, warmup=5),  # config 2 (state fits L2: said so in the line)
  "kinematic_16m": dict(filter="kinematic", batch=1 << 24, steps=100, warmup=5),  # 1.2 GB of state: larger than L2, a true HBM measurement
  "live_rts": dict(filter="live", batch=125_000, steps=2, warmup=1),            # config 4: 1M / 8 GPUs = 125k per GPU, forward + RTS over a long history
  "msckf_10k": dict(filter="msckf", batch=10_000, steps=100, warmup=5),         # config 5: triangulation + gated feature update + augment
}
LIVE_R = {4: [0.025**2] * 3, 10: [0.5**2] * 3, 12: [5.0**2] * 3}
L2_BYTES = 126 << 20


def bytes_per_step(dim, edim, m, ea=0):
  """ALGORITHMIC bytes of one fused step (SURVEY.md section 8d): P and x read+written, z and R read, y written, dt read."""
  return 8 * (2 * edim * edim + 2 * dim + m + m * m + m + ea + 1)


def measured_peaks():
  try:
    with open(os.path.join(REPO, "MEASURED_PEAKS.json"), encoding="utf-8") as f:
      return float(json.load(f)["hbm_gbs"]), "measured"
  except Exception:  # pylint: disable=broad-except
    return 6650.0, "fallback"


DUMP_BYTES = 60_000_000   # --dump-outputs stays under 64 MB, .npy headers included


def dump_sample(B, doubles_per_filter):
  """Sorted filter indices whose outputs --dump-outputs writes: every filter when they fit in DUMP_BYTES, else a fixed
  seeded sample (the same for every run with the same batch size)."""
  n = min(B, DUMP_BYTES // (8 * doubles_per_filter))
  if n == B:
    return np.arange(B, dtype=np.int64)
  return np.sort(np.random.default_rng(0).choice(B, n, replace=False))


def write_dump(folder, arrays):
  os.makedirs(folder, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(folder, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def kind_schedule(filter_name, n):
  if filter_name == "kinematic":
    return [1] * n
  return [12 if i % 100 == 0 else (4 if i % 2 else 10) for i in range(n)]


class ClockSampler:
  """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
  Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

  def __init__(self, gpu_index):
    self.rows, self.proc, self.idx = [], None, gpu_index

  def __enter__(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except OSError:
      self.proc = None
    return self

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(",")])

  def __exit__(self, *a):
    if self.proc:
      time.sleep(0.15)
      self.proc.terminate()
      self.thread.join(timeout=2)

  def summary(self):
    sm, mx, reasons = [], [], set()
    for r in self.rows:
      try:
        sm.append(float(r[0])); mx.append(float(r[1]))
      except (ValueError, IndexError):
        continue
      for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
        if v.lower().startswith("active"):
          reasons.add(name)
    if not sm:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- synthetic problem ---
def make_problem(filter_name, B, seed, lib_dir):
  """Synthetic states/covariances and per-kind observation pools (host numpy).  The observation mean
  h_k(x_true) is obtained through the product's own leaf entry points (<name>_h_<k>, one filter)."""
  rng = np.random.default_rng(seed)
  if filter_name == "kinematic":
    from rednose_b200.filters.kinematic import KinematicKalman as F
    x = np.tile(F.initial_x, (B, 1)) + rng.normal(size=(B, 2))
    P = np.diag(F.initial_P_diag)
    pools = {1: (rng.normal(0.0, 0.1, (4, B, 1)), np.tile(np.array([[0.1**2]]), (B, 1, 1)))}
    return x, P, F.Q.copy(), pools, (2, 2), []
  from rednose_b200.ekf_sym import EKF_sym
  from rednose_b200.filters.live import LiveKalman as F
  x_true = F.initial_x.copy()
  x_true[3:7] = [0.7, 0.1, -0.5, 0.5]
  x_true[3:7] /= np.linalg.norm(x_true[3:7])
  kf = EKF_sym(lib_dir, "live", F.Q, F.initial_x, np.diag(F.initial_P_diag), 23, 22)
  x = np.tile(x_true, (B, 1))
  x[:, 0:3] += rng.normal(0, 10.0, (B, 3))
  x[:, 7:10] += rng.normal(0, 1.0, (B, 3))
  x[:, 10:13] += rng.normal(0, 0.05, (B, 3))
  x[:, 17:20] += rng.normal(0, 0.3, (B, 3))
  pdiag = np.array([25.0] * 3 + [0.05**2] * 3 + [1.0] * 3 + [0.1**2] * 3 + [0.01**2] * 3 + [0.01**2] + [0.5**2] * 3 + [0.01**2] * 3)
  P = np.diag(pdiag)   # one covariance, broadcast to the batch on the device
  pools = {}
  for k, rdiag in LIVE_R.items():
    hz = np.zeros(3)
    kf.hs[k](x_true, np.zeros(1), hz)
    noise = rng.normal(size=(2, B, 3)) * np.sqrt(np.array(rdiag))
    pools[k] = (hz[None, None, :] + noise, np.tile(np.diag(rdiag), (B, 1, 1)))
  return x, P, F.Q.copy(), pools, (23, 22), [3]


# ----------------------------------------------------------------------------------- GPU arm ---
def run_gpu(args):
  import torch
  import torch.distributed as dist
  from rednose_b200.batched import BatchedEKF
  from rednose_b200.filters import ensure_generated

  wl = WORKLOADS[args.workload]
  fname, B = wl["filter"], (args.batch or wl["batch"])
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  if world != args.gpus:
    if world == 1 and args.gpus > 1:
      raise SystemExit("launch with torch.distributed.run for --gpus > 1")
  torch.cuda.set_device(local_rank)
  dev = torch.device("cuda", local_rank)
  from rednose_b200.sharding import bind_to_gpu_numa
  orig_affinity = os.sched_getaffinity(0)
  numa_node = bind_to_gpu_numa(local_rank)   # before any pinned allocation: staging buffers land on the GPU's socket
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)

  if fname == "kinematic":
    from rednose_b200.filters.kinematic import KinematicKalman as FilterCls
  else:
    from rednose_b200.filters.live import LiveKalman as FilterCls
  # only one rank per node may (re)build the filter library; the others wait
  if local_rank == 0:
    lib_dir = ensure_generated(FilterCls)
  if world > 1:
    dist.barrier()
  lib_dir = ensure_generated(FilterCls)

  x0, P0, Q, pools, (dim, edim), quat = make_problem(fname, B, seed=1234 + rank, lib_dir=lib_dir)
  eng = BatchedEKF(lib_dir, fname, Q, x0, P0, device=dev, quaternion_idxs=quat)
  dpools = {k: (torch.as_tensor(z).to(dev), torch.as_tensor(R).to(dev)) for k, (z, R) in pools.items()}
  dt_arr = torch.full((B,), 0.01, dtype=torch.float64, device=dev)
  zdim = {k: z.shape[-1] for k, (z, R) in pools.items()}
  zwork = {k: torch.empty(B, 1, zdim[k], dtype=torch.float64, device=dev) for k in pools}

  sched = kind_schedule(fname, args.warmup + args.steps)

  def one_step(i, kind):
    zp, R = dpools[kind]
    zwork[kind][:, 0, :].copy_(zp[i % zp.shape[0]])  # fresh observations (the kernel overwrites z with y)
    eng.step(kind, dt_arr, zwork[kind], R)

  def sync_all():
    torch.cuda.synchronize(dev)
    if world > 1:
      dist.barrier()
      torch.cuda.synchronize(dev)

  # ---- device-resident throughput ----
  for i in range(args.warmup):
    one_step(i, sched[i])
  sync_all()
  ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
  t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  launches0 = eng.launches
  with ClockSampler(local_rank) as clocks:
    sync_all()
    t0.record()
    for j in range(args.steps):
      i = args.warmup + j
      kind = sched[i]
      zp, R = dpools[kind]
      zwork[kind][:, 0, :].copy_(zp[i % zp.shape[0]])
      ev[j][0].record()
      eng.step(kind, dt_arr, zwork[kind], R)
      ev[j][1].record()
    t1.record()
    sync_all()
  elapsed_ms = t0.elapsed_time(t1)
  launches = eng.launches - launches0
  dumped = None
  if args.dump_outputs and rank == 0:   # what the last timed step returned, before anything else steps the filters
    idx = dump_sample(B, 1 + dim + edim * edim + zdim[sched[args.warmup + args.steps - 1]])
    sel = torch.as_tensor(idx, device=dev)
    dumped = {"filter_index": idx, "x": eng.x[sel].cpu().numpy(), "P": eng.P[sel].cpu().numpy(),
              "y": zwork[sched[args.warmup + args.steps - 1]][sel, 0, :].cpu().numpy()}
  if world > 1:
    tmax = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    elapsed_ms = float(tmax.item())
  per_kind = {}
  for j in range(args.steps):
    per_kind.setdefault(sched[args.warmup + j], []).append(ev[j][0].elapsed_time(ev[j][1]))
  assert bool(torch.isfinite(eng.x).all()), "filter diverged during the benchmark"

  # ---- sustained figure: the same loop for >= args.sustain seconds (power-capped clocks, not a burst) ----
  sustained = None
  if args.sustain > 0:
    n_s = max(args.steps, int(args.sustain * 1e3 / max(elapsed_ms / args.steps, 1e-3)))
    sched_s = kind_schedule(fname, n_s)
    with ClockSampler(local_rank) as clocks_s:
      sync_all()
      s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      s0.record()
      for i in range(n_s):
        one_step(i, sched_s[i])
      s1.record()
      sync_all()
    sus_ms = s0.elapsed_time(s1)
    if world > 1:
      tmax = torch.tensor([sus_ms], dtype=torch.float64, device=dev)
      dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
      sus_ms = float(tmax.item())
    sustained = {"value": B * n_s * world / (sus_ms * 1e-3), "unit": "steps/s", "steps": n_s, "seconds": sus_ms * 1e-3, "clocks": clocks_s.summary()}
    assert bool(torch.isfinite(eng.x).all())

  # ---- end to end through the public API: observations from pinned host memory, estimates back ----
  # HostStreamer.submit(t, kind, z_pinned_host, R) -> fused step -> x, y in pinned host memory, every step;
  # copies of consecutive steps overlap the kernel on separate streams.  P stays resident on the GPU.
  from rednose_b200.streaming import HostStreamer
  e2e_steps = max(3, args.e2e_steps)
  hz = {k: [torch.as_tensor(pools[k][0][j]).contiguous().pin_memory() for j in range(pools[k][0].shape[0])] for k in pools}
  Rsh = {k: torch.as_tensor(pools[k][1][0]).to(dev) for k in pools}   # one R per kind, shared by the batch (get_R semantics)
  streamer = HostStreamer(eng, zdim)
  eng.filter_time = 0.0
  tnow = 0.0

  def e2e_step(i, kind):
    nonlocal tnow
    tnow += 0.01
    return streamer.submit(tnow, kind, hz[kind][i % len(hz[kind])], Rsh[kind])

  for i in range(3):
    e2e_step(i, sched[i])
  streamer.wait()
  sync_all()
  streamer.h2d_bytes = streamer.d2h_bytes = 0
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for j in range(e2e_steps):
    e2e_step(j, sched[args.warmup + j])
  streamer.wait()                       # host-visible results of every step
  torch.cuda.current_stream(dev).wait_stream(streamer.s_out)
  e1.record()
  sync_all()
  e2e_ms = e0.elapsed_time(e1)
  if world > 1:
    tmax = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    e2e_ms = float(tmax.item())
  h2d = streamer.h2d_bytes / e2e_steps
  d2h = streamer.d2h_bytes / e2e_steps
  assert bool(torch.isfinite(streamer.x_host[0]).all())
  # the same loop when the caller asks only for the pose columns back (HostStreamer(out_cols=...)): live_kf position + attitude
  e2e_pose = None
  if fname == "live":
    del streamer
    streamer = HostStreamer(eng, zdim, out_cols=range(7))
    for i in range(3):
      e2e_step(i, sched[i])
    streamer.wait(); sync_all()
    streamer.h2d_bytes = streamer.d2h_bytes = 0
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for j in range(e2e_steps):
      e2e_step(j, sched[args.warmup + j])
    streamer.wait()
    torch.cuda.current_stream(dev).wait_stream(streamer.s_out)
    p1.record()
    sync_all()
    pose_ms = p0.elapsed_time(p1)
    if world > 1:
      tmax = torch.tensor([pose_ms], dtype=torch.float64, device=dev)
      dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
      pose_ms = float(tmax.item())
    e2e_pose = {"value": B * e2e_steps * world / (pose_ms * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": streamer.h2d_bytes / e2e_steps,
                "d2h_bytes_per_step": streamer.d2h_bytes / e2e_steps, "what": "as e2e, but only state columns 0..6 (ECEF position + attitude quaternion) and the innovations come back"}

  # ---- the stateless C-ABI entry point with HOST buffers: <name>_host_step_<kind>(x, P, Q, ..., z, R, ...) copies the
  #      whole state in and out (what calling the reference's <name>_predict + <name>_update_<k> on caller-owned
  #      host arrays does); PCIe-bound by construction (2 x (EDIM^2 + DIM) doubles per filter-step) ----
  host_abi = None
  if rank == 0:
    try:
      Bh = min(B, 131072)
      kind_h = sched[args.warmup + 1]
      ffi, lib = eng._ffi, eng._lib
      hx = eng.x[:Bh].cpu().pin_memory()
      hP = eng.P[:Bh].cpu().pin_memory()
      hzz = hz[kind_h][0][:Bh].clone().pin_memory()
      hRR = torch.as_tensor(pools[kind_h][1][:Bh]).contiguous().pin_memory()
      Qh = torch.as_tensor(np.ascontiguousarray(Q)).pin_memory()
      qi = ffi.new("int[]", list(quat) or [0])
      fn = getattr(lib, f"{fname}_host_step_{kind_h}")
      pp = lambda t: ffi.cast("double *", t.data_ptr())
      def host_call():
        fn(pp(hx), pp(hP), ffi.cast("const double *", Qh.data_ptr()), ffi.NULL, 0.01, pp(hzz), ffi.cast("const double *", hRR.data_ptr()),
           ffi.NULL, 1, Bh, qi, len(quat), eng.flags)
      host_call()
      t_h = time.perf_counter()
      n_h = 5
      for _ in range(n_h):
        host_call()                       # synchronous: returns when the results are back in the host arrays
      dt_h = (time.perf_counter() - t_h) / n_h
      host_abi = {"value": Bh / dt_h, "unit": "steps/s", "filters": Bh, "ms_per_call": dt_h * 1e3,
                  "h2d_bytes_per_step": 8 * Bh * (dim + edim * edim + zdim[kind_h] + zdim[kind_h]**2),
                  "d2h_bytes_per_step": 8 * Bh * (dim + edim * edim + zdim[kind_h]),
                  "what": f"{fname}_host_step_{kind_h}: x, P, z, R in pinned HOST memory in, x, P, y out, every call (chunked over 3 streams inside the library)"}
    except Exception as ex:  # pylint: disable=broad-except
      host_abi = {"error": repr(ex)[:200]}

  # ---- the reference's own calling pattern: ONE filter, host arrays, <name>_predict + <name>_update_<k> per call through the
  #      Python driver (BASELINE config 1 is this plumbing; the number says what a user who does NOT batch pays per call) ----
  single = None
  if rank == 0:
    try:
      from rednose_b200.ekf_sym import EKF_sym
      kf1 = EKF_sym(lib_dir, fname, Q, x0[0], P0 if P0.ndim == 2 else P0[0], dim, edim, quaternion_idxs=quat)
      k1 = sched[args.warmup + 1]
      z1, R1 = pools[k1][0][0][:1], pools[k1][1][:1]
      tt = 0.0
      for _ in range(20):
        tt += 0.01; kf1.predict_and_update_batch(tt, k1, z1, R1)
      n1 = 300
      t_s = time.perf_counter()
      for _ in range(n1):
        tt += 0.01; kf1.predict_and_update_batch(tt, k1, z1, R1)
      dt1 = (time.perf_counter() - t_s) / n1
      single = {"us_per_predict_and_update_batch": dt1 * 1e6, "steps_per_s": 1.0 / dt1, "kind": k1,
                "what": f"EKF_sym.predict_and_update_batch on ONE filter with host arrays: {fname}_predict + {fname}_update_{k1} through the C-ABI, each = one pinned staging copy in, a B = 1 launch, one copy out (cpu_baseline.python_driver_per_filter_steps_per_s is the same call pattern on the CPU library)"}
    except Exception as ex:  # pylint: disable=broad-except
      single = {"error": repr(ex)[:200]}

  # ---- final gather of the state estimates (the only collective of the system, SURVEY.md 8e) ----
  gather_ms = None
  if world > 1:
    from rednose_b200.sharding import gather_filters
    sync_all()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    out = gather_filters(eng.x, world * B)
    g1.record()
    sync_all()
    gather_ms = g0.elapsed_time(g1)
    # ... and the covariances (SURVEY.md section 8e: x and P), in slices of filters so that the gathered copy fits beside the state
    gp0, gp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    chunk = max(1, min(B, (8 << 30) // (world * edim * edim * 8)))
    gp0.record()
    for lo in range(0, B, chunk):
      outP = gather_filters(eng.P[lo:lo + chunk], world * min(chunk, B - lo))
    gp1.record()
    sync_all()
    gather_P_ms = gp0.elapsed_time(gp1)
    del out, outP

  # ---- the same K steps captured once into a CUDA graph and replayed (one driver call for the whole loop); measured LAST so that nothing else depends on it ----
  graph_line = None
  try:
    x_keep, P_keep = eng.x.clone(), eng.P.clone()
    def k_steps():
      for j in range(args.steps):
        one_step(args.warmup + j, sched[args.warmup + j])
    g = eng.capture(k_steps)
    eng.x.copy_(x_keep); eng.P.copy_(P_keep)
    sync_all()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.replay()                                   # warm
    eng.x.copy_(x_keep); eng.P.copy_(P_keep)
    sync_all()
    g0.record()
    g.replay()
    g1.record()
    sync_all()
    g_ms = g0.elapsed_time(g1)
    if world > 1:
      tmax = torch.tensor([g_ms], dtype=torch.float64, device=dev)
      dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
      g_ms = float(tmax.item())
    graph_line = {"value": B * args.steps * world / (g_ms * 1e-3), "unit": "steps/s", "ms_per_step": g_ms / args.steps,
                  "what": f"the same {args.steps} steps (observation refresh + fused launch each) captured into ONE CUDA graph (BatchedEKF.capture) and replayed"}
    assert bool(torch.isfinite(eng.x).all())
    del g
  except Exception as ex:  # pylint: disable=broad-except
    graph_line = {"error": repr(ex)[:200]}

  if rank == 0:
    peak, peak_kind = measured_peaks()
    dom = max(per_kind, key=lambda k: sum(per_kind[k]))
    dom_ms = float(np.mean(per_kind[dom]))
    algo = bytes_per_step(dim, edim, zdim[dom]) * B
    achieved = algo / (dom_ms * 1e-3) / 1e9
    traffic, traffic_src = None, "no ncu capture of this kernel at this batch size is committed"
    try:  # measured DRAM bytes per launch of this kernel from the committed ncu capture (same batch size only)
      with open(os.path.join(REPO, "profiles", "traffic.json"), encoding="utf-8") as f:
        tj = json.load(f)
      key = f"ekf_step<{fname}, kind {dom}>"
      if B == int(tj.get("batch", 1 << 20)) and key in tj:
        traffic, traffic_src = tj[key], f"profiles/traffic.json ({tj.get('capture', 'ncu --set full capture')}), not measured in this run"
    except Exception:  # pylint: disable=broad-except
      pass
    if edim <= 6:
      kern = "ekf_step_thread"
    elif edim <= 32:
      kern = "ekf_step_pair" if (edim % 2 == 0 and not os.environ.get("REDNOSE_B200_WARP_KERNEL", "").startswith("s")) else "ekf_step_warp"
    else:
      kern = "ekf_step_cta"
    total_steps = B * args.steps * world
    line = {
      "metric": "fused EKF predict+update steps/s (batched, float64)",
      "value": total_steps / (elapsed_ms * 1e-3),
      "unit": "steps/s",
      "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
      "ms_per_step": elapsed_ms / args.steps,
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "f64", "data": "synthetic",
      "config": {"workload": args.workload, "filter": fname, "filters_per_gpu": B, "dim": dim, "edim": edim,
                 "kind_schedule": "live: kinds 4/10 alternating + kind 12 every 100 steps" if fname == "live" else "kind 1",
                 "l2": f"inputs larger than L2 ({8 * B * edim * edim / 2**20:.0f} MiB of P per GPU vs 126 MiB)" if 8 * B * edim * edim > L2_BYTES else "inputs FIT in L2 (126 MiB)",
                 "sharding": "independent filters per GPU, no data-path collective"},
      "gpu_launches": launches,
      "per_kind_ms": {str(k): float(np.mean(v)) for k, v in per_kind.items()},
      "roofline": {"bound": "hbm", "kernel": f"{kern}<{fname}, kind {dom}>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                   "frac": achieved / peak, "peak_source": peak_kind, "algorithmic_bytes_per_step": bytes_per_step(dim, edim, zdim[dom]), "algorithmic_bytes_per_launch": algo,
                   "traffic": traffic, "traffic_source": traffic_src},
      "e2e": {"value": B * e2e_steps * world / (e2e_ms * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
              "steps": e2e_steps, "d2h_GBps_per_gpu": d2h / (e2e_ms / e2e_steps * 1e-3) / 1e9, "h2d_GBps_per_gpu": h2d / (e2e_ms / e2e_steps * 1e-3) / 1e9,
              "what": "HostStreamer.submit(t, kind, z_pinned_host, R_kind): H2D of z, fused step, D2H of x and y into pinned host memory EVERY step (3 streams overlap consecutive steps); P stays resident; bound by the device-to-host link (d2h_GBps_per_gpu vs ~55-63 GB/s for PCIe Gen5 x16)"},
      "clocks": clocks.summary(),
    }
    if e2e_pose is not None:
      line["e2e_pose_columns_only"] = e2e_pose
    if host_abi is not None:
      line["e2e_stateless_host_c_abi"] = host_abi
    if single is not None:
      line["single_filter_dropin"] = single
    if gather_ms is not None:
      line["final_gather_ms"] = gather_ms
      line["final_gather_P_ms"] = gather_P_ms
      line["final_gather_what"] = f"NCCL all-gather of x [{world * B}, {dim}] ({world * B * dim * 8 / 1e6:.0f} MB) and of P [{world * B}, {edim}, {edim}] ({world * B * edim * edim * 8 / 1e9:.2f} GB, in slices)"
    if sustained is not None:
      line["sustained"] = sustained
    if graph_line is not None:
      line["cuda_graph_replay"] = graph_line
    line["numa_node"] = numa_node
    line["timed_region"] = f"{args.steps} steps = {elapsed_ms:.1f} ms: a burst figure; 'sustained' repeats the loop for >= {args.sustain} s"
    if not args.no_cpu_baseline:
      os.sched_setaffinity(0, orig_affinity)   # the CPU arm may use every core the container has, not only the GPU's socket
      line["cpu_baseline"] = cpu_reference(fname, args.workload, budget_s=args.cpu_budget)
    if args.extras and world == 1:
      del eng, streamer, dpools
      torch.cuda.empty_cache()
      try:
        line["extras"] = run_extras(dev, peak)
      except Exception as ex:  # pylint: disable=broad-except
        line["extras"] = {"error": repr(ex)[:300]}
    print(json.dumps(line), flush=True)
  if dumped is not None:
    write_dump(args.dump_outputs, dumped)
  if world > 1:
    dist.barrier()   # the other ranks wait here while rank 0 times the CPU baseline
    dist.destroy_process_group()



# ------------------------------------------------- BASELINE config 4: forward + RTS over a long history ---
def _dist_setup(args):
  import torch
  import torch.distributed as dist
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  if world != args.gpus and world == 1 and args.gpus > 1:
    raise SystemExit("launch with torch.distributed.run for --gpus > 1")
  torch.cuda.set_device(local_rank)
  dev = torch.device("cuda", local_rank)
  from rednose_b200.sharding import bind_to_gpu_numa
  orig = os.sched_getaffinity(0)
  numa = bind_to_gpu_numa(local_rank)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  return torch, dist, rank, world, local_rank, dev, numa, orig


def _max_over_ranks(torch, dist, world, dev, vals):
  if world == 1:
    return [float(v) for v in vals]
  t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
  dist.all_reduce(t, op=dist.ReduceOp.MAX)
  return [float(v) for v in t.tolist()]


def run_rts(args):
  """live_kf sharded over the GPUs (125 000 filters per GPU = 1M over 8), forward filter + RTS smoother over a T-step
  history (--rts-steps, 10 000 in BASELINE.json; default 1 000 so that the default run takes a minute; cost is linear in T).
  The 81 MB per filter of a 10k-step history never materialises: CheckpointedSmoother keeps a checkpoint every `segment`
  steps, re-filters one segment with history and smooths it (rednose_b200/smoothing.py).  One bench "step" = one complete
  forward + backward job over the whole history; `value` = smoothed filter-steps per second (each one costs a plain fused
  step, a fused step that records history, and one RTS backward step)."""
  torch, dist, rank, world, local_rank, dev, numa, orig_aff = _dist_setup(args)
  from rednose_b200.filters import ensure_generated
  from rednose_b200.filters.live import LiveKalman
  from rednose_b200.smoothing import CheckpointedSmoother
  if local_rank == 0:
    ensure_generated(LiveKalman)
  if world > 1:
    dist.barrier()
  d = ensure_generated(LiveKalman)
  B, T, S = (args.batch or WORKLOADS["live_rts"]["batch"]), args.rts_steps, args.rts_segment
  x0, P0, Q, pools, (dim, edim), quat = make_problem("live", B, seed=4321 + rank, lib_dir=d)
  x0d = torch.as_tensor(x0).to(dev)
  P0d = torch.as_tensor(P0).to(dev).expand(B, -1, -1)
  # observations in pinned HOST memory (two realisations per kind), copied to the device inside the timed region every step
  hz = {k: [torch.as_tensor(np.ascontiguousarray(z[j])).pin_memory() for j in range(z.shape[0])] for k, (z, _) in pools.items()}
  Rk = {k: torch.as_tensor(R[0]).to(dev) for k, (_, R) in pools.items()}
  sched = kind_schedule("live", T)
  counters = {"h2d": 0, "d2h": 0}
  # observations: pinned host -> device on a copy stream, one step ahead of the kernels (two device slots), so the 3 MB
  # per step ride under the previous step's kernel instead of in front of it (same idea as streaming.HostStreamer)
  zslot = [torch.empty(B, 3, dtype=torch.float64, device=dev) for _ in range(2)]
  s_in = torch.cuda.Stream(dev)
  ev_in = [torch.cuda.Event() for _ in range(2)]
  ev_used = [torch.cuda.Event() for _ in range(2)]
  pre = {"k": None, "n": 0}

  def _enqueue(k, lo, hi, slot, wait_used):
    kind = sched[k]
    src = hz[kind][k % len(hz[kind])]
    if wait_used:
      s_in.wait_event(ev_used[slot])                  # the kernel that last used this slot has been enqueued and finished
    with torch.cuda.stream(s_in):
      zslot[slot][lo:hi].copy_(src[lo:hi], non_blocking=True)
      ev_in[slot].record(s_in)
    counters["h2d"] += (hi - lo) * 3 * 8

  def obs_fn(k, lo, hi):
    main = torch.cuda.current_stream(dev)
    n = pre["n"]
    if n:
      ev_used[(n - 1) % 2].record(main)               # everything enqueued so far (incl. the previous step) precedes this point
    slot = n % 2
    if pre["k"] != (k, lo, hi):                       # not prefetched (first step of a pass / segment)
      _enqueue(k, lo, hi, slot, n >= 2)
    main.wait_event(ev_in[slot])
    if k + 1 < T:
      _enqueue(k + 1, lo, hi, (n + 1) % 2, n >= 1)
      pre["k"] = (k + 1, lo, hi)
    else:
      pre["k"] = None
    pre["n"] = n + 1
    return 0.01 * (k + 1), sched[k], zslot[slot][lo:hi], Rk[sched[k]]

  # --dump-outputs: smoothed x and P of the last timed pass at a fixed seeded sample of steps and filters
  dump = {"on": False}
  if args.dump_outputs and rank == 0:
    d_steps = np.sort(np.random.default_rng(1).choice(T, min(T, 16), replace=False))
    d_filt = dump_sample(B, 1 + d_steps.size * (dim + edim * edim))
    dump.update(step_pos=np.full(T, -1), filt_pos=np.full(B, -1),
                x=torch.full((d_steps.size, d_filt.size, dim), float("nan"), dtype=torch.float64, device=dev),
                P=torch.full((d_steps.size, d_filt.size, edim, edim), float("nan"), dtype=torch.float64, device=dev))
    dump["step_pos"][d_steps] = np.arange(d_steps.size)
    dump["filt_pos"][d_filt] = np.arange(d_filt.size)

  def dump_block(lo, hi, k0, xs, Ps):
    sp, fp = dump["step_pos"][k0:k0 + xs.shape[0]], dump["filt_pos"][lo:hi]
    ts, fs = np.flatnonzero(sp >= 0), np.flatnonzero(fp >= 0)
    if ts.size and fs.size:
      rows, cols = torch.as_tensor(sp[ts], device=dev)[:, None], torch.as_tensor(fp[fs], device=dev)[None, :]
      ts, fs = torch.as_tensor(ts, device=dev), torch.as_tensor(fs, device=dev)
      dump["x"][rows, cols] = xs[ts][:, fs]
      dump["P"][rows, cols] = Ps[ts][:, fs]

  cs = CheckpointedSmoother(d, "live", Q, dim, edim, quaternion_idxs=quat, device=dev, hbm_budget_bytes=int(args.hbm_budget_gb) << 30, segment=S)
  tile, _ntiles = cs.plan(B, T)
  cs.tile = tile            # the warm-up run (shorter history) must use the same tiles as the timed run
  # smoothed pose columns go back to pinned host memory, segment by segment (the result a caller keeps; P stays on the device)
  pose_cols = 7
  # two slots: the device-to-host copy of one segment's poses runs on a side stream under the next segment's kernels
  host_out = [torch.empty(min(S + 1, T), tile, pose_cols, dtype=torch.float64).pin_memory() for _ in range(2)]
  stage = [torch.empty(min(S + 1, T), tile, pose_cols, dtype=torch.float64, device=dev) for _ in range(2)]
  s_out = torch.cuda.Stream(dev)
  ev_ready = [torch.cuda.Event() for _ in range(2)]
  ev_done = [torch.cuda.Event() for _ in range(2)]
  chk = {"finite": True, "n": 0, "k": 0}

  def sink(lo, hi, k0, xs, Ps):
    n = xs.shape[0]
    slot = chk["k"] % 2
    main = torch.cuda.current_stream(dev)
    if chk["k"] >= 2:
      main.wait_event(ev_done[slot])                     # the slot's previous copy has left the device
    stage[slot][:n, :hi - lo].copy_(xs[:, :, :pose_cols])
    ev_ready[slot].record(main)
    s_out.wait_event(ev_ready[slot])
    with torch.cuda.stream(s_out):
      host_out[slot][:n, :hi - lo].copy_(stage[slot][:n, :hi - lo], non_blocking=True)
      ev_done[slot].record(s_out)
    chk["k"] += 1
    counters["d2h"] += n * (hi - lo) * pose_cols * 8
    chk["n"] += n * (hi - lo)
    if k0 == 0:
      chk["finite"] = chk["finite"] and bool(torch.isfinite(xs[0]).all()) and bool(torch.isfinite(Ps[0]).all())
    if dump["on"]:
      dump_block(lo, hi, k0, xs, Ps)

  def sync_all():
    torch.cuda.synchronize(dev)
    if world > 1:
      dist.barrier()
      torch.cuda.synchronize(dev)

  # warm-up: a short history through the same objects (allocations, attribute setup), then W full-length passes only if asked
  Tw = min(T, 2 * S + 3)
  cs.run(x0d, P0d, Tw, obs_fn, sink, norm_quats=True)
  sync_all()
  from rednose_b200.batched import BatchedEKF  # noqa: F401  (launch counter lives on the engine)
  launches0 = cs._engine.launches
  counters["h2d"] = counters["d2h"] = 0
  chk["n"] = 0
  acc = {"forward_ms": 0.0, "reforward_with_history_ms": 0.0, "backward_ms": 0.0}
  t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  with ClockSampler(local_rank) as clocks:
    sync_all()
    t0.record()
    for i in range(args.steps):
      dump["on"] = args.dump_outputs is not None and rank == 0 and i == args.steps - 1
      cs.run(x0d, P0d, T, obs_fn, sink, norm_quats=True)
      for k_ in acc:
        acc[k_] += cs.stats[k_]
    torch.cuda.current_stream(dev).wait_stream(s_out)   # the last poses are in host memory before the clock stops
    t1.record()
    sync_all()
  elapsed_ms, fwd_ms, refwd_ms, bwd_ms = _max_over_ranks(torch, dist, world, dev, [t0.elapsed_time(t1), acc["forward_ms"], acc["reforward_with_history_ms"], acc["backward_ms"]])
  launches = cs._engine.launches - launches0
  assert chk["finite"] and chk["n"] == B * T * args.steps, (chk, B * T * args.steps)
  if rank == 0:
    peak, peak_kind = measured_peaks()
    K = args.steps
    nseg = cs.stats["segments"]
    bwd_steps = B * (T - 1) * K                       # backward recursions (the last step of the history only starts it)
    refwd_steps = B * (T + nseg - 1) * K              # each segment re-filters one extra step (the next segment's first)
    ach = 12176 * bwd_steps / (bwd_ms * 1e-3) / 1e9
    line = {
      "metric": "RTS-smoothed filter-steps/s (forward filter + checkpointed re-filter with history + RTS backward pass, float64)",
      "value": B * T * K * world / (elapsed_ms * 1e-3), "unit": "steps/s",
      "n_gpus": world, "steps": K, "warmup": 1, "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "f64", "data": "synthetic",
      "config": {"workload": "live_rts", "filter": "live", "filters_per_gpu": B, "history_steps": T, "baseline_history_steps": 10_000,
                 "extrapolation": "cost is linear in history_steps (per-step rates below); --rts-steps 10000 runs BASELINE.json's length",
                 "segment_steps": S, "segments": nseg, "tile_filters": cs.stats["tile_filters"], "tiles_per_pass": cs.stats["tiles"],
                 "hbm_bytes_per_filter": cs.stats["bytes_per_filter"], "full_history_bytes_per_filter": 8 * (2 * edim * edim + 2 * dim + 1) * T,
                 "kind_schedule": "kinds 4/10 alternating + kind 12 every 100 steps (first step is a position fix)", "norm_quats": True,
                 "l2": "inputs larger than L2", "sharding": "independent filters per GPU, no data-path collective"},
      "gpu_launches": launches,
      "phases": {"forward_steps_per_s": B * T * K / (fwd_ms * 1e-3), "reforward_with_history_steps_per_s": refwd_steps / (refwd_ms * 1e-3),
                 "backward_steps_per_s": bwd_steps / (bwd_ms * 1e-3), "forward_ms": fwd_ms, "reforward_with_history_ms": refwd_ms, "backward_ms": bwd_ms,
                 "other_ms": elapsed_ms - fwd_ms - refwd_ms - bwd_ms,
                 "reforward_frac_of_peak": (8240 + 8120) * refwd_steps / (refwd_ms * 1e-3) / 1e9 / peak, "forward_frac_of_peak": 8240 * B * T * K / (fwd_ms * 1e-3) / 1e9 / peak},
      "roofline": {"bound": "hbm", "kernel": "ekf_rts_warp_mma<live>", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_kind,
                   "algorithmic_bytes_per_step": 12176, "traffic": None, "traffic_source": "see profiles/ (ncu capture of the backward kernel)",
                   "note": "the backward step is ~45k FP64 FMA per filter-step (LDL^T, two triangular solves, two 24^3 products): at 64 FMA/clk/SM that alone is ~0.7 of this HBM roofline, so the kernel is FP64-pipe/latency bound, not bandwidth bound (DESIGN.md)"},
      "e2e": {"value": B * T * K * world / (elapsed_ms * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": counters["h2d"] / K, "d2h_bytes_per_step": counters["d2h"] / K,
              "what": "the timed region IS end to end: every step's observations are copied from pinned host memory (twice: both forward passes) and the smoothed pose columns of every step go back to pinned host memory"},
      "clocks": clocks.summary(), "numa_node": numa,
    }
    if not args.no_cpu_baseline:
      os.sched_setaffinity(0, orig_aff)
      line["cpu_baseline"] = cpu_rts_reference(budget_s=args.cpu_budget)
    print(json.dumps(line), flush=True)
  if dump["on"]:
    write_dump(args.dump_outputs, {"step_index": d_steps, "filter_index": d_filt, "x": dump["x"].cpu().numpy(), "P": dump["P"].cpu().numpy()})
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


def cpu_rts_reference(budget_s=15.0, T=40):
  """The reference's path for config 4 on the host: forward filter (oracle C, all usable cores) + rts_smooth, which the
  reference only has in Python/numpy (ekf_sym.py:651-690) -- timed one filter at a time, as shipped."""
  from oracle import build_ref
  from oracle.handle import Oracle
  from oracle.rts_numpy import rts_smooth
  o = Oracle(build_ref.OUT, "live")
  x, P, Q, pools, (dim, edim), quat = _cpu_problem("live", 8)
  P = np.tile(P, (8, 1, 1))
  sched = kind_schedule("live", T)
  hx_p, hx_f, hP_p, hP_f = [], [], [], []
  t0 = time.perf_counter()
  for k in range(T):
    xp, Pp = o.predict(x, P, Q, 0.01)
    for q in xp:
      q[3:7] /= np.linalg.norm(q[3:7])
    zp, R = pools[sched[k]]
    x, P, _ = o.update(sched[k], xp, Pp, zp[k % 2], R)
    for q in x:
      q[3:7] /= np.linalg.norm(q[3:7])
    hx_p.append(xp); hP_p.append(Pp); hx_f.append(x.copy()); hP_f.append(P.copy())
  t_fwd = time.perf_counter() - t0
  ts = 0.01 * (1 + np.arange(T))
  t1 = time.perf_counter()
  n = 0
  while n < 8 and time.perf_counter() - t1 < budget_s:
    rts_smooth(o, np.stack(hx_p)[:, n], np.stack(hx_f)[:, n], np.stack(hP_p)[:, n], np.stack(hP_f)[:, n], ts, 23, 22, norm_quats=True)
    n += 1
  t_bwd = time.perf_counter() - t1
  per_step = t_bwd / (n * (T - 1))
  return {"value": 1.0 / per_step, "unit": "steps/s", "cores": 1, "kind": "port", **_cpu_info(),
          "sample": f"{n} filters x {T - 1} backward steps of rts_smooth (numpy + cffi leaf calls, one filter at a time: the reference has no batched or C smoother)",
          "backward_steps_per_s_one_core": 1.0 / per_step, "what": "oracle/rts_numpy.py = restatement of rednose/helpers/ekf_sym.py:651-690 on the oracle library's leaf functions"}


# ---------------------------------------- BASELINE config 5: MSCKF, feature tracks with Mahalanobis rejection ---
def run_msckf(args):
  """10 000 MSCKF filters (live main state + 10 cloned camera poses, DIM 93 / EDIM 82).  One step = one camera frame:
  triangulate the tracked point from its 10 observations (compute_pos_batch, the front-end of SURVEY.md 8f-3), fused
  predict + null-space-projected, Mahalanobis-gated feature update with that point as extra_args, then augment (clone
  window shift).  5 % of the tracks are gross outliers (x50 noise) so that the gate fires."""
  torch, dist, rank, world, local_rank, dev, numa, orig_aff = _dist_setup(args)
  from rednose_b200.batched import BatchedEKF
  from rednose_b200.features import FeatureFrontend, to_c_matrix
  from rednose_b200.filters import ensure_generated
  from rednose_b200.filters.msckf import DIM, EDIM, MsckfKalman
  if local_rank == 0:
    ensure_generated(MsckfKalman); FeatureFrontend(10)
  if world > 1:
    dist.barrier()
  d = ensure_generated(MsckfKalman)
  fe = FeatureFrontend(10)
  B = args.batch or WORKLOADS["msckf_10k"]["batch"]
  g = torch.Generator(device=dev); g.manual_seed(77 + rank)
  f64 = dict(dtype=torch.float64, device=dev)

  def quat2rot_t(q):
    w, x, y, z = q.unbind(-1)
    return torch.stack([w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (w * y + x * z),
                        2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                        2 * (x * z - w * y), 2 * (w * x + y * z), w * w - x * x - y * y + z * z], -1).reshape(q.shape[:-1] + (3, 3))

  # initial state: the vehicle drives forward at 10 m/s, camera frames every 0.05 s -> clones 0.5 m apart
  dt, speed = 0.05, 10.0
  x0 = torch.as_tensor(MsckfKalman.initial_x).to(dev).repeat(B, 1)
  q = torch.randn(B, 4, generator=g, **f64); q = q / q.norm(dim=1, keepdim=True)
  Rm = quat2rot_t(q)
  x0[:, 0:3] += torch.randn(B, 3, generator=g, **f64) * 100.0
  x0[:, 3:7] = q
  x0[:, 7:10] = Rm[:, :, 0] * speed
  for c in range(10):
    o = 23 + 7 * c
    x0[:, o:o + 3] = x0[:, 0:3] - Rm[:, :, 0] * (speed * dt) * (10 - c)
    x0[:, o + 3:o + 7] = q
  pd = np.concatenate([[25.0] * 3 + [0.05**2] * 3 + [1.0] * 3 + [0.1**2] * 3 + [0.01**2] * 3 + [0.01**2] + [0.5**2] * 3 + [0.01**2] * 3] + [[1.0] * 3 + [0.02**2] * 3] * 10)
  eng = BatchedEKF(d, "msckf", MsckfKalman.Q, x0, np.diag(pd), device=dev, quaternion_idxs=[3] + [26 + 7 * c for c in range(10)])
  sigma = 1e-3
  Rk = torch.eye(20, **f64) * sigma**2
  to_c = torch.as_tensor(to_c_matrix().reshape(9)).to(dev)
  z_host = torch.empty(B, 20, dtype=torch.float64).pin_memory()
  x_host = torch.empty(B, DIM, dtype=torch.float64).pin_memory()
  stats = {"gated": 0, "tracks": 0, "bad_triangulations": 0, "count_bad": False}

  def make_obs():
    """a new landmark 15-50 m ahead of the newest clone, projected into the 10 clones (+ noise, 5 % gross outliers)"""
    clones = eng.x[:, 23:].reshape(B, 10, 7)
    Rl = quat2rot_t(clones[:, 9, 3:7])
    local = torch.stack([torch.rand(B, generator=g, **f64) * 35 + 15, torch.rand(B, generator=g, **f64) * 10 - 5, torch.rand(B, generator=g, **f64) * 6 - 3], 1)
    point = clones[:, 9, 0:3] + torch.einsum('bij,bj->bi', Rl, local)
    pc = torch.einsum('bcji,bcj->bci', quat2rot_t(clones[:, :, 3:7]), point[:, None, :] - clones[:, :, 0:3])   # R^T (p - pos)
    z = torch.stack([pc[:, :, 1] / pc[:, :, 0], pc[:, :, 2] / pc[:, :, 0]], -1).reshape(B, 20)
    noise = torch.randn(B, 20, generator=g, **f64) * sigma
    out = torch.rand(B, generator=g, device=dev) < 0.05
    noise[out] *= 50.0
    return (z + noise).contiguous(), out

  def hot_path(z):
    poses = eng.x[:, 23:].contiguous()                     # the 10 clones ARE the poses of the track: [B, 70]
    # a track whose triangulation does not converge (gross outliers: Gauss-Newton hits its 30-iteration cap or leaves the
    # finite range) gets a finite stand-in point 30 m down the optical axis (compute_pos_batch(fallback_depth=30)): its
    # huge residual is then what the Mahalanobis gate (ekf_c.c:88-94) exists to reject
    pos, param, iters = fe.compute_pos_batch(to_c, poses, z, fallback_depth=30.0)
    eng.step(17, dt, z, Rk, ea=pos, augment=True)          # fused predict + gated update + clone-window shift: one launch pair
    return pos

  def sync_all():
    torch.cuda.synchronize(dev)
    if world > 1:
      dist.barrier()
      torch.cuda.synchronize(dev)

  for _ in range(args.warmup):
    z, _o = make_obs()
    hot_path(z)
  sync_all()
  K = args.steps
  ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
  launches0 = eng.launches
  tr0 = None
  with ClockSampler(local_rank) as clocks:
    sync_all()
    for j in range(K):
      z, outl = make_obs()                                  # synthetic camera frame: NOT part of the timed hot path
      ev[j][0].record()
      last_pos = hot_path(z)
      ev[j][1].record()
      stats["tracks"] += B
    sync_all()
  dumped = None
  if args.dump_outputs and rank == 0:   # what the last timed frame returned, before the un-timed frames below step the filters
    idx = dump_sample(B, 1 + DIM + EDIM * EDIM + 20 + 3)
    sel = torch.as_tensor(idx, device=dev)
    dumped = {"filter_index": idx, "x": eng.x[sel].cpu().numpy(), "P": eng.P[sel].cpu().numpy(), "y": z[sel].cpu().numpy(),
              "point": last_pos[sel].cpu().numpy()}
  hot_ms = sum(a.elapsed_time(b) for a, b in ev)
  (hot_ms,) = _max_over_ranks(torch, dist, world, dev, [hot_ms])
  launches = 2 * (eng.launches - launches0) + K   # leaf + CTA kernel per fused step (the augment rides in the CTA kernel), + compute_pos per frame
  assert bool(torch.isfinite(eng.x).all()) and bool(torch.isfinite(eng.P).all()), "MSCKF diverged during the benchmark"
  # how often the gate fires (one extra un-timed frame, read off the clone block of the covariance)
  z, outl = make_obs()
  poses = eng.x[:, 23:].contiguous()
  pos, _, iters = fe.compute_pos_batch(to_c, poses, z, fallback_depth=30.0)
  ok = iters > 0
  maha_before = torch.einsum('bii->b', eng.P[:, 22:, 22:]).clone()
  eng.step(17, dt, z.clone(), Rk, ea=pos)
  gated = (torch.einsum('bii->b', eng.P[:, 22:, 22:]) > maha_before * (1 - 1e-9))
  eng.augment()
  # ---- e2e: observations from pinned host memory in, state estimate out, every frame ----
  e2e_K = min(K, 20)
  frames = []
  for _ in range(e2e_K):
    zf, _o = make_obs()
    frames.append(zf.cpu().pin_memory())
    hot_path(zf)
  eng.init_state(x0, torch.as_tensor(np.diag(pd)).to(dev), None)
  zd = torch.empty(B, 20, **f64)
  sync_all()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for j in range(e2e_K):
    zd.copy_(frames[j], non_blocking=True)
    hot_path(zd)
    x_host.copy_(eng.x, non_blocking=True)
  e1.record()
  sync_all()
  (e2e_ms,) = _max_over_ranks(torch, dist, world, dev, [e0.elapsed_time(e1)])
  if rank == 0:
    peak, peak_kind = measured_peaks()
    bs = 8 * (2 * EDIM * EDIM + 2 * DIM + 20 + 400 + 17 + 3 + 1)
    step_ms = hot_ms / K
    line = {
      "metric": "MSCKF camera-frame steps/s (triangulation + fused predict + gated feature update + augment, float64)",
      "value": B * K * world / (hot_ms * 1e-3), "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": step_ms,
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
      "config": {"workload": "msckf_10k", "filter": "msckf", "filters_per_gpu": B, "dim": DIM, "edim": EDIM, "clones": 10, "zdim": 20, "projected_dim": 17,
                 "outlier_fraction": 0.05, "gated_fraction_measured": float(gated.double().mean()), "outliers_among_gated": float((outl & gated).sum() / max(1, int(gated.sum()))),
                 "gauss_newton_iterations_mean": float(iters.abs().double().mean()), "triangulations_failed_fraction": float((~ok).double().mean()),
                 "l2": f"state {B * EDIM * EDIM * 8 / 2**20:.0f} MiB of P vs 126 MiB of L2: {'larger than L2' if B * EDIM * EDIM * 8 > L2_BYTES else 'FITS in L2'}",
                 "timing": "CUDA events around the hot-path calls of every frame; the synthetic observation generator between frames is excluded",
                 "sharding": "independent filters per GPU, no data-path collective"},
      "gpu_launches": launches,
      "roofline": {"bound": "hbm", "kernel": "ekf_step_cta<msckf, kind 17> (+ leaf, compute_pos, augment in the same timed region)", "achieved": bs * B / (step_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                   "frac": bs * B / (step_ms * 1e-3) / 1e9 / peak, "peak_source": peak_kind, "algorithmic_bytes_per_step": bs, "traffic": None,
                   "traffic_source": "see profiles/ (ncu capture of ekf_step_cta)"},
      "e2e": {"value": B * e2e_K * world / (e2e_ms * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": B * 20 * 8, "d2h_bytes_per_step": B * DIM * 8, "steps": e2e_K,
              "what": "per frame: z [B, 20] from pinned host memory, compute_pos + fused step + augment, x [B, 93] back to pinned host memory; P stays resident"},
      "clocks": clocks.summary(), "numa_node": numa,
    }
    if not args.no_cpu_baseline:
      os.sched_setaffinity(0, orig_aff)
      line["cpu_baseline"] = cpu_msckf_reference(budget_s=args.cpu_budget)
    print(json.dumps(line), flush=True)
  if dumped is not None:
    write_dump(args.dump_outputs, dumped)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


def cpu_msckf_reference(budget_s=15.0):
  """reference-generated MSCKF C (dense 82 x 82 Joseph form, full-pivot LU kernel of He) on all usable host cores."""
  from oracle import build_ref
  from oracle.handle import Oracle
  from tests.util import msckf_batch, msckf_feature_obs
  o = Oracle(build_ref.OUT, "msckf")
  cores = _threads()
  Bs = 64 * cores
  x, P, Q, point = msckf_batch(Bs, seed=5)
  z, R, _ = msckf_feature_obs(o, x, point, seed=6, outlier_frac=0.05)
  quats = [3] + [26 + 7 * c for c in range(10)]
  o.batch_step(17, x[:cores], P[:cores], Q, 0.01, z[:cores], R[:cores], ea=point[:cores], quat_idxs=quats, flags=3, nthreads=cores)
  t = time.perf_counter()
  n = 0
  while time.perf_counter() - t < budget_s and n < 20:
    o.batch_step(17, x, P, Q, 0.01, z, R, ea=point, quat_idxs=quats, flags=3, nthreads=cores)
    n += 1
  el = time.perf_counter() - t
  return {"value": Bs * n / el, "unit": "steps/s", "cores": cores, "threads": cores, "kind": "port", **_cpu_info(),
          "sample": f"{Bs} filters x {n} fused feature steps (predict + update_17), {el:.1f} s; includes the harness's array copies (~0.1 MB per filter-step against ~2 Mflop of dense algebra)",
          "what": "reference-generated leaf C + Eigen-free restatement of ekf_c.c, g++ -O2; compute_pos / augment not included (they are negligible beside the dense 82^3 products)"}


# ------------------------------------------------------------------ secondary kernels (extras) ---
def _time_ms(fn, iters, torch, dev):
  fn(); torch.cuda.synchronize(dev)
  t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t0.record()
  for _ in range(iters):
    fn()
  t1.record(); torch.cuda.synchronize(dev)
  return t0.elapsed_time(t1) / iters


def run_extras(dev, peak):
  """Short measurements of the other kernels of the path so every one has a number beside its roofline:
  kinematic (thread-per-filter), RTS backward pass, forward pass with history, MSCKF (CTA-per-filter)."""
  import torch
  from rednose_b200.batched import BatchedEKF
  from rednose_b200.filters import ensure_generated
  out = {}
  # kinematic: 1M (fits L2) and 16M (HBM)
  from rednose_b200.filters.kinematic import KinematicKalman
  d = ensure_generated(KinematicKalman)
  for label, B in (("kinematic_1m", 1 << 20), ("kinematic_16m", 1 << 24)):
    x0, P0, Q, pools, _, _ = make_problem("kinematic", B, 7, d)
    e = BatchedEKF(d, "kinematic", Q, x0, P0, device=dev)
    zp, R = torch.as_tensor(pools[1][0][0]).to(dev), torch.as_tensor(pools[1][1]).to(dev)
    dt = torch.full((B,), 0.01, dtype=torch.float64, device=dev)
    zw = torch.empty(B, 1, 1, dtype=torch.float64, device=dev)
    def step():
      zw[:, 0, :].copy_(zp)
      e.step(1, dt, zw, R)
    ms = _time_ms(step, 50, torch, dev)
    # the kernel alone (events around the launch only, the observation refresh copy outside)
    kms = []
    for _ in range(20):
      zw[:, 0, :].copy_(zp)
      k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      k0.record(); e.step(1, dt, zw, R); k1.record(); torch.cuda.synchronize(dev)
      kms.append(k0.elapsed_time(k1))
    kms = float(np.median(kms))
    out[label] = {"ms_per_step": ms, "steps_per_s": B / (ms * 1e-3), "kernel_ms": kms, "kernel_GBps_algorithmic": bytes_per_step(2, 2, 1) * B / (kms * 1e-3) / 1e9,
                  "kernel_frac_of_peak": bytes_per_step(2, 2, 1) * B / (kms * 1e-3) / 1e9 / peak,
                  "GBps_algorithmic": bytes_per_step(2, 2, 1) * B / (ms * 1e-3) / 1e9,
                  "frac_of_peak": bytes_per_step(2, 2, 1) * B / (ms * 1e-3) / 1e9 / peak, "note": "ms_per_step includes the 8 B/filter observation refresh copy; kernel_* do not"}
    del e, zp, R, dt, zw
  # live: forward with history + RTS backward (tile of filters sized so the history fits comfortably)
  from rednose_b200.filters.live import LiveKalman
  d = ensure_generated(LiveKalman)
  B, T = 1 << 16, 16
  x0, P0, Q, pools, _, quat = make_problem("live", B, 11, d)
  e = BatchedEKF(d, "live", Q, x0, P0, device=dev, quaternion_idxs=quat)
  dpool = {k: (torch.as_tensor(z[0]).to(dev), torch.as_tensor(R[0]).to(dev)) for k, (z, R) in pools.items()}
  hist = e.new_history(T)
  sched = kind_schedule("live", T)
  torch.cuda.synchronize(dev)
  t0, t1, t2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
  t0.record()
  for k in range(T):
    zk, Rk = dpool[sched[k]]
    e.step_recorded(hist, sched[k], 0.01 * (k + 1), zk.clone(), Rk)
  t1.record(); torch.cuda.synchronize(dev)
  _fwd_ms = t0.elapsed_time(t1) / T
  xs, Ps = e.rts_smooth(hist, norm_quats=True)   # warm-up (allocates the output slabs)
  torch.cuda.synchronize(dev)
  t1.record()
  xs, Ps = e.rts_smooth(hist, norm_quats=True, out=(xs, Ps))
  t2.record(); torch.cuda.synchronize(dev)
  bwd_ms = t1.elapsed_time(t2) / (T - 1)
  torch.cuda.synchronize(dev)
  fwd_ms = _fwd_ms
  out["live_forward_with_history"] = {"filters": B, "T": T, "ms_per_step": fwd_ms, "steps_per_s": B / (fwd_ms * 1e-3),
                                      "GBps_algorithmic": (8240 + 8120) * B / (fwd_ms * 1e-3) / 1e9, "frac_of_peak": (8240 + 8120) * B / (fwd_ms * 1e-3) / 1e9 / peak}
  out["live_rts_backward"] = {"filters": B, "T": T, "ms_per_step": bwd_ms, "steps_per_s": B / (bwd_ms * 1e-3),
                              "GBps_algorithmic": 12176 * B / (bwd_ms * 1e-3) / 1e9, "frac_of_peak": 12176 * B / (bwd_ms * 1e-3) / 1e9 / peak,
                              "finite": bool(torch.isfinite(xs).all() and torch.isfinite(Ps).all())}
  del e, hist, xs, Ps
  # config 4 in miniature: forward + RTS over a history that is tiled over filters (history = 8.1 kB per filter-step)
  try:
    from rednose_b200.smoothing import TiledSmoother
    B, T, tile = 32768, 32, 8192
    x0, P0, Q, pools, _, quat = make_problem("live", B, 17, d)
    P0 = np.broadcast_to(P0, (B, 22, 22))
    x0d, P0d = torch.as_tensor(x0).to(dev), torch.as_tensor(np.ascontiguousarray(P0)).to(dev)
    zp = {k: torch.as_tensor(v[0][0]).to(dev) for k, v in pools.items()}
    Rk = {k: torch.as_tensor(v[1][0]).to(dev) for k, v in pools.items()}
    sched = kind_schedule("live", T)
    acc = {"n": 0}
    def obs_fn(k, lo, hi):
      return 0.01 * (k + 1), sched[k], zp[sched[k]][lo:hi].clone(), Rk[sched[k]]
    def sink(lo, hi, xs, Ps):
      acc["n"] += int(torch.isfinite(xs).all())
    ts = TiledSmoother(d, "live", Q, 23, 22, quaternion_idxs=quat, device=dev, tile=tile)
    ts.run(x0d[:tile], P0d[:tile], T, obs_fn, sink, norm_quats=True)   # warm-up: allocations
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    ntiles = ts.run(x0d, P0d, T, obs_fn, sink, norm_quats=True)
    torch.cuda.synchronize(dev)
    el = time.perf_counter() - t0
    out["live_tiled_forward_plus_rts"] = {"filters": B, "T": T, "tile": tile, "tiles": ntiles, "seconds": el,
                                          "filter_steps_per_s": B * T / el, "finite_tiles": acc["n"],
                                          "note": "forward with history + backward RTS per tile, smoothed track handed to a sink; config 4 (1M x 10k over 8 GPUs) = 125k filters/GPU in tiles of ~1.8k"}
    del ts, x0d, P0d
  except Exception as ex:  # pylint: disable=broad-except
    out["live_tiled_forward_plus_rts"] = {"error": repr(ex)[:200]}
  # ragged streams: every tick ~60 % of 1M live filters see one observation of kind 4 / 10 / 12, the rest nothing
  try:
    from rednose_b200.scheduler import RaggedScheduler
    B = 1 << 20
    x0, P0, Q, pools, _, quat = make_problem("live", B, 13, d)
    e = BatchedEKF(d, "live", Q, x0, P0, device=dev, quaternion_idxs=quat)
    sch = RaggedScheduler(e)
    g = torch.Generator(device=dev); g.manual_seed(3)
    ticks = []
    for tk in range(6):
      act = (torch.rand(B, device=dev, generator=g) < 0.6).nonzero(as_tuple=True)[0]
      kk = torch.tensor([4, 10, 12], device=dev)[torch.randint(0, 3, (act.numel(),), device=dev, generator=g)]
      zs = {k: torch.as_tensor(pools[k][0][0]).to(dev)[act[kk == k]] for k in (4, 10, 12)}
      ticks.append((act, 0.01 * (tk + 1), kk, zs))
    Rs = {k: torch.as_tensor(pools[k][1][0]).to(dev) for k in (4, 10, 12)}
    sch.tick(ticks[0][0], ticks[0][1], ticks[0][2], ticks[0][3], Rs)   # warm-up
    torch.cuda.synchronize(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 0
    t0.record()
    for act, tt, kk, zs in ticks[1:]:
      sch.tick(act, tt, kk, zs, Rs)
      n += act.numel()
    t1.record(); torch.cuda.synchronize(dev)
    ms = t0.elapsed_time(t1)
    out["live_ragged_scheduler"] = {"filters": B, "ticks": len(ticks) - 1, "observations": n, "steps_per_s": n / (ms * 1e-3),
                                    "note": "bucketing by kind (torch index ops) + 3 indexed fused launches per tick", "finite": bool(torch.isfinite(e.x).all())}
    del e, sch, ticks
  except Exception as ex:  # pylint: disable=broad-except
    out["live_ragged_scheduler"] = {"error": repr(ex)[:200]}
  # MSCKF 10k: fused predict + feature-track update (null-space projection + gate), CTA-per-filter
  try:
    from rednose_b200.ekf_sym import EKF_sym
    from rednose_b200.filters.msckf import DIM, EDIM, MsckfKalman
    d = ensure_generated(MsckfKalman)
    B = 10_000
    rng = np.random.default_rng(5)
    xt = MsckfKalman.initial_x.copy()
    q = np.array([0.7, 0.1, -0.5, 0.5]); q /= np.linalg.norm(q)
    from rednose_b200.geometry import quat2rot
    Rm = quat2rot(q)
    xt[3:7] = q
    for c in range(10):
      o = 23 + 7 * c
      xt[o:o + 3] = xt[0:3] - Rm[:, 0] * 0.5 * (10 - c)
      xt[o + 3:o + 7] = q
    point = xt[0:3] + Rm @ np.array([30.0, 2.0, -1.0])
    kf = EKF_sym(d, "msckf", MsckfKalman.Q, xt, np.diag(MsckfKalman.initial_P_diag), 23, 22, N=10, dim_augment=7, dim_augment_err=6)
    hz = np.zeros(20)
    kf.hs[17](xt, point, hz)
    x0 = np.tile(xt, (B, 1)); x0[:, 0:3] += rng.normal(0, 0.5, (B, 3))
    pd = np.concatenate([[25.0] * 3 + [0.05**2] * 3 + [1.0] * 3 + [0.1**2] * 3 + [0.01**2] * 3 + [0.01**2] + [0.5**2] * 3 + [0.01**2] * 3] + [[1.0] * 3 + [0.02**2] * 3] * 10)
    e = BatchedEKF(d, "msckf", MsckfKalman.Q, x0, np.diag(pd), batch=B, device=dev, quaternion_idxs=[3] + [26 + 7 * c for c in range(10)])
    zp = torch.as_tensor(hz[None, :] + rng.normal(0, 1e-3, (B, 20))).to(dev)
    Rk = torch.as_tensor(np.eye(20) * 1e-6).to(dev)
    ea = torch.as_tensor(np.tile(point, (B, 1))).to(dev)
    def mstep():   # one camera frame: fused predict + gated feature update + clone-window shift (augment=True) in one launch pair
      e.step(17, 0.01, zp.clone(), Rk, ea=ea, augment=True)
    ms = _time_ms(mstep, 10, torch, dev)
    bs = 8 * (2 * EDIM * EDIM + 2 * DIM + 20 + 400 + 17 + 3 + 1)
    out["msckf_10k_feature_step"] = {"filters": B, "ms_per_step": ms, "steps_per_s": B / (ms * 1e-3), "GBps_algorithmic": bs * B / (ms * 1e-3) / 1e9,
                                     "frac_of_peak": bs * B / (ms * 1e-3) / 1e9 / peak, "finite": bool(torch.isfinite(e.x).all())}
  except Exception as ex:  # pylint: disable=broad-except
    out["msckf_10k_feature_step"] = {"error": repr(ex)[:200]}
  return out


# ------------------------------------------------------------------- reference arm / CPU baseline ---
CPU_WHAT = ("reference-generated leaf C (rednose gen_code, unmodified) + Eigen-free restatement of ekf_c.c, g++ -O2 -g -fPIC (SConstruct:25-38); "
            "per filter the call order of ekf_sym.cc:206-213; state resident in one arena first-touched and stepped IN PLACE by a pool of "
            "pinned worker threads (oracle/batch_runner.inc), no per-step array copies")


class CpuArm:
  """The reference's C path (oracle/_ref) on the host cores over a resident batch of filters, stepped in place."""

  def __init__(self, fname, B, nthreads=None, seed=99, pin=True):
    from oracle import build_ref
    from oracle.handle import Arena, Oracle
    if build_ref.reference_available():
      build_ref.build(fname)
    self.fname, self.B = fname, B
    self.o = Oracle(build_ref.OUT, fname)
    x, P, self.Q, self.pools, (self.dim, self.edim), self.quat = _cpu_problem(fname, B, seed)
    self.Q = np.ascontiguousarray(self.Q, dtype=np.float64)
    self.arena = Arena(self.o, B, nthreads=nthreads, pin=pin)
    self.arena.load(x, P)             # P [EDIM, EDIM] is broadcast; pages are first-touched by the workers
    self.sched = kind_schedule(fname, 4096)
    self.it = 0

  def step(self):
    k = self.sched[self.it % len(self.sched)]
    zp, R = self.pools[k]
    self.arena.step(k, self.Q, 0.01, zp[self.it % zp.shape[0]], R, quat_idxs=self.quat, flags=3)
    self.it += 1

  def finite(self):
    n = min(self.B, 4096)
    x, P = self.arena.read(0, n)
    return bool(np.isfinite(x).all() and np.isfinite(P).all())

  def close(self):
    self.arena.close()


def _cpu_limits():
  """(logical CPUs this process may run on, cgroup CPU quota in CPUs or None).  The GPU boxes of this pool run the
  container under a CFS quota (cpu.max) far below the 128 logical CPUs the affinity mask shows; threads beyond the quota
  are throttled, not run (measured: linear to the quota, then flat, then worse -- profiles/r02_cpu_thread_sweep.txt)."""
  try:
    n = len(os.sched_getaffinity(0))
  except AttributeError:
    n = os.cpu_count() or 1
  quota = None
  try:
    with open("/sys/fs/cgroup/cpu.max", encoding="utf-8") as f:       # cgroup v2: "<quota> <period>" or "max <period>"
      q, per = f.read().split()[:2]
      if q != "max":
        quota = float(q) / float(per)
  except (OSError, ValueError):
    try:
      with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", encoding="utf-8") as f:   # cgroup v1
        q = float(f.read())
      with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us", encoding="utf-8") as f:
        per = float(f.read())
      if q > 0:
        quota = q / per
    except (OSError, ValueError):
      pass
  return n, quota


def _threads():
  """host threads the reference arm uses: every CPU it can actually get (affinity mask capped by the cgroup quota)."""
  n, quota = _cpu_limits()
  if quota is not None:
    n = max(1, min(n, int(quota + 0.5)))
  return n


def _cpu_info():
  n, quota = _cpu_limits()
  return {"logical_cpus": n, "cgroup_cpu_quota": quota}


def _best_threads(fname):
  """(threads, pinned?) for the reference arm: the CPUs the container can actually get, verified by a short sweep.  The
  GPU boxes are shared and run the container under a CFS quota: a thread count at the quota can be SLOWER than one
  below it (any other runnable thread of the container pushes the group over its budget and the whole group is
  throttled for the rest of the period), and pinning to fixed CPUs can land on CPUs other tenants keep busy -- so both
  are measured, not assumed."""
  n = _threads()
  cands = []
  for c in sorted({n, max(1, n - 1), max(1, n - 2), max(1, (3 * n) // 4)}, reverse=True):
    cands += [(c, True), (c, False)]
  rates = {}
  for c, pin in cands:
    rates[(c, pin)] = 1.0 / _calibrate(fname, c, n=4096, pin=pin)
  best = max(rates, key=rates.get)
  return best[0], best[1], {f"{c}{'p' if pin else 'u'}": v for (c, pin), v in rates.items()}


def _calibrate(fname, nthreads, n=4096, pin=True):
  """seconds per filter-step with `nthreads` workers (small resident sample, warm)."""
  arm = CpuArm(fname, n * max(1, nthreads // 4), nthreads=nthreads, pin=pin)
  arm.step()
  t = time.perf_counter()
  for _ in range(3):
    arm.step()
  per = (time.perf_counter() - t) / 3 / arm.B
  arm.close()
  return max(per, 1e-10)


def cpu_reference(fname, workload, budget_s=15.0, steps=None, full_batch=None):
  """cpu_baseline of the GPU line: the reference's C path on all host cores over a bounded resident sample of the
  same workload (same kind schedule), plus one-thread and per-filter-Python-driver figures for context."""
  cores, pin, sweep = _best_threads(fname)
  n_steps = steps or 20
  per = _calibrate(fname, cores, pin=pin)
  full = full_batch or WORKLOADS[workload]["batch"]
  Bs = int(max(1024, min(full, budget_s / (per * (n_steps + 2)))))
  arm = CpuArm(fname, Bs, nthreads=cores, pin=pin)
  arm.step(); arm.step()
  t = time.perf_counter()
  for _ in range(n_steps):
    arm.step()
  el = time.perf_counter() - t
  assert arm.finite()
  pinned = arm.arena.pinned
  arm.close()
  n1 = 4096
  one = CpuArm(fname, n1, nthreads=1)
  one.step()
  t1 = time.perf_counter()
  for _ in range(3):
    one.step()
  one_thread = 3 * n1 / (time.perf_counter() - t1)
  py_driver = None
  try:
    from oracle import build_ref
    from rednose_b200.ekf_sym import EKF_sym
    x, P = one.arena.read(0, 1)
    kf = EKF_sym(build_ref.OUT, fname, one.Q, x[0], P[0], one.dim, one.edim, quaternion_idxs=one.quat)   # Python driver on the CPU oracle library
    k = one.sched[1]
    zp, R = one.pools[k]
    tt, n_calls = 0.0, 300
    t2 = time.perf_counter()
    for i in range(n_calls):
      tt += 0.01
      kf.predict_and_update_batch(tt, k, zp[0][i:i + 1], R[i:i + 1])
    py_driver = n_calls / (time.perf_counter() - t2)
  except Exception:  # pylint: disable=broad-except
    pass
  one.close()
  v = Bs * n_steps / el
  return {"value": v, "unit": "steps/s", "cores": cores, "threads": cores, "threads_pinned": pinned, "kind": "port", **_cpu_info(),
          "one_thread_steps_per_s": one_thread, "thread_scaling_efficiency": v / (cores * one_thread), "copy_bytes_per_step": 0,
          "thread_sweep_steps_per_s": sweep, "thread_sweep_key": "<threads>p = pinned (spread over the affinity mask), u = unpinned", "python_driver_per_filter_steps_per_s": py_driver,
          "sample": f"{Bs} {fname} filters resident x {n_steps} in-place steps of workload {workload} (same kind schedule), {el:.1f} s",
          "same_batch_as_gpu_arm": Bs == full, "what": CPU_WHAT}


def _cpu_problem(fname, B, seed=99):
  # the oracle arm must not touch the CUDA libraries: build the same synthetic problem with the oracle's own h_k.
  # P is ONE [EDIM, EDIM] matrix (broadcast by the arena, as the GPU arm broadcasts it on the device); R is per filter.
  rng = np.random.default_rng(seed)
  if fname == "kinematic":
    from rednose_b200.filters.kinematic import KinematicKalman as F
    x = np.tile(F.initial_x, (B, 1)) + rng.normal(size=(B, 2))
    P = np.diag(F.initial_P_diag).astype(np.float64)
    return x, P, F.Q.copy(), {1: (rng.normal(0.0, 0.1, (4, B, 1)), np.tile(np.array([[0.1**2]]), (B, 1, 1)))}, (2, 2), []
  from oracle import build_ref
  from rednose_b200.filters.live import LiveKalman as F
  from oracle.handle import Oracle
  o = Oracle(build_ref.OUT, "live")
  x_true = F.initial_x.copy()
  x_true[3:7] = [0.7, 0.1, -0.5, 0.5]
  x_true[3:7] /= np.linalg.norm(x_true[3:7])
  x = np.tile(x_true, (B, 1))
  x[:, 0:3] += rng.normal(0, 10.0, (B, 3))
  x[:, 7:10] += rng.normal(0, 1.0, (B, 3))
  x[:, 10:13] += rng.normal(0, 0.05, (B, 3))
  x[:, 17:20] += rng.normal(0, 0.3, (B, 3))
  pdiag = np.array([25.0] * 3 + [0.05**2] * 3 + [1.0] * 3 + [0.1**2] * 3 + [0.01**2] * 3 + [0.01**2] + [0.5**2] * 3 + [0.01**2] * 3)
  P = np.diag(pdiag)
  pools = {}
  for k, rdiag in LIVE_R.items():
    hz = np.zeros(3)
    o.leaf(f"h_{k}", np.ascontiguousarray(x_true), np.zeros(1), hz)
    pools[k] = (hz[None, None, :] + rng.normal(size=(2, B, 3)) * np.sqrt(np.array(rdiag)), np.tile(np.diag(rdiag), (B, 1, 1)))
  return x, P, F.Q.copy(), pools, (23, 22), [3]


def run_reference(args):
  """Reference arm: the reference's C path (oracle/_ref) on ALL host cores, same workload / metric / unit as the GPU arm.
  One step = one in-place pass of predict + update_<kind> (the workload's kind schedule) over the resident batch: the
  workload's full batch when warm-up + K steps fit in ~150 s on this box's cores, else the largest sample that does."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  wl = WORKLOADS[args.workload]
  fname, full = wl["filter"], (args.batch or wl["batch"])
  cores, pin, sweep = _best_threads(fname)
  per = _calibrate(fname, cores, pin=pin)
  total_budget = 150.0
  Bs = int(max(cores * 8, min(full, total_budget / (args.steps + args.warmup) / per)))
  arm = CpuArm(fname, Bs, nthreads=cores, pin=pin)
  times = []
  for i in range(args.warmup + args.steps):
    t = time.perf_counter()
    arm.step()
    if i >= args.warmup:
      times.append(time.perf_counter() - t)
  assert arm.finite()
  pinned, resident = arm.arena.pinned, arm.arena.bytes_resident
  arm.close()
  one = CpuArm(fname, 4096, nthreads=1)
  one.step()
  t1 = time.perf_counter()
  for _ in range(3):
    one.step()
  one_thread = 3 * 4096 / (time.perf_counter() - t1)
  one.close()
  v = Bs / float(np.mean(times))
  cb = {"value": v, "unit": "steps/s", "cores": cores, "threads": cores, "threads_pinned": pinned, "kind": "port", **_cpu_info(),
        "one_thread_steps_per_s": one_thread, "thread_scaling_efficiency": v / (cores * one_thread), "copy_bytes_per_step": 0,
        "thread_sweep_steps_per_s": sweep, "thread_sweep_key": "<threads>p = pinned (spread over the affinity mask), u = unpinned", "resident_bytes": resident,
        "sample": f"{Bs} {fname} filters resident ({'the full workload batch' if Bs == full else f'of {full}'}), one in-place pass per step, {args.steps} timed steps, workload {args.workload} kind schedule",
        "what": CPU_WHAT}
  line = {"impl": "reference", "metric": "fused EKF predict+update steps/s (batched, float64)", "value": v, "unit": "steps/s",
          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(times)) * 1e3, "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": {"workload": args.workload, "filter": fname, "filters_per_gpu": Bs, "dim": arm.dim, "edim": arm.edim, "sample_filters": Bs,
                     "same_batch_as_gpu_arm": Bs == full},
          "cpu_baseline": cb,
          "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
  print(json.dumps(line))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=None, help="timed steps (default: the workload's own)")
  ap.add_argument("--warmup", type=int, default=None)
  ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
  ap.add_argument("--workload", default="live_1m", choices=sorted(WORKLOADS))
  ap.add_argument("--batch", type=int, default=0, help="override filters per GPU")
  ap.add_argument("--e2e-steps", type=int, default=20)
  ap.add_argument("--cpu-budget", type=float, default=15.0)
  ap.add_argument("--sustain", type=float, default=2.0, help="seconds of the sustained figure beside the K-step burst (0 = skip)")
  ap.add_argument("--rts-steps", type=int, default=1000, help="live_rts: history length T (BASELINE.json: 10000)")
  ap.add_argument("--rts-segment", type=int, default=50, help="live_rts: steps between checkpoints")
  ap.add_argument("--hbm-budget-gb", type=float, default=140.0, help="live_rts: HBM the smoother may use per GPU")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-extras", dest="extras", action="store_false",
                  help="skip the short measurements of the other kernels (kinematic / history / RTS / ragged / MSCKF, ~1 min)")
  ap.add_argument("--extras", dest="extras", action="store_true", default=True)
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="write what the last timed step returned (all filters, or a fixed seeded sample, under 64 MB) as DIR/<name>.npy")
  args = ap.parse_args()
  wl = WORKLOADS[args.workload]
  if args.dump_outputs and args.impl != "b200":
    # the reference arm sizes its batch from a timing calibration, so its inputs differ from run to run
    ap.error("--dump-outputs writes what this engine computed (--impl b200)")
  if args.steps is None:
    args.steps = wl["steps"]
  if args.warmup is None:
    args.warmup = wl["warmup"]
  if args.impl == "reference":
    args.warmup = max(args.warmup, 3)
    run_reference(args)
  elif args.workload == "live_rts":
    args.warmup = max(args.warmup, 1)
    run_rts(args)
  elif args.workload == "msckf_10k":
    args.warmup = max(args.warmup, 3)
    run_msckf(args)
  else:
    args.warmup = max(args.warmup, 3)
    run_gpu(args)


if __name__ == "__main__":
  main()
