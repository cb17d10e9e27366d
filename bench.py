#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched physics step on humanoid.xml (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--nworld 8192] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1], reference benchmarks/humanoid/__init__.py): humanoid, nworld=8192 per GPU, nconmax=24,
njmax=64, keyframe 0 (squat), Newton / pyramidal / Euler, deterministic Ornstein-Uhlenbeck ctrl noise (cli.py:103-145).
A "step" is one pass of the hot path (ctrl-noise kernel + mjb_step) over all worlds of the rank.  Weak scaling: every rank
owns its own 8192 worlds on its own GPU, no collective inside the step; the timed region is bracketed by barrier +
synchronize, timed with CUDA events, MAX over ranks.

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the roofline / algorithmic-bytes definitions.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from mujoco_warp_b200.scenes import WORKLOADS  # noqa: E402  (paths + sizes only; the package imports torch lazily)


def metric_name(wl):
  return "env-steps/sec (whole box) on humanoid.xml at nworld=8192 per GPU" if wl == "humanoid" else f"env-steps/sec (whole box) on {wl} at nworld={WORKLOADS[wl]['nworld']} per GPU"


def parse():
  p = argparse.ArgumentParser()
  p.add_argument("--gpus", type=int, default=1)
  p.add_argument("--steps", type=int, default=200)
  p.add_argument("--warmup", type=int, default=20)
  p.add_argument("--impl", default="ours", choices=["ours", "reference"])
  p.add_argument("--workload", default="humanoid", choices=sorted(WORKLOADS), help="BASELINE configs[1] (default), [2] g1, [3] convex_mesh stand-in, three_humanoids")
  p.add_argument("--nworld", type=int, default=None, help="worlds per GPU (default: the workload's)")
  p.add_argument("--no-graph", action="store_true", help="launch kernels directly instead of replaying a CUDA graph")
  p.add_argument("--cpu-sample-worlds", type=int, default=None)
  p.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (kernel A/B sweeps)")
  p.add_argument("--dump-outputs", metavar="DIR", default=None,
                 help="after the timed steps, write the Data arrays of the last one as DIR/<name>.npy (a fixed world sample, at most 64 MB)")
  a = p.parse_args()
  if a.steps < 1 or a.warmup < 0:
    p.error("--steps must be >= 1 and --warmup >= 0")
  return a


def usable_cores() -> int:
  """Host cores this process may actually use: min(affinity mask, cgroup cpu quota)."""
  n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
  try:
    quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
    if quota != "max":
      n = min(n, max(1, int(int(quota) / int(period))))
  except Exception:
    pass
  return n


# --------------------------------------------------------------------------------------------- clocks


class ClockSampler:
  """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

  Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

  def __init__(self, gpu_index):
    self.gpu, self.rows, self.proc = gpu_index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.t = threading.Thread(target=self._read, daemon=True)
      self.t.start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([x.strip() for x in line.split(",")])

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
    mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
    reasons = set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      if len(r) >= 9:
        for n, v in zip(names, r[5:9]):
          if v.lower().startswith("active"):
            reasons.add(n)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------- algorithmic bytes


def algorithmic_words(mjm, tabs, ncon_mean, nefc_mean, nv_pad):
  """Per-env-step algorithmic fp32/int32 words per kernel: every Data output written once, every input read once;
  Model constants and workspace count zero (SURVEY.md §8d)."""
  nq, nv, nu, nb, nj, ng = mjm.nq, mjm.nv, mjm.nu, mjm.nbody, mjm.njnt, mjm.ngeom
  ng_dyn = int((np.asarray(mjm.body_weldid)[np.asarray(mjm.geom_bodyid)] != 0).sum())
  nC, nJ, qld = tabs["nC"], tabs["nJmom"], tabs["qld_total"]
  w = {}
  w["position"] = nq + (3 + 4 + 9 + 3 + 9) * nb + 6 * nj + 12 * ng_dyn + 12 * mjm.nsite + 12 * mjm.ncam + 6 * mjm.nlight + (3 + 10) * nb + 6 * nv + 10 * nb + nC + 3 * nu + 2 * nJ
  w["collision"] = 12 * ng + 39 * ncon_mean + 2
  w["constraint"] = nq + nv + 6 * nv + 3 * nb + 39 * ncon_mean + nefc_mean * nv_pad + 8 * nefc_mean + 4 * ncon_mean + 4
  w["velocity"] = nv + 6 * nv + 10 * nb + nu + nC + 2 * nJ + nu + nu + 6 * nb + 6 * nv + 6 * nv + 12 * nb + nu + qld + nv + nv
  w["solver"] = nefc_mean * nv_pad + 3 * nefc_mean + nC + 2 * nv + 3 * nv + 2 * nefc_mean + 1
  w["integrate"] = nq + 2 * nv + nq + 2 * nv + 1
  return w


# --------------------------------------------------------------------------------------------- CPU arm (oracle)


def load_workload(name):
  """Model + initial host state + (optional) control trajectory of a workload."""
  from mujoco_warp_b200._src import io as mio
  from mujoco_warp_b200._src import mjcf
  from mujoco_warp_b200._src.mjcf import MjDataLite, reset_data_keyframe

  wl = WORKLOADS[name]
  mjm = mjcf.load_any(wl["model"])
  mjd = MjDataLite(mjm)
  ctrls = None
  if wl["replay"]:
    ctrls = mio.load_trajectory(wl["replay"], mjm, mjd)
  elif mjm.nkey > 0:
    reset_data_keyframe(mjm, mjd, 0)
  return wl, mjm, mjd, ctrls


def ctrl_noise_np(mjm, ctrl, step, center, noise_std=0.01, noise_rate=0.1):
  """numpy restatement of the harness control noise (reference cli.py:103-145; the GPU arm's k_ctrl_noise): per (world, actuator)
  ctrl <- rate ctrl + (1 - rate) centre + scale halfrange (2 halton((step + 1)(world + 1), actuator + 2) - 1), clipped to ctrlrange."""
  nworld, nu = ctrl.shape
  rate = np.exp(-float(mjm.opt.timestep) / noise_rate)
  scale = noise_std * np.sqrt(1.0 - rate * rate)
  limited = np.asarray(mjm.actuator_ctrllimited).astype(bool)
  lo, hi = np.asarray(mjm.actuator_ctrlrange)[:, 0], np.asarray(mjm.actuator_ctrlrange)[:, 1]
  halfrange = np.where(limited, 0.5 * (hi - lo), 1.0)
  n = np.tile(((step + 1) * (np.arange(nworld, dtype=np.int64) + 1))[:, None], (1, nu))
  base = (np.arange(nu, dtype=np.int64) + 2)[None, :]
  f = 1.0 / base
  h = np.zeros((nworld, nu))
  while (n > 0).any():  # radical inverse, all (world, actuator) pairs at once
    h += f * (n % base)
    n //= base
    f = f / base
  out = rate * ctrl + (1.0 - rate) * center[None, :] + scale * halfrange[None, :] * (2.0 * h - 1.0)
  return np.where(limited[None, :], np.clip(out, lo[None, :], hi[None, :]), out)


def cpu_run(name, nworld, nsteps, nthreads):
  """Times the CPU restatement (oracle, fp64, OpenMP over worlds) on a bounded sample; returns env-steps/s."""
  from tests import util
  from oracle import orc  # noqa: F401  (bench.py's cpu_baseline / --impl reference legs are allowed to use the oracle)

  wl, mjm, mjd, ctrls = load_workload(name)
  o = util.make_oracle(mjm, nworld, wl["nconmax"], wl["njmax"])
  o.set_state(qpos=np.asarray(mjd.qpos), qvel=np.asarray(mjd.qvel), ctrl=np.asarray(mjd.ctrl))
  center = np.asarray(mjd.ctrl, dtype=np.float64)
  o.step(nthreads)
  t0 = time.perf_counter()
  for i in range(nsteps):
    if ctrls is not None:
      o.d["ctrl"][:] = ctrls[i % len(ctrls)]
    elif mjm.nu:  # the same control process as the GPU arm: OU noise around the keyframe controls, Halton sequence (cli.py:103-145)
      o.d["ctrl"][:] = ctrl_noise_np(mjm, o.d["ctrl"], i, center)
    o.step(nthreads)
  dt = time.perf_counter() - t0
  return nworld * nsteps / dt, dt


def run_reference(args):
  """--impl reference: the reference's algorithm on the box's host cores.  The reference itself (Warp + mujoco) cannot be
  installed here (no wheels, no network: DESIGN.md), so this arm times the CPU restatement in oracle/ (kind = "port")."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  wl = WORKLOADS[args.workload]
  nworld = args.nworld or wl["nworld"]
  cores = usable_cores()
  nw = args.cpu_sample_worlds or nworld
  for _ in range(max(1, min(args.warmup, 3))):
    cpu_run(args.workload, nw, 1, cores)
  rate, dt = cpu_run(args.workload, nw, args.steps, cores)
  sample = f"{nw} worlds x {args.steps} steps of the oracle (fp64 C, OpenMP {cores} threads) per run"
  line = {
    "impl": "reference", "metric": metric_name(args.workload), "value": rate, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
    "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
    "config": {"workload": f"{wl['label']}; CPU sample of {nw} worlds per step (bounded sample of nworld={nworld}/GPU), same OU / Halton ctrl noise as the GPU arm" if not wl["replay"] else f"{wl['label']}; CPU sample of {nw} worlds per step"},
    "cpu_baseline": {"value": rate, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
    "e2e": {"value": rate, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    "gpu_launches": 0,
  }
  print(json.dumps(line))


# --------------------------------------------------------------------------------------------- GPU arm

DUMP_BYTES = 60 * 2**20  # array payload; with the .npy headers the dump stays below 64 MB however a megabyte is counted


def dump_outputs(d, out_dir, seed=0):
  """Writes the Data arrays a caller of the step receives as out_dir/<name>.npy: the top-level and efc_* fields of a fixed, seeded
  sample of worlds (all of them when they fit DUMP_BYTES), and the contact_* fields of those worlds' contacts, grouped by world in
  pool order (at most nconmax per sampled world on average).  Float fields stay float32; integer fields are written as float64
  (exact).  worlds.npy lists the sampled world ids.  The sample depends on the sizes only, so two builds dump the same worlds."""
  import torch

  nworld = d.nworld
  per_world = {("efc_" if s is d.efc else "") + k: v for s in (d, d.efc) for k, v in vars(s).items()
               if isinstance(v, torch.Tensor) and v.dim() and v.shape[0] == nworld and v.numel() and not k.startswith("_")}
  nacon = min(int(d.nacon[0]), d.naconmax)
  contact = {"contact_" + k: v[:nacon] for k, v in vars(d.contact).items() if isinstance(v, torch.Tensor) and v.dim() and v.shape[0] == d.naconmax}
  row = lambda v: (4 if v.dtype == torch.float32 else 8) * v[0].numel()  # bytes of one world's / contact's entry as written
  world_bytes = 8 + sum(row(v) for v in per_world.values()) + d.nconmax * sum(row(v) for v in contact.values())
  k = max(1, min(nworld, DUMP_BYTES // world_bytes))
  worlds = np.sort(np.random.default_rng(seed).choice(nworld, k, replace=False)) if k < nworld else np.arange(nworld)
  idx = torch.from_numpy(worlds).to(d.qpos.device)
  out = {"worlds": worlds.astype(np.float64)}
  out.update({n: v.index_select(0, idx) for n, v in per_world.items()})
  wid = d.contact.worldid[:nacon].long()
  keep = torch.nonzero(torch.isin(wid, idx)).squeeze(1)
  keep = keep[torch.argsort(wid[keep], stable=True)][: k * d.nconmax]  # grouped by world, pool order inside a world
  out.update({n: v[keep] for n, v in contact.items()})
  # the efc_id of a contact row is a contact-pool slot, and worlds claim slots in no fixed order: it is written as the contact's
  # index within its world (as listed in contact_*), -1 on rows past nefc
  from mujoco_warp_b200._src import constants as C

  local = torch.full((max(nacon, 1),), -1, dtype=torch.long, device=wid.device)
  local[keep] = torch.arange(len(keep), device=wid.device) - torch.searchsorted(wid[keep], wid[keep])
  efc_id, efc_type = out["efc_id"].long(), out["efc_type"]
  live = torch.arange(efc_id.shape[1], device=efc_id.device)[None, :] < out["nefc"][:, None]
  is_contact = (efc_type >= C.CNSTR_CONTACT_FRICTIONLESS) & (efc_type <= C.CNSTR_CONTACT_ELLIPTIC)
  out["efc_id"] = torch.where(is_contact, torch.where(live, local[efc_id.clamp(0, max(nacon - 1, 0))], -1), efc_id)
  os.makedirs(out_dir, exist_ok=True)
  for n, v in out.items():
    a = v.cpu().numpy() if isinstance(v, torch.Tensor) else v
    np.save(os.path.join(out_dir, n + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def run_ours(args):
  import torch

  torch.set_num_threads(max(1, min(4, usable_cores())))  # host-side tensor ops in the e2e loop stay within the cpu quota
  import mujoco_warp_b200 as mjw
  from mujoco_warp_b200._src import io as mio

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  torch.cuda.set_device(local)
  dist = None
  if world > 1:
    import torch.distributed as dist

    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

  def barrier():
    if dist is not None:
      dist.barrier()
    torch.cuda.synchronize()

  wl, mjm, mjd, ctrls = load_workload(args.workload)
  tabs = mio.derive_tables(mjm)
  m = mjw.put_model(mjm)
  nworld = args.nworld or wl["nworld"]
  NCONMAX, NJMAX = wl["nconmax"], wl["njmax"]
  d = mjw.put_data(mjm, mjd, nworld=nworld, nconmax=NCONMAX, njmax=NJMAX, m=m)
  center = torch.from_numpy(np.asarray(mjd.ctrl, dtype=np.float32)).cuda()
  traj = torch.from_numpy(np.asarray(ctrls, dtype=np.float32)).cuda() if ctrls is not None else None  # (nstep, nu), device resident
  data_mb = sum(t.numel() * t.element_size() for o in (d, d.efc, d.contact) for t in vars(o).values() if isinstance(t, torch.Tensor)) / 2**20
  # timing rule: a per-step working set below the 126 MB L2 is flushed between timed steps (each step then gets its own event pair)
  flush = torch.empty(256 * 2**20 // 4, dtype=torch.float32, device="cuda") if data_mb <= 126 else None
  # ranks use shifted Halton step indices so their noise streams differ
  world_offset = rank * nworld

  stream = torch.cuda.Stream()
  graph = None
  step_idx = [0]
  # every Data array, efc_* rows past nefc and accumulated overflow bits included: restoring all of them makes the Data the timed
  # window starts from (and so every array it leaves) independent of how many untimed steps ran before
  arrays = list({id(t): t for o in (d, d.efc, d.contact) for t in vars(o).values() if isinstance(t, torch.Tensor)}.values())

  def snapshot():
    return [t.clone() for t in arrays]

  def restore(snap):
    for t, v in zip(arrays, snap):
      t.copy_(v)

  initial = snapshot()

  def set_ctrl():
    if traj is not None:  # trajectory replay, zero-order hold (cli.py:154-158): every world gets the step's control row
      d.ctrl.copy_(traj[step_idx[0] % traj.shape[0]].unsqueeze(0).expand(nworld, -1))
    elif mjm.nu:
      mjw.ctrl_noise(m, d, step_idx[0] + world_offset, center)

  def one_step():
    set_ctrl()
    if graph is not None:
      graph.replay()
    else:
      mjw.step(m, d)
    step_idx[0] += 1

  with torch.cuda.stream(stream):
    for _ in range(3):
      one_step()
    stream.synchronize()
    launches_per_step = 1 + mjw.last_launch_count()
    if not args.no_graph:
      g = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g, stream=stream):
        mjw.step(m, d)
      graph = g
    # The simulated state inside the timed window is deterministic: the Data is put back to its put_data state after graph capture,
    # advanced by exactly `warmup` steps, snapshotted, and restored right before the timed region.  nvidia-smi needs a few hundred
    # ms before its first row, so the same load keeps running (on the live state) until it reports; those extra steps are undone
    # by the restore.
    restore(initial)
    step_idx[0] = 0
    sampler = ClockSampler(local)
    if rank == 0:
      sampler.start()
    for _ in range(args.warmup):
      one_step()
    stream.synchronize()
    snap, snap_idx = snapshot(), step_idx[0]
    t_wait = time.perf_counter() + 3.0
    while rank == 0 and sampler.proc is not None and len(sampler.rows) < 1 and time.perf_counter() < t_wait:
      one_step()
      stream.synchronize()
    restore(snap)
    step_idx[0] = snap_idx
    sim_steps_before_timed = snap_idx

    # ---- timed region: K steps, device-resident inputs, CUDA events on the launching stream
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if flush is None:
      e0.record(stream)
      for _ in range(args.steps):
        one_step()
      e1.record(stream)
      stream.synchronize()
      ms = e0.elapsed_time(e1)
    else:
      evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
      for a, b in evs:
        flush.fill_(0.0)
        a.record(stream)
        one_step()
        b.record(stream)
      stream.synchronize()
      ms = sum(a.elapsed_time(b) for a, b in evs)
    barrier()
    if args.dump_outputs and rank == 0:
      dump_outputs(d, args.dump_outputs)
    # ---- statistics of the run (untimed), taken from the last timed step
    ncon_mean = float(d.nacon.cpu()[0]) / nworld
    nefc_mean = float(d.nefc.float().mean().cpu())
    niter_mean = float(d.solver_niter.float().mean().cpu())
    niter_hist = torch.bincount(d.solver_niter.clamp(0, 4).long().cpu(), minlength=5).tolist()  # worlds with 0, 1, 2, 3, >= 4 Newton iterations
    ovf = int((d.overflow != 0).sum().cpu())
    ovf_bits = int(np.bitwise_or.reduce(d.overflow.cpu().numpy().astype(np.int64))) if nworld else 0
    nan_worlds = int(torch.isnan(d.qpos).any(dim=1).sum().cpu())
    n_rows, t_wait = len(sampler.rows), time.perf_counter() + 1.0
    while rank == 0 and sampler.proc is not None and len(sampler.rows) <= n_rows and time.perf_counter() < t_wait:
      one_step()  # same load, untimed, until one more 100 ms sample lands after the timed region
      stream.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    restore(snap)  # the per-kernel pass and the e2e loop below start from the same state as the timed region
    step_idx[0] = snap_idx

    # ---- per-kernel durations (separate pass with event pairs around each kernel)
    nprof = 20
    acc = None
    for _ in range(nprof):
      set_ctrl()
      step_idx[0] += 1
      r = mjw.step_profile(m, d)
      acc = r if acc is None else {k: acc[k] + r[k] for k in r}
    kms = {k: v / nprof for k, v in acc.items()}

    # ---- e2e: same metric through the public API with HOST buffers: every step's controls come from pinned host memory (H2D) and
    # every step's qpos + qvel go back to pinned host memory (D2H), all inside the timed region.  The loop is software-pipelined one
    # step deep, as an asynchronous actor would run it: the two copy engines work on their own streams (upload of step k + 1's
    # controls and download of step k - 1's state overlap the kernels of step k; small device-to-device copies decouple the buffers
    # the step graph reads / writes from the ones in flight), and the host consumes the read-back of step k - 1 (event wait, not a
    # stream sync) to produce the controls of step k + 1.
    nbuf, nq_, nv_ = 2, mjm.nq, mjm.nv
    ctrl_host = [torch.empty((nworld, mjm.nu), dtype=torch.float32).pin_memory() for _ in range(nbuf)]
    state_host = [torch.empty((nworld, nq_ + nv_), dtype=torch.float32).pin_memory() for _ in range(nbuf)]
    ctrl_dev = [torch.empty_like(d.ctrl) for _ in range(nbuf)]
    state_dev = [torch.empty((nworld, nq_ + nv_), dtype=torch.float32, device="cuda") for _ in range(nbuf)]
    h2d_done, ctrl_used, snap_done, d2h_done = ([torch.cuda.Event() for _ in range(nbuf)] for _ in range(4))
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    for c in ctrl_host:
      c.copy_(d.ctrl.cpu())
    e2e_steps = max(10, args.steps // 2)

    def upload(b):
      with torch.cuda.stream(s_in):
        s_in.wait_event(ctrl_used[b])
        ctrl_dev[b].copy_(ctrl_host[b], non_blocking=True)
        h2d_done[b].record(s_in)

    stream.synchronize()
    barrier()
    t0 = time.perf_counter()
    upload(0)
    tr = [0.0] * 5 if os.environ.get('MJB_E2E_TRACE') else None
    for i in range(e2e_steps):
      b = i % nbuf
      ta = time.perf_counter()
      stream.wait_event(h2d_done[b])
      if mjm.nu:
        d.ctrl.copy_(ctrl_dev[b], non_blocking=True)
      ctrl_used[b].record(stream)
      if graph is not None:
        graph.replay()
      else:
        mjw.step(m, d)
      stream.wait_event(d2h_done[b])  # the download that last read state_dev[b] (step i - 2)
      state_dev[b][:, :nq_].copy_(d.qpos, non_blocking=True)
      state_dev[b][:, nq_:].copy_(d.qvel, non_blocking=True)
      snap_done[b].record(stream)
      with torch.cuda.stream(s_out):
        s_out.wait_event(snap_done[b])
        state_host[b].copy_(state_dev[b], non_blocking=True)
        d2h_done[b].record(s_out)
      tb = time.perf_counter()
      p = (i + 1) % nbuf
      if i > 0:  # host-side policy stand-in on the PREVIOUS step's read-back, while this step runs on the GPU
        d2h_done[p].synchronize()
        tc = time.perf_counter()
        ctrl_host[p].add_(0.001 * float(state_host[p][0, 2])).clamp_(-1, 1)
      else:
        tc = tb
      td = time.perf_counter()
      upload(p)  # controls of step i + 1
      if tr is not None:
        te = time.perf_counter()
        for k, v in enumerate((tb - ta, tc - tb, td - tc, te - td)):
          tr[k] += v
    for e in d2h_done:
      e.synchronize()
    if tr is not None:
      print('e2e host us/step: launch %.1f wait %.1f policy %.1f upload %.1f' % tuple(1e6 * v / e2e_steps for v in tr[:4]), file=sys.stderr)
    stream.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()

  from mujoco_warp_b200._src import shard  # the measurement path's only collectives: MAX over ranks of the device-timed durations

  ms_max, e2e_ms_max = shard.reduce_max_elapsed(ms, dist), shard.reduce_max_elapsed(e2e_s * 1e3, dist)
  total_worlds = nworld * world
  value = shard.whole_job_rate(nworld * args.steps, ms_max * 1e-3, world)
  e2e_value = shard.whole_job_rate(nworld * e2e_steps, e2e_ms_max * 1e-3, world)

  if rank == 0:
    peaks = {}
    try:
      peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
      pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    words = algorithmic_words(mjm, tabs, ncon_mean, nefc_mean, m.nv_pad)
    top = max(kms, key=kms.get)
    bytes_launch = 4.0 * words[top] * nworld
    achieved = bytes_launch / (kms[top] * 1e-3) / 1e9
    traffic, issue = None, None
    try:  # DRAM bytes of the same kernel from the committed `ncu --set full` capture (profiles/r02_kernels.md); humanoid only
      if args.workload == "humanoid":
        prof = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        traffic = prof["traffic_bytes"].get("k_" + top)
        traffic = traffic * nworld / 8192.0 if traffic is not None else None
        # second roofline (context; the kernels are issue / latency bound, DESIGN.md section 3): warp instructions of the same capture
        # against the SM's issue rate -- 148 SMs x 4 schedulers x one warp instruction per cycle at the SM clock sampled under load
        winst = prof.get("warp_inst", {}).get("k_" + top)
        mhz = float((clocks or {}).get("sm_mhz") or 0.0)
        if winst and mhz > 0:
          rate = winst * nworld / 8192.0 / (kms[top] * 1e-3)
          issue = {"warp_inst_per_launch": winst * nworld / 8192.0, "achieved_warp_inst_per_s": rate, "peak_warp_inst_per_s": 148 * 4 * mhz * 1e6,
                   "frac": rate / (148 * 4 * mhz * 1e6), "source": "smsp__inst_executed.sum of profiles/r02_kernels.md"}
    except Exception:
      pass
    step_bytes = 4.0 * sum(words.values()) * nworld
    cpu = None
    if world == 1 and not args.no_cpu:  # reported baseline, rank 0 at N = 1 only: a bounded sample of the same workload on the host cores
      cores = usable_cores()
      cpu_steps = 50
      nws = args.cpu_sample_worlds or nworld
      rate, dt = cpu_run(args.workload, nws, cpu_steps, cores)
      cpu = {"value": rate, "unit": "env-steps/s", "cores": cores, "kind": "port",
             "sample": f"{nws} worlds x {cpu_steps} steps of the fp64 C oracle (OpenMP {cores} threads), {dt:.1f} s wall"}
    line = {
      "metric": metric_name(args.workload), "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
      "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": value / 2729192.0 if args.workload == "humanoid" else None,
      "dtype": "f32", "data": "synthetic",
      "config": {
        "workload": wl["label"] if nworld == wl["nworld"] else wl["label"].replace(f"nworld={wl['nworld']}", f"nworld={nworld}"),
        "cuda_graph": graph is not None, "l2": f"per-step Data working set ({data_mb:.0f} MB of Data tensors at {nworld} worlds) exceeds the 126 MB L2; no explicit flush" if data_mb > 126 else f"Data tensors are {data_mb:.0f} MB (< 126 MB L2): 256 MB scratch buffer written between timed steps",
        "vs_baseline_note": "2,729,192 steps/s is the reference's only published number (benchmarks/README.md:48), hardware unstated",
        "sim_steps_before_timed": sim_steps_before_timed, "ncon_mean": ncon_mean, "nefc_mean": nefc_mean, "solver_niter_mean": niter_mean, "solver_niter_hist_0_1_2_3_4plus": niter_hist, "overflow_worlds": ovf, "overflow_bits_or": hex(ovf_bits), "nan_worlds": nan_worlds,
      },
      "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": int(nworld * mjm.nu * 4), "d2h_bytes_per_step": int(nworld * (mjm.nq + mjm.nv) * 4), "steps": e2e_steps,
              "pipeline": "one step deep: host consumes step k-1 while the GPU runs step k; H2D / D2H on their own streams (two pinned buffer sets, event waits)"},
      "gpu_launches": launches_per_step * args.steps,
      "kernel_ms": kms,
      "roofline": {"bound": "hbm", "kernel": "k_" + top, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                   "traffic": traffic, "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                   "algorithmic_bytes_per_launch": bytes_launch, "step_algorithmic_bytes": step_bytes,
                   "step_frac": step_bytes / (ms_max / args.steps * 1e-3) / 1e9 / peak, "issue": issue},
      "cpu_baseline": cpu,
      "clocks": clocks,
    }
    print(json.dumps(line))
  if dist is not None:
    dist.destroy_process_group()


if __name__ == "__main__":
  a = parse()
  if a.impl == "reference":
    run_reference(a)
  else:
    run_ours(a)
