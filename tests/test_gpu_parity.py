"""GPU parity: CUDA path (through the C-ABI) vs the CPU oracle on identical seeded inputs.

Tolerances follow the reference's own tests: smooth/forward atol=rtol=5e-4 (smooth_test.py:32-38), constraint 5e-4
(constraint_test.py:32), solver qacc/force within 0.1 absolute on O(100) magnitudes (solver_test.py:34-38) -- we hold the
solver to a tighter 5e-3 relative-to-scale bound.  Integer outputs (counts, contact geoms, row types/ids) are exact.
"""

import numpy as np
import pytest
import torch

from tests import util

pytestmark = pytest.mark.gpu

NWORLD, NCONMAX, NJMAX = 32, 24, 64


@pytest.fixture(scope="module")
def scene(built):
  import mujoco_warp_b200 as mjw

  mjm = mjw.mjcf.load_any(util.HUMANOID)
  m = mjw.put_model(mjm)
  return mjw, mjm, m


def _setup(scene, nworld=NWORLD, seed=42):
  mjw, mjm, m = scene
  d = mjw.make_data(mjm, nworld=nworld, nconmax=NCONMAX, njmax=NJMAX, m=m)
  o = util.make_oracle(mjm, nworld, NCONMAX, NJMAX)
  qpos, qvel, ctrl, warm = util.seeded_state(mjm, nworld, seed=seed)
  f32 = lambda a: a.astype(np.float32)
  for name, val in (("qpos", qpos), ("qvel", qvel), ("ctrl", ctrl), ("qacc_warmstart", warm)):
    getattr(d, name).copy_(torch.from_numpy(f32(val)))
  # oracle gets the same fp32-rounded inputs
  o.set_state(qpos=f32(qpos), qvel=f32(qvel), ctrl=f32(ctrl), qacc_warmstart=f32(warm))
  return d, o


def _compare_forward(scene, d, o, solver_tol=5e-3):
  mjw, mjm, m = scene
  torch.cuda.synchronize()
  od = o.d
  for name in util.SMOOTH_FIELDS:
    got = getattr(d, name).cpu().numpy()
    util.assert_close(name, got.reshape(od[name].shape), od[name], atol=5e-4, rtol=5e-4)
  # counts: exact
  for name in ("ne", "nf", "nl", "nefc"):
    np.testing.assert_array_equal(getattr(d, name).cpu().numpy(), od[name], err_msg=name)
  nacon = int(d.nacon.cpu()[0])
  assert nacon == int(od["ncon"].sum())
  assert int(d.ncollision.cpu()[0]) == int(od["ncollision"].sum())
  J = util.dense_J(d)
  for w in range(d.nworld):
    ids = util.world_contacts(d, w)
    n = int(od["ncon"][w])
    assert len(ids) == n, f"world {w}: {len(ids)} contacts vs {n}"
    if n:
      assert (np.diff(ids) == 1).all(), "a world's contacts must be contiguous in the pool"
      c = d.contact
      np.testing.assert_array_equal(c.geom[ids].cpu().numpy(), od["con_geom"][w, :n])
      np.testing.assert_array_equal(c.dim[ids].cpu().numpy(), od["con_dim"][w, :n])
      np.testing.assert_array_equal(c.geomcollisionid[ids].cpu().numpy(), od["con_geomcollisionid"][w, :n])
      for f, of in (("dist", "con_dist"), ("pos", "con_pos"), ("frame", "con_frame"), ("includemargin", "con_includemargin"), ("friction", "con_friction"),
                    ("solref", "con_solref"), ("solreffriction", "con_solreffriction"), ("solimp", "con_solimp")):
        util.assert_close(f"contact.{f}[w{w}]", getattr(c, f)[ids].cpu().numpy(), od[of][w, :n], atol=5e-4, rtol=5e-4)
      adr = c.efc_address[ids].cpu().numpy()
      np.testing.assert_array_equal(adr, od["con_efc_address"][w, :n])
    ne = int(od["nefc"][w])
    np.testing.assert_array_equal(d.efc.type[w, :ne].cpu().numpy(), od["efc_type"][w, :ne])
    eid = d.efc.id[w, :ne].cpu().numpy().copy()
    is_con = od["efc_type"][w, :ne] >= 5
    if n:
      eid[is_con] -= ids[0]
    np.testing.assert_array_equal(eid, od["efc_id"][w, :ne])
    util.assert_close(f"efc.J[w{w}]", J[w, :ne, : mjm.nv], od["efc_J"][w, :ne], atol=5e-4, rtol=5e-4)
    for f in ("pos", "margin", "vel", "frictionloss"):
      util.assert_close(f"efc.{f}[w{w}]", getattr(d.efc, f)[w, :ne].cpu().numpy(), od["efc_" + f][w, :ne], atol=5e-4, rtol=5e-4)
    util.assert_close(f"efc.D[w{w}]", d.efc.D[w, :ne].cpu().numpy(), od["efc_D"][w, :ne], atol=1e-3, rtol=1e-3)
    util.assert_close(f"efc.aref[w{w}]", d.efc.aref[w, :ne].cpu().numpy(), od["efc_aref"][w, :ne], atol=1e-3, rtol=1e-3)
  # solver
  scale = max(1.0, float(np.abs(od["qacc"]).max()))
  util.assert_close("qacc", d.qacc.cpu().numpy(), od["qacc"], atol=solver_tol * scale, rtol=0)
  fscale = max(1.0, float(np.abs(od["efc_force"]).max()))
  for w in range(d.nworld):
    ne = int(od["nefc"][w])
    util.assert_close(f"efc.force[w{w}]", d.efc.force[w, :ne].cpu().numpy(), od["efc_force"][w, :ne], atol=solver_tol * fscale, rtol=0)
  util.assert_close("qfrc_constraint", d.qfrc_constraint.cpu().numpy(), od["qfrc_constraint"], atol=solver_tol * fscale, rtol=0)
  assert (d.overflow.cpu().numpy() == 0).all()
  assert (od["overflow"] == 0).all()


def test_forward_matches_oracle(scene):
  mjw, mjm, m = scene
  d, o = _setup(scene)
  mjw.forward(m, d)
  o.forward()
  _compare_forward(scene, d, o)
  np.testing.assert_array_equal(d.solver_niter.cpu().numpy() > 0, o.d["solver_niter"] > 0)


def test_step_rollout_matches_oracle(scene):
  """20 steps from the squat keyframe + noise: state stays within tolerance and contact/efc counts stay identical."""
  mjw, mjm, m = scene
  d, o = _setup(scene, seed=7)
  for i in range(20):
    mjw.step(m, d)
    o.step()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(d.nefc.cpu().numpy(), o.d["nefc"], err_msg=f"nefc at step {i}")
    util.assert_close(f"qpos@{i}", d.qpos.cpu().numpy(), o.d["qpos"], atol=1e-3, rtol=1e-3)
    util.assert_close(f"qvel@{i}", d.qvel.cpu().numpy(), o.d["qvel"], atol=2e-2, rtol=1e-2)
  util.assert_close("time", d.time.cpu().numpy(), o.d["time"], atol=1e-6, rtol=1e-6)
  assert (d.overflow.cpu().numpy() == 0).all()


def test_stagewise_matches_fused(scene):
  """Calling the stages one by one (public stage API) gives the same Data as the fused forward()."""
  mjw, mjm, m = scene
  d1, _ = _setup(scene, seed=3)
  d2, _ = _setup(scene, seed=3)
  mjw.forward(m, d1)
  for fn in (mjw.kinematics, mjw.com_pos, mjw.camlight, mjw.crb, mjw.collision, mjw.make_constraint, mjw.transmission,
             mjw.fwd_velocity, mjw.fwd_actuation, mjw.fwd_acceleration, mjw.solve):
    fn(m, d2)
  torch.cuda.synchronize()
  for name in util.SMOOTH_FIELDS + ["qacc", "qfrc_constraint"]:
    np.testing.assert_array_equal(getattr(d1, name).cpu().numpy(), getattr(d2, name).cpu().numpy(), err_msg=name)
  np.testing.assert_array_equal(d1.nefc.cpu().numpy(), d2.nefc.cpu().numpy())


def test_determinism(scene):
  """Two runs from the same state are bit-identical per world (ordered reductions; no float atomics)."""
  mjw, mjm, m = scene
  outs = []
  for _ in range(2):
    d, _ = _setup(scene, seed=11)
    for _ in range(5):
      mjw.step(m, d)
    torch.cuda.synchronize()
    outs.append((d.qpos.cpu().numpy().copy(), d.qvel.cpu().numpy().copy(), d.efc.force.cpu().numpy().copy()))
  for a, b in zip(outs[0], outs[1]):
    np.testing.assert_array_equal(a, b)


# --------------------------------------------------------------------------------------------- unitree G1 (BASELINE configs[2])


def test_g1_replay_matches_oracle(built):
  """unitree_g1 scene_flat: nv=35 (dense J in this version), implicitfast, position actuators, replayed shuffle_dance ctrl.
  100 steps from the trajectory's first frame; per-step contact/constraint counts identical, state within tolerance."""
  import mujoco_warp_b200 as mjw
  from mujoco_warp_b200._src.mjcf import MjDataLite

  mjm = mjw.mjcf.load_any(util.G1)
  mjd = MjDataLite(mjm)
  ctrls = mjw.load_trajectory(util.G1_TRAJ, mjm, mjd)
  nworld, nconmax, njmax = 8, 48, 192
  m = mjw.put_model(mjm)
  d = mjw.put_data(mjm, mjd, nworld=nworld, nconmax=nconmax, njmax=njmax, m=m)
  o = util.make_oracle(mjm, nworld, nconmax, njmax)
  o.set_state(qpos=mjd.qpos.astype(np.float32), qvel=mjd.qvel.astype(np.float32))
  rng = np.random.default_rng(5)
  jitter = (0.02 * rng.uniform(-1, 1, (nworld, mjm.nu))).astype(np.float32)
  jitter[0] = 0
  mismatched = 0
  for i in range(100):
    c = (ctrls[i][None, :] + jitter).astype(np.float32)
    d.ctrl.copy_(torch.from_numpy(c))
    o.d["ctrl"][:] = c
    mjw.step(m, d)
    o.step()
    torch.cuda.synchronize()
    mismatched += int((d.nefc.cpu().numpy() != o.d["nefc"]).sum())
    util.assert_close(f"g1 qpos@{i}", d.qpos.cpu().numpy(), o.d["qpos"], atol=2e-3, rtol=2e-3)
  util.assert_close("g1 qvel", d.qvel.cpu().numpy(), o.d["qvel"], atol=5e-2, rtol=2e-2)
  # contact make/break decisions happen at |dist - margin| ~ 1e-7 boundaries; allow a handful of one-step disagreements
  assert mismatched <= 8, mismatched
  assert not (d.overflow.cpu().numpy() & ~int(mjw.OverflowType.LS_ITERATIONS)).any()


# --------------------------------------------------------------------------------------------- mixed-feature scene


@pytest.fixture(scope="module", params=["pyramidal", "elliptic"])
def mixed(built, request):
  import mujoco_warp_b200 as mjw

  xml = util.MIXED_XML
  if request.param == "elliptic":  # elliptic cones + impratio != 1 + a friction-specific solref on every contact
    xml = xml.replace('<option timestep="0.004"', '<option cone="elliptic" impratio="2" timestep="0.004"')
    assert "elliptic" in xml
  mjm = mjw.mjcf.load_string(xml)
  return mjw, mjm, mjw.put_model(mjm)


@pytest.fixture(scope="module")
def scene_elliptic(built):
  import mujoco_warp_b200 as mjw
  from mujoco_warp_b200._src import constants as C

  mjm = mjw.mjcf.load_any(util.HUMANOID)
  mjm.opt.cone = C.CONE_ELLIPTIC
  return mjw, mjm, mjw.put_model(mjm)


def test_elliptic_humanoid_forward_and_rollout(scene_elliptic):
  """Elliptic friction cones on the benchmark scene (nv <= 32 register path): row layout (condim rows per contact, type
  CONTACT_ELLIPTIC), cone-zone forces/states and the Newton solution match the oracle; then a 20-step rollout."""
  mjw, mjm, m = scene_elliptic
  d, o = _setup(scene_elliptic, seed=11)
  mjw.forward(m, d)
  o.forward()
  _compare_forward(scene_elliptic, d, o)
  od = o.d
  assert (od["efc_type"] == 7).any() and (od["efc_state"] == 4).any(), "scene must exercise the CONE zone"
  st = d.efc.state.cpu().numpy()
  agree = total = 0
  for w in range(d.nworld):
    ne = int(od["nefc"][w])
    agree += int((st[w, :ne] == od["efc_state"][w, :ne]).sum()); total += ne
  assert agree >= 0.98 * total, (agree, total)  # zone boundaries can flip on fp32 rounding
  for i in range(20):
    mjw.step(m, d)
    o.step()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(d.nefc.cpu().numpy(), od["nefc"], err_msg=f"nefc at step {i}")
    util.assert_close(f"qpos@{i}", d.qpos.cpu().numpy(), od["qpos"], atol=1e-3, rtol=1e-3)
    util.assert_close(f"qvel@{i}", d.qvel.cpu().numpy(), od["qvel"], atol=2e-2, rtol=1e-2)
  assert (d.overflow.cpu().numpy() == 0).all()


def test_mixed_scene_forward_and_rollout(mixed):
  """Own scene covering the remaining code paths: slide / ball joints, several trees, dof friction-loss rows, joint limits on a
  slide joint, implicit Euler damping (eulerdamp on), position / velocity / motor actuators with force and joint-force
  clamps, sphere-sphere, sphere-capsule, capsule-capsule (incl. the parallel two-contact case), plane-sphere contacts,
  condim 1 / 3 / 4 / 6 pyramids, geom priority / solmix / margin / gap mixing, applied wrenches and joint forces."""
  mjw, mjm, m = mixed
  assert mjm.ntree == 7 and mjm.nv == 41 and (mjm.dof_frictionloss > 0).sum() == 2
  nworld, nconmax, njmax = 16, 32, 128
  d = mjw.make_data(mjm, nworld=nworld, nconmax=nconmax, njmax=njmax, m=m)
  o = util.make_oracle(mjm, nworld, nconmax, njmax)
  # every world is perturbed: at the exact keyframe two capsule pairs are perfectly parallel, where the reference's
  # `abs(det) >= MJ_MINVAL` branch (collision_primitive_core.py:158) is decided by fp32/FMA rounding noise
  qpos, qvel, ctrl, warm = util.seeded_state(mjm, nworld, key=0, seed=9, qpos_noise=0.01, qvel_noise=0.3, ctrl_noise=1.5, exact_world0=False)
  rng = np.random.default_rng(2)
  xfrc = np.zeros((nworld, mjm.nbody, 6), dtype=np.float32)
  xfrc[1::2, 1] = rng.uniform(-1, 1, (nworld // 2, 6))  # wrench on ball0 in every second world
  xfrc[:, 9, :3] = rng.uniform(-0.5, 0.5, (nworld, 3))  # force on the pendulum
  qapp = (0.2 * rng.uniform(-1, 1, (nworld, mjm.nv))).astype(np.float32)
  f32 = lambda a: a.astype(np.float32)
  for name, val in (("qpos", qpos), ("qvel", qvel), ("ctrl", ctrl), ("qacc_warmstart", warm), ("xfrc_applied", xfrc), ("qfrc_applied", qapp)):
    getattr(d, name).copy_(torch.from_numpy(f32(val)).reshape(getattr(d, name).shape))
  o.set_state(qpos=f32(qpos), qvel=f32(qvel), ctrl=f32(ctrl), qacc_warmstart=f32(warm))
  o.d["xfrc_applied"][:] = xfrc
  o.d["qfrc_applied"][:] = qapp
  mjw.forward(m, d)
  o.forward()
  torch.cuda.synchronize()
  od = o.d
  assert od["nf"].min() == 2 and od["ncon"].max() >= 5 and (od["con_dim"][0, : od["ncon"][0]] == 6).any()
  for name in util.SMOOTH_FIELDS + ["site_xpos", "site_xmat"]:
    util.assert_close(name, getattr(d, name).cpu().numpy().reshape(od[name].shape), od[name], atol=5e-4, rtol=5e-4)
  for name in ("ne", "nf", "nl", "nefc"):
    np.testing.assert_array_equal(getattr(d, name).cpu().numpy(), od[name], err_msg=name)
  J = util.dense_J(d)
  for w in range(nworld):
    ids = util.world_contacts(d, w)
    n = int(od["ncon"][w])
    assert len(ids) == n
    np.testing.assert_array_equal(d.contact.geom[ids].cpu().numpy(), od["con_geom"][w, :n])
    np.testing.assert_array_equal(d.contact.dim[ids].cpu().numpy(), od["con_dim"][w, :n])
    for f, of in (("dist", "con_dist"), ("pos", "con_pos"), ("frame", "con_frame"), ("friction", "con_friction"), ("solref", "con_solref"), ("solimp", "con_solimp"), ("includemargin", "con_includemargin")):
      util.assert_close(f"contact.{f}[w{w}]", getattr(d.contact, f)[ids].cpu().numpy(), od[of][w, :n], atol=5e-4, rtol=5e-4)
    ne = int(od["nefc"][w])
    np.testing.assert_array_equal(d.efc.type[w, :ne].cpu().numpy(), od["efc_type"][w, :ne])
    util.assert_close(f"efc.J[w{w}]", J[w, :ne, : mjm.nv], od["efc_J"][w, :ne], atol=5e-4, rtol=5e-4)
    for f in ("pos", "margin", "vel", "frictionloss"):
      util.assert_close(f"efc.{f}[w{w}]", getattr(d.efc, f)[w, :ne].cpu().numpy(), od["efc_" + f][w, :ne], atol=5e-4, rtol=5e-4)
    util.assert_close(f"efc.D[w{w}]", d.efc.D[w, :ne].cpu().numpy(), od["efc_D"][w, :ne], atol=1e-3, rtol=2e-3)
    util.assert_close(f"efc.aref[w{w}]", d.efc.aref[w, :ne].cpu().numpy(), od["efc_aref"][w, :ne], atol=2e-3, rtol=2e-3)
  scale = max(1.0, float(np.abs(od["qacc"]).max()))
  util.assert_close("qacc", d.qacc.cpu().numpy(), od["qacc"], atol=1e-2 * scale, rtol=0)
  # rollout with implicit joint damping in the Euler step
  mismatched = 0
  for i in range(30):
    mjw.step(m, d)
    o.step()
    torch.cuda.synchronize()
    mismatched += int((d.nefc.cpu().numpy() != od["nefc"]).sum())
    util.assert_close(f"qpos@{i}", d.qpos.cpu().numpy(), od["qpos"], atol=3e-3, rtol=3e-3)
  assert mismatched <= 10, mismatched


def test_more_than_32_contacts_in_one_world(built):
  """The contact-row builder of k_constraint works in batches of 32 contacts (phase A: lane = contact, phase C: lane = row of the batch):
  a rigid rake of 40 spheres on a plane gives 40 contacts per world with 1, 4 and 6 rows per contact (contact dimensions 1, 3, 4), i.e. a
  second batch, the generic row path next to the condim-3 fast path, and a row map with mixed row counts.  The fp64 oracle reproduces the
  reference on every fixture; here it is the checker for a case no reference-generated fixture covers (none has more than 28 contacts in a
  world)."""
  import mujoco_warp_b200 as mjw

  mjm = mjw.mjcf.load_string(util.rake_xml())
  m = mjw.put_model(mjm)
  nworld, nconmax, njmax = 8, 64, 256
  d = mjw.make_data(mjm, nworld=nworld, nconmax=nconmax, njmax=njmax, m=m)
  o = util.make_oracle(mjm, nworld, nconmax, njmax)
  qpos, qvel, ctrl, warm = util.seeded_state(mjm, nworld, seed=3, qpos_noise=0.0005, qvel_noise=0.05)
  f32 = lambda a: a.astype(np.float32)
  for name, val in (("qpos", qpos), ("qvel", qvel), ("qacc_warmstart", warm)):
    getattr(d, name).copy_(torch.from_numpy(f32(val)))
  o.set_state(qpos=f32(qpos), qvel=f32(qvel), qacc_warmstart=f32(warm))
  mjw.forward(m, d)
  o.forward()
  assert int(o.d["ncon"].max()) > 32 and set(np.unique(o.d["con_dim"][0, : o.d["ncon"][0]]).tolist()) == {1, 3, 4}
  _compare_forward((mjw, mjm, m), d, o, solver_tol=2e-2)  # 144 coupled rows on one 6-dof body: a stiffer system than the humanoid's
