"""CPU tests of the host side: constants, MJCF compiler, derived index tables, C-ABI library symbols, no-CUDA behaviour."""

import ctypes
import os

import numpy as np
import pytest

from tests import util


@pytest.fixture(scope="module")
def mjm(built):
  from mujoco_warp_b200._src import mjcf

  return mjcf.load_any(util.HUMANOID)


def test_constants_self_consistent():
  from mujoco_warp_b200._src import constants as C
  from mujoco_warp_b200._src import types as T

  assert [int(x) for x in T.JointType] == [0, 1, 2, 3]
  assert T.GeomType.PLANE == 0 and T.GeomType.CAPSULE == 3 and T.GeomType.BOX == 6 and T.GeomType.MESH == 7
  assert T.SolverType.NEWTON == 2 and T.ConeType.PYRAMIDAL == 0 and T.IntegratorType.IMPLICITFAST == 3
  assert T.ConstraintType.LIMIT_JOINT == 3 and T.ConstraintType.CONTACT_PYRAMIDAL == 6
  assert T.ConstraintState.QUADRATIC == 1
  bits = list(C.DISABLE_FLAGS.values())
  assert len(set(bits)) == len(bits) and all(b & (b - 1) == 0 for b in bits)
  assert T.OverflowType.ITERATIONS == 1 << 9 and T.OverflowType.LS_ITERATIONS == 1 << 10  # reference types.py:149-176
  try:
    import mujoco
  except ImportError:
    return
  assert C.MJ_MINVAL == mujoco.mjMINVAL and C.MJ_MINIMP == mujoco.mjMINIMP and C.MJ_MINMU == mujoco.mjMINMU
  assert C.DSBL_EULERDAMP == mujoco.mjtDisableBit.mjDSBL_EULERDAMP and C.JNT_HINGE == mujoco.mjtJoint.mjJNT_HINGE


def test_capi_library_exports_every_header_symbol(built):
  from mujoco_warp_b200._src import _lib

  names = _lib.exported_symbols_in_header()
  assert len(names) >= 30
  L = ctypes.CDLL(_lib.LIB_PATH)
  missing = [n for n in names if not hasattr(L, n)]
  assert not missing, missing
  L.mjb_version.restype = ctypes.c_char_p
  assert b"sm_100a" in L.mjb_version()


def test_capi_name_registry_without_gpu(built):
  """Model build-by-name works on the host (no device calls): unknown names and bad batch sizes are rejected."""
  from mujoco_warp_b200._src import _lib

  L = _lib.lib()
  h = L.mjb_model_create()
  assert L.mjb_model_set_int(h, b"nv", 27) == 0
  assert L.mjb_model_set_int(h, b"not_a_field", 1) != 0 and b"unknown" in L.mjb_last_error()
  assert L.mjb_model_set_float(h, b"timestep", 0.005) == 0
  assert L.mjb_model_set_array(h, b"body_pos", 0x1000, 2) != 0  # batched model fields unsupported
  assert L.mjb_model_finalize(h) != 0 and b"not set" in L.mjb_last_error()
  L.mjb_model_destroy(h)


def test_product_path_fails_loudly_without_cuda(mjm):
  import torch

  import mujoco_warp_b200 as mjw

  if torch.cuda.is_available():
    pytest.skip("CUDA present")
  with pytest.raises(RuntimeError, match="CUDA"):
    mjw.put_model(mjm)


def test_product_package_never_imports_oracle():
  import re

  pkg = os.path.join(util.ROOT, "mujoco_warp_b200")
  for dp, _, fs in os.walk(pkg):
    for f in fs:
      if f.endswith((".py", ".cu", ".cuh", ".h")):
        txt = open(os.path.join(dp, f)).read()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), f


def test_mjcf_compiler_matches_fixture(mjm, tmp_path):
  """Compiling the reference's humanoid.xml reproduces the committed .npz fixture exactly."""
  from mujoco_warp_b200._src import mjcf

  a = mjcf.load(os.path.join(util.reference_models(tmp_path), "benchmarks", "humanoid", "humanoid.xml"))
  for k in ("body_mass", "body_inertia", "body_ipos", "body_iquat", "geom_size", "geom_pos", "geom_quat", "jnt_range", "dof_invweight0", "body_invweight0", "key_qpos", "M_colind"):
    np.testing.assert_array_equal(np.asarray(getattr(a, k)), np.asarray(getattr(mjm, k)), err_msg=k)


def test_compiled_humanoid_physical_sanity(mjm):
  assert mjm.body_mass.sum() == pytest.approx(40.84, abs=0.01)  # density-1000 capsule humanoid
  names = mjm.names.body
  for side in ("thigh", "shin", "foot", "upper_arm", "lower_arm", "hand"):
    r, l = names.index(side + "_right"), names.index(side + "_left")
    assert mjm.body_mass[r] == pytest.approx(mjm.body_mass[l], rel=1e-12)
    np.testing.assert_allclose(np.sort(mjm.body_inertia[r]), np.sort(mjm.body_inertia[l]), rtol=1e-9)
  assert (mjm.body_inertia[1:] > 0).all()
  assert mjm.jnt_limited.sum() == 21 and mjm.nkey == 3
  assert mjm.opt.disableflags == 1 << 15 and mjm.opt.timestep == 0.005 and mjm.opt.iterations == 100
  # capsule geom: rbound = radius + half length; plane rbound 0 (collision_driver.py:318-320)
  assert mjm.geom_rbound[0] == 0 and mjm.geom_rbound[1] == pytest.approx(0.07 + 0.07)
  # triangle inequality of principal inertias
  I = np.sort(mjm.body_inertia[1:], axis=1)
  assert (I[:, 0] + I[:, 1] >= I[:, 2] - 1e-12).all()


def test_derived_tables(mjm):
  from mujoco_warp_b200._src import io as mio

  t = mio.derive_tables(mjm)
  # levels partition the bodies, parents sit one level above
  assert sorted(t["level_body"].tolist()) == list(range(mjm.nbody))
  depth = np.zeros(mjm.nbody, int)
  for l in range(t["nlevel"]):
    depth[t["level_body"][t["level_adr"][l] : t["level_adr"][l + 1]]] = l
  assert (depth[1:] == depth[mjm.body_parentid[1:]] + 1).all()
  # child lists invert body_parentid
  for b in range(mjm.nbody):
    kids = t["body_childid"][t["body_childadr"][b] : t["body_childadr"][b + 1]]
    assert sorted(kids.tolist()) == [c for c in range(1, mjm.nbody) if mjm.body_parentid[c] == b]
  # symmetric gather tables reproduce dense M @ v
  rng = np.random.default_rng(0)
  Mcsr = rng.normal(size=t["nC"])
  v = rng.normal(size=mjm.nv)
  M = np.zeros((mjm.nv, mjm.nv))
  for e in range(t["nC"]):
    i, j = t["M_entry_row"][e], mjm.M_colind[e]
    M[i, j] = M[j, i] = Mcsr[e]
  got = np.array([sum(Mcsr[t["mulm_madr"][k]] * v[t["mulm_col"][k]] for k in range(t["mulm_rowadr"][i], t["mulm_rowadr"][i + 1])) for i in range(mjm.nv)])
  np.testing.assert_allclose(got, M @ v, atol=1e-12)
  # NXN pairs: humanoid keeps floor-vs-body and non-adjacent body pairs, excludes parent-child and same-body pairs
  pairs = t["nxn_geom_pair_filtered"]
  assert 0 < len(pairs) <= 190
  b = mjm.geom_bodyid
  assert all(b[p] != b[q] for p, q in pairs)
  assert all(mjm.body_parentid[b[p]] != b[q] and mjm.body_parentid[b[q]] != b[p] or 0 in (b[p], b[q]) for p, q in pairs)
  assert t["nmaxpyramid"] == 4 and t["nJmom"] == mjm.nu and len(t["jnt_limited_slide_hinge_adr"]) == 21
  assert mio.is_sparse(mjm) is False


def test_unsupported_features_raise():
  from mujoco_warp_b200._src import io as mio
  from mujoco_warp_b200._src import mjcf

  # the fully implicit integrator is carried (k_implicit.cu) up to the body count whose derivative scratch fits one block's shared memory
  xml = """<mujoco><option integrator="implicit"/><worldbody><body><joint type="hinge"/><geom size="0.1"/></body></worldbody></mujoco>"""
  mio._validate(mjcf.load_string(xml))
  many = "".join(f'<body pos="{i} 0 0"><joint type="hinge"/><geom size="0.1"/></body>' for i in range(100))
  with pytest.raises(NotImplementedError, match="implicit integrator"):
    mio._validate(mjcf.load_string(f'<mujoco><option integrator="implicit"/><worldbody>{many}</worldbody></mujoco>'))
  # box-box goes through GJK / EPA + multi-contact recovery (16 EPA iterations when it is the only convex pair type);
  # with nativeccd disabled it is a primitive pair.  The convex box path does not support margins (reference io.py:693-717).
  two = '<body pos="0 0 1"><freejoint/><geom type="box" size=".1 .1 .1"{m}/></body><body pos="0 0 2"><freejoint/><geom type="{t}" size=".1 .1 .1"/></body>'
  xml = "<mujoco><worldbody>" + two.format(t="box", m="") + "</worldbody></mujoco>"
  t = mio.derive_tables(mjcf.load_string(xml))
  assert t["has_convex_pair"] == 1 and t["epa_iterations"] == 16
  t = mio.derive_tables(mjcf.load_string(xml.replace("<worldbody>", '<option><flag nativeccd="disable"/></option><worldbody>')))
  assert t["has_convex_pair"] == 0
  with pytest.raises(NotImplementedError, match="margin"):
    mio.derive_tables(mjcf.load_string("<mujoco><worldbody>" + two.format(t="box", m=' margin="0.01"') + "</worldbody></mujoco>"))
  # cylinder-box goes through the GJK / EPA pass
  xml = "<mujoco><worldbody>" + two.format(t="cylinder", m="") + "</worldbody></mujoco>"
  t = mio.derive_tables(mjcf.load_string(xml))
  assert t["has_convex_pair"] == 1 and t["epa_iterations"] == 35
  # mesh geoms go through the convex pass of the mesh build of the collision kernel (k_collision_mesh.cu); height fields are refused
  from tests import util

  t = mio.derive_tables(mjcf.load_string(util.mesh_xml()))
  assert t["has_convex_pair"] == 1 and t["epa_iterations"] == 35


def test_shard_worlds():
  from mujoco_warp_b200._src import shard

  for total, ws in ((65536, 8), (10, 3), (7, 8)):
    blocks = [shard.shard_worlds(total, ws, r) for r in range(ws)]
    assert sum(c for _, c in blocks) == total
    assert all(blocks[r][0] + blocks[r][1] == blocks[r + 1][0] for r in range(ws - 1))
    assert max(c for _, c in blocks) - min(c for _, c in blocks) <= 1
  assert shard.whole_job_rate(8192 * 100, 0.5, world_size=8) == 8 * 8192 * 100 / 0.5


def test_put_model_and_make_data_host_path(monkeypatch):
  """The Python side of put_model / make_data (table derivation, field specs, C-ABI registration order) runs for every fixture
  model against a stub of the C library: no device, no compute -- it catches host-logic slips the GPU tests would only show later."""
  import torch

  from mujoco_warp_b200._src import _lib
  from mujoco_warp_b200._src import io as mio
  from mujoco_warp_b200._src import mjcf

  calls = []

  class Stub:
    def __getattr__(self, name):
      def f(*a, **k):
        calls.append(name)
        return 1 if name in ("mjb_model_create", "mjb_data_create") else 0

      return f

  monkeypatch.setattr(mio, "_require_cuda", lambda: torch.device("cpu"))
  monkeypatch.setattr(_lib, "lib", lambda: Stub())
  scenes = {
    "humanoid": mjcf.load_any(util.HUMANOID), "g1": mjcf.load_any(util.G1), "three_humanoids": mjcf.load_any(util.THREE_HUMANOIDS),
    "sensors": mjcf.load_string(util.sensor_xml()), "equality": mjcf.load_string(util.EQUALITY_XML), "boxccd": mjcf.load_string(util.boxccd_xml()),
  }
  for name, mjm in scenes.items():
    m = mio.put_model(mjm)
    d = mio.make_data(mjm, nworld=3, nconmax=32, njmax=128, m=m)
    assert d.sensordata.shape == (3, getattr(mjm, "nsensordata", 0) if getattr(mjm, "nsensor", 0) else 0), name
    assert d.qpos.shape == (3, mjm.nq) and d.efc.J.shape[0] == 3, name
  assert "mjb_model_finalize" in calls and "mjb_data_finalize" in calls
  bad = mjcf.load_string(util.sensor_xml().replace('<clock name="clk"/>', '<rangefinder name="rf" site="imu"/>'))
  with pytest.raises(NotImplementedError, match="rangefinder"):
    mio.put_model(bad)


def test_d_structure_of_the_compiled_model():
  """MjModel's D-structure as the MJCF compiler writes it (types.py:1343-1347): symmetric tree sparsity, ascending columns, the diagonal
  index, mapM2D onto the lower-triangular M -- and the same rows as the symmetric gather tables put_model derives for mul_m."""
  from mujoco_warp_b200._src import io as mio
  from mujoco_warp_b200._src import mjcf

  for path in (util.HUMANOID, util.G1, util.THREE_HUMANOIDS):
    mjm = mjcf.load_any(path)
    nv = mjm.nv
    assert mjm.nD == 2 * mjm.nC - nv == int(mjm.D_rownnz.sum())
    pat = np.zeros((nv, nv), dtype=bool)
    for i in range(nv):
      cols = mjm.D_colind[mjm.D_rowadr[i] : mjm.D_rowadr[i] + mjm.D_rownnz[i]]
      assert (np.diff(cols) > 0).all() and cols[mjm.D_diag[i]] == i
      pat[i, cols] = True
      for k, j in enumerate(cols):
        e = mjm.mapM2D[mjm.D_rowadr[i] + k]
        r = int(np.searchsorted(mjm.M_rowadr, e, side="right") - 1)
        assert (r, int(mjm.M_colind[e])) == (max(i, j), min(i, j))
    assert (pat == pat.T).all()
    # coupled <=> one dof is an ancestor of the other
    anc = np.zeros((nv, nv), dtype=bool)
    for i in range(nv):
      d = i
      while d >= 0:
        anc[i, d] = True
        d = mjm.dof_parentid[d]
    assert (pat == (anc | anc.T)).all()
    t = mio.derive_tables(mjm)
    np.testing.assert_array_equal(t["mulm_col"], mjm.D_colind)
    np.testing.assert_array_equal(t["mulm_madr"], mjm.mapM2D)
    np.testing.assert_array_equal(t["mulm_rowadr"][:-1], mjm.D_rowadr)
