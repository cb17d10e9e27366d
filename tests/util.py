"""Shared helpers for parity tests: scene setup, seeded states, oracle/CUDA field comparison."""

import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from mujoco_warp_b200.scenes import DATA as SCENES, G1, G1_TRAJ, HUMANOID, THREE_HUMANOIDS  # noqa: E402,F401

REFERENCE_MODELS = os.path.join(ROOT, "tests", "golden", "reference_models.tar.xz")


def reference_models(dest):
  """Unpacks the reference's MJCF model files (tools/make_reference_models.py) under `dest`, keeping their relative layout so that
  <include> and mesh paths resolve; returns `dest`."""
  import tarfile

  with tarfile.open(REFERENCE_MODELS) as tar:
    tar.extractall(dest, filter="data")
  return str(dest)


def seeded_state(mjm, nworld, key=0, seed=42, qpos_noise=0.05, qvel_noise=0.5, ctrl_noise=0.5, exact_world0=True):
  """Per-world states around a keyframe, like the reference fixture's seeded uniform noise (test_data/__init__.py:82-98)."""
  from mujoco_warp_b200._src import constants as C

  rng = np.random.default_rng(seed)
  qpos = np.tile(mjm.key_qpos[key] if key is not None and mjm.nkey > key else mjm.qpos0, (nworld, 1)).astype(np.float64)
  qpos += qpos_noise * rng.uniform(-1, 1, qpos.shape)
  if exact_world0:  # world 0 stays exactly at the keyframe
    qpos[0] = mjm.key_qpos[key] if key is not None and mjm.nkey > key else mjm.qpos0
  for j in range(mjm.njnt):
    qa = mjm.jnt_qposadr[j]
    if mjm.jnt_type[j] == C.JNT_FREE:
      qpos[:, qa + 3 : qa + 7] /= np.linalg.norm(qpos[:, qa + 3 : qa + 7], axis=1, keepdims=True)
    elif mjm.jnt_type[j] == C.JNT_BALL:
      qpos[:, qa : qa + 4] /= np.linalg.norm(qpos[:, qa : qa + 4], axis=1, keepdims=True)
  qvel = qvel_noise * rng.uniform(-1, 1, (nworld, mjm.nv))
  if exact_world0:
    qvel[0] = 0
  ctrl = ctrl_noise * rng.uniform(-1, 1, (nworld, mjm.nu))
  warm = rng.uniform(-1, 1, (nworld, mjm.nv))
  return qpos, qvel, ctrl, warm


def seeded_act(mjm, nworld, seed=4321, scale=0.4):
  """Per-world activations of a model with stateful actuators (na > 0), fp32-representable."""
  rng = np.random.default_rng(seed)
  return (scale * rng.uniform(-1, 1, (nworld, int(getattr(mjm, "na", 0))))).astype(np.float32).astype(np.float64)


def make_oracle(mjm, nworld, nconmax, njmax, dtype=np.float64, clamp_tolerance=True):
  from mujoco_warp_b200._src import mjcf
  from oracle import orc

  kin = mjcf.kinematics_np(mjm, mjm.qpos0)
  return orc.Oracle(mjm, nworld=nworld, nconmax=nconmax, njmax=njmax, dtype=dtype, static_kin=kin, clamp_tolerance=clamp_tolerance)


def dense_J(d):
  """Constraint Jacobian as dense (nworld, njmax, nv_pad) rows: Data.efc.J itself, or -- for models the reference treats as sparse --
  the CSR arrays (J_rownnz / J_rowadr / J_colind / J, reference types.py:2021-2072) expanded row by row."""
  if not hasattr(d.efc, "J_dense"):
    return d.efc.J.cpu().numpy()
  J, nnz, adr, col = d.efc.J.cpu().numpy()[:, 0], d.efc.J_rownnz.cpu().numpy(), d.efc.J_rowadr.cpu().numpy(), d.efc.J_colind.cpu().numpy()[:, 0]
  nefc = np.minimum(d.nefc.cpu().numpy(), d.njmax)
  out = np.zeros_like(d.efc.J_dense.cpu().numpy())
  for w in range(d.nworld):
    for r in range(int(nefc[w])):
      k = np.arange(adr[w, r], adr[w, r] + nnz[w, r])
      out[w, r, col[w, k]] = J[w, k]
  return out


def world_contacts(d, w):
  """Indices of world w's contacts in the global pool, in pool order."""
  nacon = int(d.nacon.cpu()[0])
  wid = d.contact.worldid[:nacon].cpu().numpy()
  return np.nonzero(wid == w)[0]


SMOOTH_FIELDS = [
  "xpos", "xquat", "xmat", "xipos", "ximat", "xanchor", "xaxis", "geom_xpos", "geom_xmat", "cam_xpos", "cam_xmat", "light_xpos", "light_xdir",
  "subtree_com", "cdof", "cinert", "crb", "M", "actuator_length", "actuator_moment", "actuator_velocity", "cvel", "cdof_dot", "qfrc_bias",
  "qfrc_spring", "qfrc_damper", "qfrc_passive", "actuator_force", "qfrc_actuator", "qfrc_smooth", "qacc_smooth", "cacc", "cfrc_int", "qLD",
]


def assert_close(name, a, b, atol, rtol):
  a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
  assert a.shape == b.shape, f"{name}: shape {a.shape} vs {b.shape}"
  err = np.abs(a - b)
  tol = atol + rtol * np.abs(b)
  if not (err <= tol).all():
    i = np.unravel_index(np.argmax(err - tol), err.shape)
    raise AssertionError(f"{name}: max violation at {i}: got {a[i]:.8g}, want {b[i]:.8g} (|err|={err[i]:.3g}, tol={tol[i]:.3g})")


MIXED_XML = """
<mujoco model="mixed">
  <option timestep="0.004" iterations="50" ls_iterations="30"/>
  <default>
    <geom friction="0.8 0.01 0.002" solref="0.02 1"/>
  </default>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 .05" condim="3" margin="0.002"/>
    <light name="l0" pos="0 0 3" mode="fixed"/>
    <camera name="c0" pos="2 0 1" mode="targetbody" target="ball0"/>
    <body name="ball0" pos="0 0 0.12">
      <freejoint/>
      <geom name="s0" type="sphere" size="0.1" condim="4" priority="1"/>
      <site name="st0" pos="0.05 0 0"/>
    </body>
    <body name="ball1" pos="0.17 0 0.13">
      <freejoint/>
      <geom name="s1" type="sphere" size="0.1" condim="1" solmix="2" margin="0.004" gap="0.001"/>
    </body>
    <body name="cap0" pos="0 0.3 0.09" euler="0 80 10">
      <freejoint/>
      <geom name="c0" type="capsule" size="0.06 0.15" condim="6"/>
    </body>
    <body name="cap1" pos="0.05 0.32 0.2" euler="0 85 40">
      <freejoint/>
      <geom name="c1" type="capsule" size="0.05 0.12" condim="3"/>
    </body>
    <body name="cap2" pos="0.5 0.5 0.3" euler="0 90 0">
      <freejoint/>
      <geom name="c2" type="capsule" size="0.04 0.1"/>
    </body>
    <body name="cap3" pos="0.5 0.5 0.385" euler="0 90 0">
      <freejoint/>
      <geom name="c3" type="capsule" size="0.04 0.1"/>
    </body>
    <body name="arm" pos="-0.6 0 0.6">
      <joint name="slide" type="slide" axis="0 0 1" range="-0.2 0.05" limited="true" damping="2" frictionloss="0.3" stiffness="5" springref="0.02"/>
      <geom type="capsule" fromto="0 0 0 0.2 0 0" size="0.03" mass="0.8"/>
      <body name="fore" pos="0.2 0 0">
        <joint name="hinge" type="hinge" axis="0 1 0" range="-40 60" limited="true" damping="0.1" armature="0.01" frictionloss="0.05" actuatorfrcrange="-3 3"/>
        <geom type="capsule" fromto="0 0 0 0.25 0 0" size="0.025" mass="0.4"/>
        <body name="pend" pos="0.25 0 0">
          <joint name="ball" type="ball" damping="0.05"/>
          <geom type="capsule" fromto="0 0 0 0 0 -0.2" size="0.02" mass="0.3"/>
          <geom name="tip" type="sphere" pos="0 0 -0.22" size="0.04" mass="0.2"/>
        </body>
      </body>
    </body>
  </worldbody>
  <actuator>
    <motor name="m_slide" joint="slide" gear="10" ctrlrange="-1 1" ctrllimited="true"/>
    <position name="p_hinge" joint="hinge" kp="20" kv="1" forcerange="-4 4" forcelimited="true"/>
    <velocity name="v_hinge" joint="hinge" kv="0.5"/>
  </actuator>
  <keyframe>
    <key name="k0" qpos="0 0 0.099 1 0 0 0  0.195 0 0.1 1 0 0 0  0 0.3 0.0595 0.7071 0 0.7071 0  0.02 0.3 0.1675 0.5 0.5 0.5 0.5  0.5 0.5 0.039 0.7071 0 0.7071 0  0.5 0.5 0.118 0.7071 0 0.7071 0  0.06 0.5  0.98 0.1 0.1 0.1"/>
  </keyframe>
</mujoco>
"""


EQUALITY_XML = """
<mujoco model="equality">
  <option timestep="0.002" iterations="50"/>
  <worldbody>
    <geom type="plane" size="0 0 .05"/>
    <body name="a1" pos="0 0 1">
      <joint name="h1" type="hinge" axis="0 1 0" damping="0.1"/>
      <geom type="capsule" fromto="0 0 0 0.3 0 0" size="0.02"/>
      <body name="a2" pos="0.3 0 0">
        <joint name="h2" type="hinge" axis="0 1 0" damping="0.1"/>
        <geom type="capsule" fromto="0 0 0 0 0 -0.3" size="0.02"/>
        <site name="sa2" pos="0 0.01 -0.1" euler="20 0 40"/>
      </body>
    </body>
    <body name="b1" pos="0 0 0.7">
      <joint name="h3" type="hinge" axis="0 1 0"/>
      <geom type="capsule" fromto="0 0 0 0.3 0 0" size="0.02" contype="0" conaffinity="0"/>
    </body>
    <body name="ballarm" pos="0 0.5 1">
      <joint name="bj" type="ball" limited="true" range="0 30" damping="0.05"/>
      <geom type="capsule" fromto="0 0 0 0 0 -0.3" size="0.03"/>
    </body>
    <body name="f1" pos="0.6 0.5 0.5"><freejoint/><geom type="sphere" size="0.05"/></body>
    <body name="f2" pos="0.8 0.5 0.5"><freejoint/><geom type="box" size="0.04 0.04 0.04"/><site name="sf2" pos="0.01 0 0.02"/></body>
    <body name="s1" pos="-0.5 0 0.5"><joint name="sl1" type="slide" axis="0 0 1"/><geom type="sphere" size="0.04"/></body>
    <body name="s2" pos="-0.7 0 0.5"><joint name="sl2" type="slide" axis="0 0 1" damping="1"/><geom type="sphere" size="0.04"/></body>
    <body name="s3" pos="-0.9 0 0.5"><joint name="sl3" type="slide" axis="1 0 0"/><geom type="sphere" size="0.04"/></body>
    <body name="target" mocap="true" pos="0.3 -0.5 0.4" quat="0.9238795 0 0.3826834 0">
      <geom name="paddle" type="box" size="0.15 0.15 0.01" contype="2" conaffinity="2"/>
      <body name="target_child" pos="0 0 0.1"><geom type="sphere" size="0.03" contype="0" conaffinity="0"/></body>
    </body>
    <body name="puck" pos="0.3 -0.5 0.47"><freejoint/><geom type="sphere" size="0.05" contype="2" conaffinity="2"/></body>
    <body name="follower" pos="0.3 -0.9 0.4"><freejoint/><geom type="sphere" size="0.04" contype="0" conaffinity="0"/><site name="sfol" pos="0 0.02 0"/></body>
  </worldbody>
  <equality>
    <connect body1="a2" body2="b1" anchor="0 0 -0.3"/>
    <weld body1="f1" body2="f2" torquescale="0.8"/>
    <joint joint1="sl1" joint2="sl2" polycoef="0 0.5 0.1 0 0"/>
    <joint joint1="sl3" polycoef="0.05 0 0 0 0" solref="0.03 1"/>
    <connect body1="s2" anchor="0.1 0 0" solimp="0.8 0.9 0.01 0.5 2"/>
    <weld body1="s1" body2="s3" active="false"/>
    <weld body1="follower" body2="target_child" solref="0.01 1"/>
  </equality>
  <sensor>
    <force name="fa2" site="sa2"/> <torque name="ta2" site="sa2"/> <force name="ff2" site="sf2"/> <torque name="tf2" site="sf2"/>
    <force name="ffol" site="sfol"/> <torque name="tfol" site="sfol"/>
  </sensor>
  <actuator>
    <motor joint="h1" gear="2"/>
    <motor joint="sl1" gear="5"/>
  </actuator>
  <keyframe>
    <key name="k0" qpos="0 0 0  0.9396926 0.3420201 0 0  0.6 0.5 0.5 1 0 0 0  0.8 0.5 0.5 1 0 0 0  0 0 0  0.3 -0.5 0.47 1 0 0 0  0.3 -0.9 0.4 1 0 0 0"/>
  </keyframe>
</mujoco>
"""


def pairs_xml():
  """MIXED_XML plus explicit contact pairs: a fully specified pair that overrides two colliding capsules (own condim,
  5-vector friction, solref / solreffriction / solimp, margin, gap) and a pair between geoms the contype filter would drop."""
  x = MIXED_XML.replace("</actuator>", """</actuator>
  <contact>
    <pair geom1="c0" geom2="c1" condim="4" friction="0.6 0.5 0.02 0.003 0.004" solref="0.015 0.9" solreffriction="0.03 1.1"
          solimp="0.85 0.97 0.002 0.4 2" margin="0.01" gap="0.003"/>
    <pair geom1="floor" geom2="s1" condim="3" friction="1.1 1.1 0.01 0.001 0.001" solref="0.02 1" solimp="0.9 0.95 0.001 0.5 2" margin="0.006" gap="0"/>
  </contact>""")
  return x.replace('<option timestep="0.004"', '<option cone="elliptic" timestep="0.004"')


def passive_xml():
  """MIXED_XML with the remaining passive-force features switched on: gravity compensation (one body routed through the
  actuators with actuatorgravcomp), a ball-joint spring and a free-joint spring / damper."""
  x = MIXED_XML
  for a, b in (
    ('<body name="pend" pos="0.25 0 0">', '<body name="pend" pos="0.25 0 0" gravcomp="0.7">'),
    ('<joint name="ball" type="ball" damping="0.05"/>', '<joint name="ball" type="ball" damping="0.05" stiffness="2"/>'),
    ('<body name="ball0" pos="0 0 0.12">\n      <freejoint/>', '<body name="ball0" pos="0 0 0.12" gravcomp="0.3">\n      <joint type="free" stiffness="3" damping="0.2"/>'),
    ('<body name="arm" pos="-0.6 0 0.6">', '<body name="arm" pos="-0.6 0 0.6" gravcomp="1">'),
    ('<joint name="slide" type="slide" axis="0 0 1"', '<joint name="slide" type="slide" actuatorgravcomp="true" axis="0 0 1"'),
  ):
    assert a in x, a
    x = x.replace(a, b)
  return x


CONVEX_XML = """
<mujoco model="convex">
  <option timestep="0.002" iterations="50"/>
  <default><geom friction="0.9 0.01 0.002"/></default>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 .05" condim="3"/>
    <body name="box_static" pos="0 0 0.099"><geom type="box" size="0.25 0.25 0.1" density="500"/></body>
    <body name="cyl_on_box" pos="0.05 0.02 0.277"><freejoint/><geom type="cylinder" size="0.07 0.08"/></body>
    <body name="ell_on_box" pos="-0.1 -0.1 0.247"><freejoint/><geom type="ellipsoid" size="0.06 0.09 0.05"/></body>
    <body name="cyl_a_static" pos="0.8 0 0.099"><geom type="cylinder" size="0.1 0.1"/></body>
    <body name="cyl_b" pos="0.82 0.03 0.277" euler="0 90 0"><freejoint/><geom type="cylinder" size="0.08 0.12"/></body>
    <body name="cap_on_cyl" pos="0.8 0.45 0.247" euler="90 0 0"><freejoint/><geom type="capsule" size="0.05 0.12"/></body>
    <body name="cyl_c_static" pos="0.8 0.45 0.099"><geom type="cylinder" size="0.12 0.1"/></body>
    <body name="ell_a_static" pos="-0.8 0 0.059"><geom type="ellipsoid" size="0.15 0.1 0.06"/></body>
    <body name="ell_b" pos="-0.78 0.02 0.165" euler="10 0 30"><freejoint/><geom type="ellipsoid" size="0.08 0.06 0.05"/></body>
    <body name="sph_on_ell" pos="-0.8 0.5 0.166"><freejoint/><geom type="sphere" size="0.05"/></body>
    <body name="ell_c_static" pos="-0.8 0.5 0.059"><geom type="ellipsoid" size="0.12 0.12 0.06"/></body>
    <body name="cap_on_ell" pos="-0.8 -0.5 0.205" euler="0 90 0"><freejoint/><geom type="capsule" size="0.04 0.1"/></body>
    <body name="ell_d_static" pos="-0.8 -0.5 0.079"><geom type="ellipsoid" size="0.15 0.1 0.08" margin="0.004"/></body>
    <body name="ell_on_cyl" pos="0 0.8 0.236"><freejoint/><geom type="ellipsoid" size="0.07 0.07 0.04"/></body>
    <body name="cyl_d_static" pos="0 0.8 0.099"><geom type="cylinder" size="0.1 0.1"/></body>
  </worldbody>
</mujoco>
"""


def boxccd_xml(mixed=False):
  """Boxes under default options: box-box goes through GJK / EPA + multi-contact recovery (collision_convex.py:875-912).
  Face-face (full, overhanging and 45-degree octagon overlap), edge-face with the edge on either geom, vertex-face and crossed edges.
  mixed=True swaps the corner-down box for a cylinder so the model has a non-box convex pair (EPA keeps ccd_iterations instead of 16)."""
  corner = ('<body pos="-0.3 0 0.1836" euler="45 35.264 0"><freejoint/><geom type="box" size="0.05 0.05 0.05"/></body>' if not mixed else
            '<body pos="-0.3 0 0.159"><freejoint/><geom type="cylinder" size="0.05 0.06"/></body>')
  return f"""
<mujoco>
  <option timestep="0.002" iterations="50"/>
  <default><geom friction="0.9 0.01 0.002" density="400"/></default>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 .05"/>
    <geom name="platform" type="box" size="0.5 0.5 0.05" pos="0 0 0.05"/>
    <body pos="-0.3 -0.3 0.149"><freejoint/><geom type="box" size="0.08 0.08 0.05"/></body>
    <body pos="-0.25 -0.27 0.238"><freejoint/><geom type="box" size="0.06 0.06 0.04"/></body>
    <body pos="0 -0.3 0.149" euler="0 0 45"><freejoint/><geom type="box" size="0.07 0.07 0.05"/></body>
    <body pos="0 -0.3 0.228"><freejoint/><geom type="box" size="0.07 0.07 0.03"/></body>
    <body pos="0.3 -0.3 0.1697" euler="45 0 0"><freejoint/><geom type="box" size="0.05 0.05 0.05"/></body>
    {corner}
    <body pos="0.3 0.2 0.2346" euler="45 0 0"><freejoint/><geom type="box" size="0.04 0.04 0.04"/></body>
    <body pos="0.3 0.2 0.139"><freejoint/><geom type="box" size="0.1 0.1 0.04"/></body>
    <body pos="0 0.3 0.1697" euler="45 0 0"><freejoint/><geom type="box" size="0.05 0.05 0.05"/></body>
    <body pos="0 0.3 0.3101" euler="0 45 0"><freejoint/><geom type="box" size="0.05 0.05 0.05"/></body>
  </worldbody>
</mujoco>"""


def sensor_xml():
  """MIXED_XML with one sensor of every type this build carries (two with cutoffs), sites on a free body and on the arm chain."""
  x = MIXED_XML.replace('<geom name="tip" type="sphere" pos="0 0 -0.22" size="0.04" mass="0.2"/>',
                        '<geom name="tip" type="sphere" pos="0 0 -0.22" size="0.04" mass="0.2"/>\n          <site name="imu" pos="0.01 0.02 -0.1" euler="10 20 30"/>')
  x = x.replace('<site name="st0" pos="0.05 0 0"/>', '<site name="st0" pos="0.05 0 0"/>\n      <site name="tz_box" type="box" size="0.12 0.12 0.12"/>\n      <site name="tz_sph" pos="0 0 -0.08" size="0.05"/>')
  x = x.replace('<geom name="c0" type="capsule" size="0.06 0.15" condim="6"/>', '<geom name="c0" type="capsule" size="0.06 0.15" condim="6"/>\n      <site name="tz_cap" type="capsule" size="0.07 0.16"/>')
  x = x.replace('<geom name="c1" type="capsule" size="0.05 0.12" condim="3"/>', '<geom name="c1" type="capsule" size="0.05 0.12" condim="3"/>\n      <site name="tz_ell" type="ellipsoid" size="0.06 0.06 0.2"/>')
  x = x.replace('<geom name="c2" type="capsule" size="0.04 0.1"/>', '<geom name="c2" type="capsule" size="0.04 0.1"/>\n      <site name="tz_cyl" type="cylinder" size="0.05 0.08"/>')
  sensors = """
  <sensor>
    <jointpos name="jp" joint="hinge"/> <jointvel name="jv" joint="slide"/> <ballquat name="bq" joint="ball"/> <ballangvel name="bv" joint="ball"/>
    <actuatorpos name="ap" actuator="p_hinge"/> <actuatorvel name="av" actuator="v_hinge"/> <actuatorfrc name="af" actuator="p_hinge" cutoff="2"/>
    <jointactuatorfrc name="jaf" joint="hinge"/>
    <gyro name="gy" site="imu"/> <velocimeter name="vm" site="imu"/> <accelerometer name="ac" site="imu" cutoff="50"/>
    <gyro name="gy0" site="st0"/> <accelerometer name="ac0" site="st0"/>
    <force name="ft_f" site="imu"/> <torque name="ft_t" site="imu"/> <force name="f0" site="st0"/> <torque name="t0" site="st0"/>
    <subtreecom name="sc" body="arm"/> <subtreelinvel name="sl" body="fore"/> <subtreeangmom name="sa" body="arm"/> <subtreeangmom name="sa0" body="cap0"/>
    <framepos name="fp" objtype="site" objname="imu"/> <framexaxis name="fx" objtype="geom" objname="tip"/> <frameyaxis name="fy" objtype="body" objname="pend"/>
    <framezaxis name="fz" objtype="xbody" objname="fore"/> <framepos name="fc" objtype="camera" objname="c0"/>
    <framequat name="fq" objtype="site" objname="imu"/> <framequat name="fqb" objtype="body" objname="pend"/> <framequat name="fqx" objtype="xbody" objname="cap0"/>
    <framequat name="fqg" objtype="geom" objname="c1"/> <framequat name="fqc" objtype="camera" objname="c0"/>
    <framelinvel name="flv" objtype="site" objname="imu"/> <frameangvel name="fav" objtype="geom" objname="tip"/> <framelinvel name="flvb" objtype="body" objname="cap1"/>
    <framelinacc name="fla" objtype="site" objname="imu"/> <frameangacc name="faa" objtype="xbody" objname="pend"/> <framelinacc name="flab" objtype="body" objname="ball0"/>
    <touch name="tb" site="tz_box"/> <touch name="ts" site="tz_sph"/> <touch name="tc" site="tz_cap"/> <touch name="te" site="tz_ell"/> <touch name="ty" site="tz_cyl" cutoff="30"/>
    <jointlimitpos name="lp_s" joint="slide"/> <jointlimitvel name="lv_s" joint="slide"/> <jointlimitfrc name="lf_s" joint="slide"/>
    <jointlimitpos name="lp_h" joint="hinge"/> <jointlimitfrc name="lf_h" joint="hinge"/>
    <framepos name="rp" objtype="site" objname="imu" reftype="body" refname="ball0"/> <framequat name="rq" objtype="geom" objname="tip" reftype="site" refname="st0"/>
    <framexaxis name="rx" objtype="xbody" objname="pend" reftype="xbody" refname="cap0"/> <framezaxis name="rz" objtype="site" objname="imu" reftype="camera" refname="c0"/>
    <framelinvel name="rlv" objtype="site" objname="imu" reftype="geom" refname="c1"/> <frameangvel name="rav" objtype="body" objname="pend" reftype="site" refname="st0"/>
    <framelinvel name="rlv2" objtype="body" objname="ball1" reftype="xbody" refname="fore"/>
    <clock name="clk"/>
  </sensor>
"""
  return x.replace("  <actuator>", sensors + "  <actuator>")


def actuators_xml(integrator="Euler"):
  """Stateful actuators (na > 0) on a three-link arm above a floor: integrator, filter, exact filter (general and <position timeconst>),
  <intvelocity>, <damper>, early activation (actearly), activation limits, a velocity-dependent gain on a filtered actuator (the
  implicit integrators' d force / d velocity path), next to stateless motors."""
  return f"""
<mujoco model="actuators">
  <option timestep="0.004" integrator="{integrator}" iterations="50" ls_iterations="30"/>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 .05" condim="3"/>
    <body name="base" pos="0 0 0.5">
      <joint name="j0" type="hinge" axis="0 1 0" damping="0.2" armature="0.01"/>
      <geom type="capsule" fromto="0 0 0 0.25 0 0" size="0.03" mass="0.6"/>
      <body name="l1" pos="0.25 0 0">
        <joint name="j1" type="hinge" axis="0 1 0" damping="0.1" range="-100 100" limited="true"/>
        <geom type="capsule" fromto="0 0 0 0.2 0 0" size="0.025" mass="0.4"/>
        <body name="l2" pos="0.2 0 0">
          <joint name="j2" type="hinge" axis="0 0 1" damping="0.05"/>
          <joint name="j3" type="slide" axis="1 0 0" damping="0.5" range="-0.05 0.1" limited="true"/>
          <geom type="capsule" fromto="0 0 0 0.15 0 0" size="0.02" mass="0.2"/>
          <geom name="tip" type="sphere" pos="0.17 0 0" size="0.03" mass="0.1"/>
        </body>
      </body>
    </body>
    <body name="cart" pos="-0.4 0 0.06">
      <joint name="cx" type="slide" axis="1 0 0" damping="1"/>
      <joint name="cz" type="slide" axis="0 0 1"/>
      <geom type="box" size="0.08 0.05 0.05" mass="1"/>
      <body name="pole" pos="0 0 0.05">
        <joint name="cp" type="hinge" axis="0 1 0" damping="0.02"/>
        <geom type="capsule" fromto="0 0 0 0 0 0.3" size="0.015" mass="0.2"/>
      </body>
    </body>
  </worldbody>
  <actuator>
    <general name="a_int" joint="j0" dyntype="integrator" gainprm="4" actlimited="true" actrange="-0.6 0.6" ctrlrange="-2 2" ctrllimited="true"/>
    <general name="a_filt" joint="j1" dyntype="filter" dynprm="0.05" gaintype="affine" gainprm="6 0.5 -0.3" biastype="affine" biasprm="0.1 -2 -0.2"/>
    <general name="a_fex" joint="j2" dyntype="filterexact" dynprm="0.02" gainprm="1.5" actearly="true" forcerange="-1 1" forcelimited="true"/>
    <position name="a_pos" joint="j3" kp="60" kv="3" timeconst="0.03"/>
    <intvelocity name="a_iv" joint="cx" kp="30" kv="2" actrange="-0.3 0.3"/>
    <damper name="a_damp" joint="cp" kv="0.4" ctrlrange="0 1"/>
    <motor name="a_mot" joint="cz" gear="3"/>
    <general name="a_int_early" joint="cp" dyntype="integrator" gainprm="0.5" actearly="true" actlimited="true" actrange="-0.2 0.2"/>
  </actuator>
  <keyframe>
    <key name="k0" qpos="0.3 -0.5 0.2 0.01 0 0 0.1"/>
  </keyframe>
</mujoco>"""


def mesh_xml():
  """Mesh geoms (inline vertex data): a 7-vertex wedge (exhaustive support search) and a cube resting on the floor, a cube stacked
  on a cube (mesh-mesh multi-contact), a 26-vertex blob (hull-graph hill climbing) on the floor, and sphere / capsule / box /
  ellipsoid / cylinder bodies resting on meshes.  Oracle-only fixture for now: the CUDA collision kernels do not take meshes."""
  rng = np.random.default_rng(5)
  blob = rng.normal(size=(26, 3))
  blob = blob / np.linalg.norm(blob, axis=1, keepdims=True) * np.array([0.12, 0.1, 0.07])
  blob_s = " ".join(f"{x:.6f}" for x in blob.reshape(-1))
  return f"""
<mujoco>
  <option timestep="0.002" iterations="50"/>
  <asset>
    <mesh name="wedge" vertex="0 0 0  1 0 0  0 1 0  0 0 1  1 1 0  0.3 0.3 0.1  1 1 1" scale="0.2 0.2 0.2"/>
    <mesh name="cube" vertex="-1 -1 -1  1 -1 -1  -1 1 -1  1 1 -1  -1 -1 1  1 -1 1  -1 1 1  1 1 1" scale="0.1 0.08 0.05"/>
    <mesh name="blob" vertex="{blob_s}"/>
  </asset>
  <default><geom friction="0.9 0.01 0.002" density="600"/></default>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 .05"/>
    <body pos="0 0 0.09" euler="180 0 0"><freejoint/><geom name="wedge" type="mesh" mesh="wedge"/></body>
    <body pos="0.05 0.03 0.215"><freejoint/><geom name="ball_on_wedge" type="sphere" size="0.05"/></body>
    <body pos="0.6 0 0.049"><freejoint/><geom name="cube_a" type="mesh" mesh="cube"/></body>
    <body pos="0.62 0.01 0.147" euler="0 0 25"><freejoint/><geom name="cube_b" type="mesh" mesh="cube"/></body>
    <body pos="0.6 0 0.2445"><freejoint/><geom name="box_on_cube" type="box" size="0.04 0.04 0.05"/></body>
    <body pos="-0.5 0.3 0.068"><freejoint/><geom name="blob" type="mesh" mesh="blob"/></body>
    <body pos="-0.5 0.3 0.176"><freejoint/><geom name="cap_on_blob" type="capsule" size="0.04 0.05" euler="90 0 0"/></body>
    <body pos="-0.5 -0.4 0.049"><freejoint/><geom name="cube_c" type="mesh" mesh="cube"/></body>
    <body pos="-0.48 -0.4 0.137"><freejoint/><geom name="ell_on_cube" type="ellipsoid" size="0.06 0.05 0.04"/></body>
    <body pos="0.1 -0.6 0.049"><freejoint/><geom name="cube_d" type="mesh" mesh="cube"/></body>
    <body pos="0.1 -0.59 0.137" euler="90 0 0"><freejoint/><geom name="cyl_on_cube" type="cylinder" size="0.04 0.06"/></body>
  </worldbody>
</mujoco>"""


def tendon_xml(integrator="Euler"):
  """Fixed tendons on two planar arms and a gripper: a limited tendon (both sides reachable), tendon spring (with a dead band) and
  damper, tendon friction loss, a tendon equality coupling two fingers (with a polynomial) and a single-tendon equality, tendon
  transmissions (motor and position servo on a tendon), next to joint actuators, limits and a contact."""
  return f"""
<mujoco model="tendons">
  <option timestep="0.004" integrator="{integrator}" iterations="50" ls_iterations="30"/>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 .05" condim="3"/>
    <body name="a0" pos="0 0 0.6">
      <joint name="a0" type="hinge" axis="0 1 0" damping="0.1" armature="0.01"/>
      <geom type="capsule" fromto="0 0 0 0.2 0 0" size="0.03" mass="0.5"/>
      <body name="a1" pos="0.2 0 0">
        <joint name="a1" type="hinge" axis="0 1 0" damping="0.05" range="-120 120" limited="true"/>
        <geom type="capsule" fromto="0 0 0 0.2 0 0" size="0.025" mass="0.3"/>
        <body name="a2" pos="0.2 0 0">
          <joint name="a2" type="hinge" axis="0 1 0" damping="0.05"/>
          <geom type="capsule" fromto="0 0 0 0.15 0 0" size="0.02" mass="0.2"/>
        </body>
      </body>
    </body>
    <body name="palm" pos="-0.4 0 0.3">
      <joint name="pz" type="slide" axis="0 0 1" damping="2"/>
      <geom type="box" size="0.05 0.04 0.02" mass="0.4"/>
      <body name="f1" pos="0.04 0 -0.02">
        <joint name="f1" type="slide" axis="1 0 0" damping="1" range="-0.03 0.03" limited="true"/>
        <geom type="box" size="0.008 0.03 0.04" pos="0 0 -0.04" mass="0.05"/>
      </body>
      <body name="f2" pos="-0.04 0 -0.02">
        <joint name="f2" type="slide" axis="-1 0 0" damping="1" range="-0.03 0.03" limited="true"/>
        <geom type="box" size="0.008 0.03 0.04" pos="0 0 -0.04" mass="0.05"/>
      </body>
    </body>
    <body name="ball" pos="0.3 0.4 0.049"><freejoint/><geom type="sphere" size="0.05" mass="0.2"/></body>
  </worldbody>
  <tendon>
    <fixed name="t_lim" limited="true" range="-0.4 0.5" margin="0.01" solreflimit="0.01 1" actuatorfrcrange="-1.2 0.4"><joint joint="a0" coef="0.5"/><joint joint="a1" coef="-0.5"/></fixed>
    <fixed name="t_spring" stiffness="8" damping="0.3" springlength="-0.1 0.2"><joint joint="a1" coef="1"/><joint joint="a2" coef="0.7"/></fixed>
    <fixed name="t_fric" frictionloss="0.2" solreffriction="0.015 1"><joint joint="a2" coef="1.5"/></fixed>
    <fixed name="t_f1"><joint joint="f1" coef="1"/></fixed>
    <fixed name="t_f2"><joint joint="f2" coef="1"/></fixed>
    <fixed name="t_grip" stiffness="20"><joint joint="f1" coef="1"/><joint joint="f2" coef="1"/></fixed>
    <fixed name="t_lift" limited="true" range="-0.05 0.2"><joint joint="pz" coef="1"/></fixed>
  </tendon>
  <equality>
    <tendon name="e_couple" tendon1="t_f1" tendon2="t_f2" polycoef="0 1 0.5 0 0" solref="0.01 1"/>
    <tendon name="e_single" tendon1="t_lift" polycoef="0.02 0 0 0 0" active="false"/>
  </equality>
  <actuator>
    <motor name="m_ten" tendon="t_lim" gear="2" ctrlrange="-1 1"/>
    <motor name="m_ten2" tendon="t_lim" gear="-1.5"/>
    <position name="p_grip" tendon="t_grip" kp="40" kv="1"/>
    <motor name="m_a0" joint="a0" gear="1.5"/>
    <general name="g_lift" tendon="t_lift" gainprm="5" biastype="affine" biasprm="0 -10 -1"/>
  </actuator>
  <sensor>
    <tendonpos name="tp" tendon="t_lim"/> <tendonvel name="tv" tendon="t_spring"/> <actuatorpos name="ap" actuator="p_grip"/> <actuatorfrc name="af" actuator="m_ten"/>
  </sensor>
  <keyframe>
    <key name="k0" qpos="0.9 -0.6 0.4  0 0.01 -0.005  0.3 0.4 0.049 1 0 0 0"/>
  </keyframe>
</mujoco>"""


def rake_xml(ngeom=40):
  """One free body carrying `ngeom` small spheres in a grid, resting on a plane: more than 32 contacts in one world (the contact-row builder
  works in batches of 32 contacts), with contact dimensions 1, 3 and 4 mixed so that the rows per contact differ (1, 4, 6)."""
  spheres = "".join(
    f'<geom type="sphere" size="0.05" pos="{0.12 * (i % 8):.3f} {0.12 * (i // 8):.3f} {0.0005 * (i % 3):.4f}" condim="{(1, 3, 4)[i % 3]}" friction="{0.6 + 0.01 * i:.2f} 0.01 0.001"/>'
    for i in range(ngeom))
  return f"""
<mujoco model="rake">
  <option timestep="0.002" iterations="50" ls_iterations="30"/>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 .05" condim="1"/>
    <body name="rake" pos="0 0 0.049">
      <freejoint/>
      {spheres}
    </body>
  </worldbody>
</mujoco>"""
