"""The MJCF compiler against the reference's model files: a file either compiles and passes put_model's feature checks, or is refused
with an exception that names the missing feature -- never compiled into a model with parts silently dropped.  The files come from
tests/golden/reference_models.tar.xz (every model of the reference's test_data/ and benchmarks/ but the three that need megabytes of
mesh assets; see tools/make_reference_models.py)."""

import glob
import os

import numpy as np
import pytest

from tests import util

# file (relative to the reference root) -> substring of the refusal; everything else must compile AND validate
REFUSED = {
  "mujoco_warp/test_data/actuation/adhesion.xml": "transmission", "mujoco_warp/test_data/actuation/site.xml": "transmission",
  "mujoco_warp/test_data/actuation/slidercrank.xml": "transmission", "mujoco_warp/test_data/pendula.xml": "transmission",
  "mujoco_warp/test_data/actuation/muscle.xml": "spatial", "mujoco_warp/test_data/constraints.xml": "fixed tendons combine",
  "mujoco_warp/test_data/convex_collision/box100.xml": "nv > 128", "mujoco_warp/test_data/primitives.xml": "nv > 128", "benchmarks/render/primitives.xml": "nv > 128",
  "mujoco_warp/test_data/hfield/hfield.xml": "height-field", "mujoco_warp/test_data/ray.xml": "height-field", "benchmarks/unitree_g1/scene_hfield.xml": "height-field",
  "benchmarks/cloth/scene.xml": "flexcomp",
}
PREFIX_REFUSED = {
  "mujoco_warp/test_data/flex/": ("flexcomp", {"mujoco_warp/test_data/flex/scene.xml"}),  # scene.xml is the flex-free base scene the others include
  "mujoco_warp/test_data/collision_sdf/": ("", {"mujoco_warp/test_data/collision_sdf/scene.xml"}),  # sdf plugins / mesh files that are not in the tree
  "mujoco_warp/test_data/tendon/": ("spatial", {"mujoco_warp/test_data/tendon/fixed.xml", "mujoco_warp/test_data/tendon/tendon_limit.xml"}),
  "benchmarks/aloha/": ("", set()), "benchmarks/franka_emika_panda/": ("", set()),  # menagerie mesh files are not in the tree
}


def _files(ref):
  return sorted(glob.glob(os.path.join(ref, "mujoco_warp/test_data/**/*.xml"), recursive=True)) + sorted(glob.glob(os.path.join(ref, "benchmarks/**/*.xml"), recursive=True))


def test_every_reference_model_compiles_or_is_refused_by_name(tmp_path):
  from mujoco_warp_b200._src import io as mio
  from mujoco_warp_b200._src import mjcf

  ref = util.reference_models(tmp_path)
  ok = 0
  for path in _files(ref):
    rel = os.path.relpath(path, ref)
    want = REFUSED.get(rel)
    for pre, (msg, keep) in PREFIX_REFUSED.items():
      if rel.startswith(pre) and rel not in keep:
        want = msg
    try:
      mjm = mjcf.load(path)
      mio._validate(mjm)
    except (NotImplementedError, FileNotFoundError, KeyError, ValueError) as e:
      assert want is not None, f"{rel}: unexpectedly refused: {e}"
      assert want in str(e) or want == "", f"{rel}: refused for another reason than '{want}': {e}"
      continue
    assert want is None, f"{rel}: expected a refusal mentioning '{want}', but the file compiled (nv {mjm.nv}, ngeom {mjm.ngeom})"
    ok += 1
    assert mjm.nbody >= 1 and np.isfinite(np.asarray(mjm.body_mass)).all()
  assert ok >= 20
  # benchmarks/kitchen/kitchen.xml, left out with its meshes, is the reference's model with shell-inertia meshes
  with pytest.raises(NotImplementedError, match="shell"):
    mjcf.load_string('<mujoco><asset><mesh name="w" inertia="shell" vertex="0 0 0  1 0 0  0 1 0  0 0 1"/></asset>'
                     '<worldbody><body><freejoint/><geom type="mesh" mesh="w"/></body></worldbody></mujoco>')
