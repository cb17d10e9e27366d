"""Packs the MJCF model files of a mujoco_warp checkout into tests/golden/reference_models.tar.xz, the input of
tests/test_mjcf_reference_models.py and of the humanoid fixture check in tests/test_host_logic.py.

  python tools/make_reference_models.py <mujoco_warp checkout>

Every *.xml under mujoco_warp/test_data/ and benchmarks/ is stored, with the few mesh files a stored model needs to
compile as it does in the checkout.  Models whose outcome depends on megabytes of mesh assets are left out (LEFT_OUT).
The archive is byte-for-byte reproducible: sorted members, zeroed owners and times, fixed modes.
"""

import glob
import io
import lzma
import os
import sys
import tarfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference_models.tar.xz")

LEFT_OUT = {
  "mujoco_warp/test_data/mug/mug.xml": "mug.obj is 2.2 MB",
  "mujoco_warp/test_data/aloha_pot/scene.xml": "its STL / OBJ meshes are 3 MB",
  "benchmarks/kitchen/kitchen.xml": "its OBJ meshes are 5 MB",
}
ASSETS = ["mujoco_warp/test_data/meshes/tetrahedron.stl", "mujoco_warp/test_data/meshes/dodecahedron.stl"]  # ray.xml


def main(src):
  rels = [os.path.relpath(p, src) for d in ("mujoco_warp/test_data", "benchmarks") for p in glob.glob(os.path.join(src, d, "**", "*.xml"), recursive=True)]
  rels = sorted(r for r in rels if r not in LEFT_OUT) + ASSETS
  buf = io.BytesIO()
  with tarfile.open(fileobj=buf, mode="w", format=tarfile.PAX_FORMAT) as tar:
    for rel in sorted(rels):
      data = open(os.path.join(src, rel), "rb").read()
      info = tarfile.TarInfo(rel)
      info.size, info.mode, info.mtime = len(data), 0o644, 0
      tar.addfile(info, io.BytesIO(data))
  with open(OUT, "wb") as f:
    f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
  print(len(rels), "files ->", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
  main(sys.argv[1])
