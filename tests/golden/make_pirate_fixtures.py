#!/usr/bin/env python
"""Regenerates the fixtures made by the reference's cache writer (oracle/_ref/write_cache, built by `make -C oracle ref`)
from meshoptimizer's pirate demo model:

  pirate_cook.npz      pirate.obj: the fp16 positions and raw meshletdata the reference cooks from, and the Meshlet[] it
                       writes (bounds and cones included) — tests/test_cook.py
  pirate_glb.z.cache   pirate.glb (the glTF importer, several meshes and materials): the compressed cache —
                       tests/test_cook.py, tests/test_scene_cache.py

The reference checkout is the one tests/refshader_lib.py names (NIAGARA_REFERENCE).

    python tests/golden/make_pirate_fixtures.py
"""
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
MODELS = {"pirate": "extern/meshoptimizer/demo/pirate.obj", "pirate_glb": "extern/meshoptimizer/demo/pirate.glb"}


def write_cache(out_dir, name):
    """Runs the reference's writer on model `name`; returns the path prefix of what it wrote (.raw.cache, .z.cache, ...)"""
    from refshader_lib import REFERENCE

    subprocess.run([os.path.join(ROOT, "oracle", "_ref", "write_cache"), os.path.join(out_dir, name), os.path.join(REFERENCE, MODELS[name])], check=True, stdout=subprocess.DEVNULL)
    return os.path.join(out_dir, name)


def cook_inputs(cache_path):
    """(positions[n, 3] as fp16 bits, meshletdata words, Meshlet[]) of a scene cache"""
    from niagara_b200 import scene_cache

    c = scene_cache.SceneCache(cache_path)
    positions = np.ascontiguousarray(c.section("vertices")).view(np.uint16).reshape(-1, 8)[:, :3]
    return np.ascontiguousarray(positions), c.section("meshletdata"), c.section("meshlets")


def main():
    from refshader_lib import REFERENCE

    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + REFERENCE], check=True)
    with tempfile.TemporaryDirectory() as tmp:
        positions, meshletdata, meshlets = cook_inputs(write_cache(tmp, "pirate") + ".raw.cache")
        np.savez_compressed(os.path.join(HERE, "pirate_cook.npz"), positions=positions, meshletdata=meshletdata, meshlets=meshlets)
        shutil.copy(write_cache(tmp, "pirate_glb") + ".z.cache", os.path.join(HERE, "pirate_glb.z.cache"))
    for name in ("pirate_cook.npz", "pirate_glb.z.cache"):
        print(name, os.path.getsize(os.path.join(HERE, name)), "bytes")


if __name__ == "__main__":
    main()
