"""CPU-only: the oracle reproduces the committed expected outputs for BASELINE configs[0] (kitten.obj, 4096 instanced
MeshDraws, frustum-only cull on the host CPU) and for the two-phase variant; tests/golden/make_c1_expected.py regenerates
them.  The draw-level decisions are additionally re-derived by the independent numpy restatement."""
import ctypes
import importlib.util
import os

import numpy as np

import numpy_ref as nr
from niagara_b200 import layout, scenes
from niagara_b200.lib import load_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _maker():
    spec = importlib.util.spec_from_file_location("make_c1_expected", os.path.join(ROOT, "tests", "golden", "make_c1_expected.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_oracle_reproduces_committed_vectors():
    want = np.load(os.path.join(ROOT, "tests", "golden", "c1_kitten_expected.npz"))
    got = _maker().compute()
    assert set(want.files) == set(got.keys())
    for k in want.files:
        a, b = np.asarray(want[k]), np.asarray(got[k])
        assert a.shape == b.shape and a.dtype == b.dtype, k
        assert a.tobytes() == b.tobytes(), k


def test_reference_shaders_reproduce_committed_vectors(request):
    """The same scenarios executed by the reference's own GLSL (oracle/refshader, one host thread = in-order dispatch):
    every committed array, including the ORDER of the commands, comes out byte for byte."""
    import reference_pins
    import refshader_lib

    want = np.load(os.path.join(ROOT, "tests", "golden", "c1_kitten_expected.npz"))
    with reference_pins.pinned(request, refshader_lib.available()):
        got = _maker().compute(refshader_lib.RefShaderPath)
        for k in want.files:
            if k == "a_lod":
                continue  # a diagnostic output of the oracle only (the shaders do not export the selected LOD)
            a, b = np.asarray(want[k]), np.asarray(got[k])
            assert a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes(), k
            reference_pins.check(k, b)  # as the shaders wrote it, order included


def test_config0_frustum_only_matches_numpy_restatement():
    want = np.load(os.path.join(ROOT, "tests", "golden", "c1_kitten_expected.npz"))
    s = scenes.instanced_scene(os.path.join(ROOT, "tests", "golden", "kitten.nvcg"), 4096)
    cd = s.cull_data(occlusion=False, cluster_occlusion=False, mesh_shading=False)
    pd = layout.CullData()
    load_library().nvc_host_pass_data(ctypes.byref(cd), 1, 0, ctypes.byref(pd))
    dvb = np.ones(len(s.draws), dtype=np.uint32)
    reached, visible, emit, lod = nr.drawcull_decisions(pd.to_numpy(), False, s.draws, s.meshes, dvb)
    assert int(emit.sum()) == int(want["a_count"]) and 50 < int(emit.sum()) < 4096
    cmds = want["a_commands"]
    assert np.array_equal(cmds[:, 0], np.nonzero(emit)[0])  # the oracle emits in ascending draw order
    mesh = s.meshes[s.draws["meshIndex"][emit]]
    sel = lod[emit]
    assert np.array_equal(cmds[:, 1], mesh["lods"]["indexCount"][np.arange(len(sel)), sel])
    assert np.array_equal(cmds[:, 3], mesh["lods"]["indexOffset"][np.arange(len(sel)), sel])
    assert (cmds[:, 2] == 1).all() and (cmds[:, 5] == 0).all()
    assert np.array_equal(want["a_lod"][emit], lod[emit].astype(np.uint8)) and (want["a_lod"][~emit] == 0xFF).all()
    assert len(np.unique(lod[emit])) >= 2  # more than one LOD is selected
