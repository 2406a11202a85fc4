"""Widening N4 — meshlet bounds + normal cones (csrc/nvc_cook.cuh / nvc_cook_meshlet_bounds).
The checker is the REFERENCE itself: the Meshlet[] its cooker wrote (scene.cpp appendMeshlet ->
meshopt_computeMeshletBounds) into caches produced by oracle/refscene/write_cache.  CPU tests run the product's header
compiled for the host (tests/cook_host.cpp); the -m gpu test runs the kernel through the C ABI."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from niagara_b200 import layout, scene_cache

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
CULL_FIELDS = 12  # center[3] + radius (fp16) + cone_axis[3] + cone_cutoff (int8): the first 12 bytes of a Meshlet


def _host_lib():
    out = os.path.join(HERE, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libcookhost.so")
    srcs = [os.path.join(HERE, "cook_host.cpp"), os.path.join(ROOT, "niagara_b200", "csrc", "nvc_cook.cuh"), os.path.join(ROOT, "include", "niagara_cull.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-x", "c++", srcs[0], "-o", so], check=True)
    return ctypes.CDLL(so)


def _inputs(cache_path):
    c = scene_cache.SceneCache(cache_path)
    assert not c.header.compressed
    vertices = np.ascontiguousarray(c.section("vertices"))  # raw bytes, 16 per vertex
    return vertices, c.section("meshletdata"), c.section("meshlets")


def _scrub(meshlets):
    m = meshlets.copy()
    m.view(np.uint8).reshape(len(m), 24)[:, :CULL_FIELDS] = 0xCD
    return m


def _check(got, want, what):
    g = got.view(np.uint8).reshape(len(got), 24)
    w = want.view(np.uint8).reshape(len(want), 24)
    bad = np.nonzero((g != w).any(1))[0]
    assert len(bad) == 0, (what, len(bad), bad[:5], got[bad[:3]], want[bad[:3]])


def test_host_instantiation_reproduces_reference_cooker_animated():
    lib = _host_lib()
    vertices, data, want = _inputs(os.path.join(GOLDEN, "animated.raw.cache"))
    got = _scrub(want)
    lib.cookhost_meshlet_bounds(vertices.ctypes.data, len(vertices) // 16, data.ctypes.data, len(data), got.ctypes.data, len(got))
    _check(got, want, "animated")
    assert len(np.unique(want["cone_cutoff"])) > 3 and (want["radius"] != 0).all()


def _pirate_fixtures():
    import importlib.util

    spec = importlib.util.spec_from_file_location("make_pirate_fixtures", os.path.join(GOLDEN, "make_pirate_fixtures.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_host_instantiation_reproduces_reference_cooker_real_meshes(tmp_path):
    """792 + ~300 meshlets cooked by the reference (all LODs, short and long reference lists, wide cones): right now where the
    reference is present — the stored copies must then be what it writes — from kitten_cook.npz + kitten.nvcg, pirate_cook.npz
    and pirate_glb.z.cache elsewhere (tests/golden/make_pirate_fixtures.py)."""
    from refshader_lib import REFERENCE

    fixtures = _pirate_fixtures()
    lib = _host_lib()
    live = os.path.isdir(os.path.join(REFERENCE, "src"))
    if live:
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + REFERENCE], check=True)
    total = 0
    for name in ("kitten", "pirate", "pirate_glb"):
        if live:
            if name == "kitten":
                subprocess.run([os.path.join(ROOT, "oracle", "_ref", "write_cache"), str(tmp_path / name), os.path.join(REFERENCE, "data", "kitten.obj")], check=True, stdout=subprocess.DEVNULL)
            else:
                fixtures.write_cache(str(tmp_path), name)
            positions, data, want = fixtures.cook_inputs(str(tmp_path / (name + ".raw.cache")))
            if name == "pirate":
                stored = np.load(os.path.join(GOLDEN, "pirate_cook.npz"))
                assert all(np.array_equal(stored[k], v) for k, v in (("positions", positions), ("meshletdata", data), ("meshlets", want)))
            elif name == "pirate_glb":
                assert open(tmp_path / "pirate_glb.z.cache", "rb").read() == open(os.path.join(GOLDEN, "pirate_glb.z.cache"), "rb").read()
        elif name == "kitten":
            z = np.load(os.path.join(GOLDEN, "kitten_cook.npz"))
            positions, data, want = z["positions"], z["meshletdata"], layout.load_nvcg(os.path.join(GOLDEN, "kitten.nvcg"))[1]
        elif name == "pirate":
            z = np.load(os.path.join(GOLDEN, "pirate_cook.npz"))
            positions, data, want = z["positions"], z["meshletdata"], z["meshlets"]
        else:  # the reference's compressed cache, read by the product's decoders (checked against the reference's in test_scene_cache.py)
            positions, data, want = fixtures.cook_inputs(os.path.join(GOLDEN, "pirate_glb.z.cache"))
        vertices = np.zeros((len(positions), 8), dtype=np.uint16)
        vertices[:, :3] = positions
        got = _scrub(want)
        lib.cookhost_meshlet_bounds(vertices.ctypes.data, len(vertices), data.ctypes.data, len(data), got.ctypes.data, len(got))
        _check(got, want, name)
        total += len(want)
    assert total > 900


def test_committed_kitten_inputs_match():
    """kitten_cook.npz (positions + raw meshletdata of the cooked kitten, for the GPU box where the reference is absent)
    reproduces kitten.nvcg's Meshlet[] through the host instantiation."""
    lib = _host_lib()
    z = np.load(os.path.join(GOLDEN, "kitten_cook.npz"))
    _, want, _ = layout.load_nvcg(os.path.join(GOLDEN, "kitten.nvcg"))
    positions, data = z["positions"], z["meshletdata"]  # keep the arrays alive while the C code reads them
    vertices = np.zeros((len(positions), 8), dtype=np.uint16)
    vertices[:, :3] = positions
    got = _scrub(want)
    lib.cookhost_meshlet_bounds(vertices.ctypes.data, len(vertices), data.ctypes.data, len(data), got.ctypes.data, len(got))
    _check(got, want, "kitten")


@pytest.mark.gpu
def test_gpu_kernel_reproduces_reference_cooker():
    import torch

    from niagara_b200.lib import check, load_library

    assert torch.cuda.is_available()
    lib = load_library()
    ctx = ctypes.c_void_p()
    check(lib.nvc_create(0, None, ctypes.byref(ctx)), None, "nvc_create")
    try:
        cases = []
        vertices, data, want = _inputs(os.path.join(GOLDEN, "animated.raw.cache"))
        cases.append(("animated", vertices, data, want))
        z = np.load(os.path.join(GOLDEN, "kitten_cook.npz"))
        _, kw, _ = layout.load_nvcg(os.path.join(GOLDEN, "kitten.nvcg"))
        kv = np.zeros((len(z["positions"]), 8), dtype=np.uint16)
        kv[:, :3] = z["positions"]
        cases.append(("kitten", kv.view(np.uint8).reshape(-1), z["meshletdata"], kw))
        for name, vertices, data, want in cases:
            dv = torch.from_numpy(np.ascontiguousarray(vertices).view(np.uint8).reshape(-1).copy()).cuda()
            dd = torch.from_numpy(np.ascontiguousarray(data).view(np.int32).copy()).cuda()
            dm = torch.from_numpy(_scrub(want).view(np.uint8).reshape(-1).copy()).cuda()
            rej = torch.full((1,), 77, dtype=torch.int32, device="cuda")
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            check(lib.nvc_cook_meshlet_bounds(ctx, stream, dv.data_ptr(), dv.numel() // 16, dd.data_ptr(), dd.numel(), dm.data_ptr(), len(want), rej.data_ptr()), ctx, "nvc_cook_meshlet_bounds")
            torch.cuda.synchronize()
            assert int(rej.item()) == 0
            _check(dm.cpu().numpy().view(layout.MESHLET_DTYPE), want, name)
            # a meshlet pointing past the arrays is rejected and left alone
            broken = _scrub(want)
            broken["dataOffset"][0] = len(data)
            broken["baseVertex"][1] = dv.numel() // 16
            dm = torch.from_numpy(broken.view(np.uint8).reshape(-1).copy()).cuda()
            check(lib.nvc_cook_meshlet_bounds(ctx, stream, dv.data_ptr(), dv.numel() // 16, dd.data_ptr(), dd.numel(), dm.data_ptr(), len(want), rej.data_ptr()), ctx, "nvc_cook_meshlet_bounds")
            torch.cuda.synchronize()
            assert int(rej.item()) == 2
            out = dm.cpu().numpy().view(layout.MESHLET_DTYPE)
            assert np.array_equal(out[:2], broken[:2])
            _check(out[2:], want[2:], name + " rest")
    finally:
        lib.nvc_destroy(ctx)


def test_host_instantiation_against_reference_bounds_on_random_meshlets(request):
    """Property test: random meshlets (smooth patches, random soups -> cones wider than a hemisphere, fans, degenerate and
    duplicated triangles, single triangles, collinear points) through meshopt_computeMeshletBounds + meshopt_quantizeHalf of
    the reference's vendored library vs the product's nvc_cook.cuh: identical center / radius / cone bytes.  Without the
    reference library the inputs are quantised by the product's restatement of meshopt_quantizeHalf, and inputs and bounds
    are held to the reference's, pinned per 100 cases."""
    import reference_pins
    import test_meshopt_decoders

    live = test_meshopt_decoders.load_ref() is not None
    with reference_pins.pinned(request, live):
        _random_meshlet_bounds(live)


def _random_meshlet_bounds(live):
    lib = _host_lib()
    lib.cookhost_quantize_half.restype = ctypes.c_ushort
    lib.cookhost_quantize_half.argtypes = [ctypes.c_float]
    if not live:
        return _random_meshlet_cases(lib, None)
    mo = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libmeshopt_ref.so"))

    class Bounds(ctypes.Structure):
        _fields_ = [("center", ctypes.c_float * 3), ("radius", ctypes.c_float), ("cone_apex", ctypes.c_float * 3), ("cone_axis", ctypes.c_float * 3),
                    ("cone_cutoff", ctypes.c_float), ("cone_axis_s8", ctypes.c_byte * 3), ("cone_cutoff_s8", ctypes.c_byte)]

    mo.meshopt_computeMeshletBounds.restype = Bounds
    mo.meshopt_computeMeshletBounds.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t]
    mo.meshopt_quantizeHalf.restype = ctypes.c_ushort
    mo.meshopt_quantizeHalf.argtypes = [ctypes.c_float]
    mo.meshopt_dequantizeHalf.restype = ctypes.c_float
    mo.meshopt_dequantizeHalf.argtypes = [ctypes.c_ushort]
    return _random_meshlet_cases(lib, mo)


def _random_meshlet_cases(lib, mo):
    """mo: the reference's meshoptimizer, or None (the reference's results are then the pinned ones)"""
    import reference_pins

    quantize = lib.cookhost_quantize_half if mo is None else mo.meshopt_quantizeHalf
    rng = np.random.default_rng(77)
    halves, bounds = [], []
    seen = {"degenerate": 0, "wide": 0, "cone": 0}
    for case in range(1500):
        vc = int(rng.integers(3, 65))
        tc = int(rng.integers(1, 97))
        style = case % 6
        grid = None
        if style in (0, 3):  # consistently wound grid patches: tight normal cones
            gx = int(rng.integers(2, 9))
            gy = int(rng.integers(2, 64 // gx + 1))
            vc = gx * gy
            u, v = np.meshgrid(np.linspace(-1, 1, gx), np.linspace(-1, 1, gy))
            uv = np.stack([u.reshape(-1), v.reshape(-1)], 1) + rng.uniform(-0.02, 0.02, (vc, 2))
            q = np.arange((gx - 1) * (gy - 1))
            x, y = q % (gx - 1), q // (gx - 1)
            a, b_, c, d = y * gx + x, y * gx + x + 1, (y + 1) * gx + x, (y + 1) * gx + x + 1
            grid = np.stack([a, b_, c, c, b_, d], 1).reshape(-1, 3)[:96]
            tc = len(grid)
        if style == 0:  # smooth height-field patch
            pos = np.concatenate([uv, 0.15 * np.sin(uv[:, :1] * 2) * np.cos(uv[:, 1:] * 3)], 1) * rng.uniform(0.01, 30)
        elif style == 1:  # random soup
            pos = rng.standard_normal((vc, 3)) * rng.uniform(0.001, 100)
        elif style == 2:  # all points on a line / duplicated points: zero-area triangles
            t = rng.uniform(-1, 1, (vc, 1))
            pos = t * rng.standard_normal((1, 3)) + (0 if rng.random() < 0.5 else rng.standard_normal((1, 3)))
            if rng.random() < 0.5:
                pos[:] = pos[0]
        elif style == 3:  # sphere cap
            d = np.concatenate([uv * rng.uniform(0.1, 0.9), np.ones((vc, 1))], 1)
            pos = d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(0.1, 5) + rng.standard_normal((1, 3))
        elif style == 4:  # planar polygon fan: every normal identical
            a = np.sort(rng.uniform(0, 2 * np.pi, vc))
            pos = np.stack([np.cos(a), np.sin(a), np.zeros(vc)], 1) * rng.uniform(0.5, 3) + rng.standard_normal((1, 3))
        else:  # tiny and huge coordinates (fp16 flush-to-zero / large magnitudes)
            pos = rng.standard_normal((vc, 3)) * (1e-5 if rng.random() < 0.5 else 2e4)
        half = np.array([quantize(float(x)) for x in pos.reshape(-1)], np.uint16).reshape(vc, 3)
        if mo is not None:
            assert np.array_equal(half.reshape(-1), [lib.cookhost_quantize_half(float(x)) for x in pos.reshape(-1)]), case
        if grid is not None:
            tris = grid.copy()
        elif style == 4:
            i = 1 + np.arange(tc) % max(1, vc - 2)
            tris = np.stack([np.zeros(tc, np.int64), i, i + 1], 1)
        else:
            tris = rng.integers(0, vc, (tc, 3))
        if rng.random() < 0.2:
            tris[rng.integers(0, tc)] = tris[rng.integers(0, tc)][[0, 0, 1]]  # a degenerate triangle in the middle
        tris = np.ascontiguousarray(tris, dtype=np.uint8)
        # make the reference list cover exactly the used prefix, as a well-formed meshlet does
        used = int(tris.max()) + 1
        base = int(rng.integers(0, 1000))
        refs = np.arange(used, dtype=np.uint32) if rng.random() < 0.5 else rng.permutation(vc).astype(np.uint32)[:used]
        short = bool(rng.integers(0, 2))

        if mo is not None:
            # the reference: float positions = dequantised halves, indexed by (baseVertex-relative) reference
            fpos = np.array([mo.meshopt_dequantizeHalf(int(h)) for h in half.reshape(-1)], np.float32).reshape(vc, 3)
            b = mo.meshopt_computeMeshletBounds(refs.ctypes.data, tris.ctypes.data, tc, fpos.ctypes.data, vc, 12)
            want = np.zeros(1, layout.MESHLET_DTYPE)
            want["center"] = [mo.meshopt_quantizeHalf(b.center[k]) for k in range(3)]
            want["radius"] = mo.meshopt_quantizeHalf(b.radius)
            want["cone_axis"] = [b.cone_axis_s8[k] for k in range(3)]
            want["cone_cutoff"] = b.cone_cutoff_s8

        # the product: Vertex[] with the fp16 positions at baseVertex, meshletdata = references (+ pad) + triangle bytes
        vertices = np.zeros((base + vc, 8), np.uint16)
        vertices[base:, :3] = half
        if short:
            words = np.zeros((used + 1) // 2, np.uint32)
            words.view(np.uint16)[:used] = refs
        else:
            words = refs.copy()
        tri_words = np.zeros((tc * 3 + 3) // 4, np.uint32)
        tri_words.view(np.uint8)[: tc * 3] = tris.reshape(-1)
        data = np.concatenate([np.zeros(5, np.uint32), words, tri_words])
        m = np.zeros(1, layout.MESHLET_DTYPE)
        m["dataOffset"], m["baseVertex"], m["vertexCount"], m["triangleCount"], m["shortRefs"] = 5, base, used, tc, int(short)
        got = m.copy()
        got.view(np.uint8).reshape(1, 24)[:, :CULL_FIELDS] = 0xCD
        lib.cookhost_meshlet_bounds(vertices.ctypes.data, len(vertices), data.ctypes.data, len(data), got.ctypes.data, 1)
        if mo is not None:
            for f in ("center", "radius", "cone_axis", "cone_cutoff"):
                assert np.array_equal(got[f], want[f]), (case, style, f, got[f], want[f])
            seen["degenerate" if (b.radius == 0 and b.cone_cutoff_s8 == 0) else ("wide" if b.cone_cutoff_s8 == 127 and not any(b.cone_axis_s8) else "cone")] += 1
        halves.append(half.reshape(-1))
        bounds.append((want if mo is not None else got).view(np.uint8)[:CULL_FIELDS])
        if len(bounds) == 100:
            reference_pins.check("cases %d-%d: inputs, bounds" % (case - 99, case), np.concatenate(halves), np.concatenate(bounds))
            halves, bounds = [], []
    if mo is not None:  # (the pinned inputs are the reference's, so is their spread over the three kinds)
        assert seen["degenerate"] > 50 and seen["wide"] > 200 and seen["cone"] > 300, seen
