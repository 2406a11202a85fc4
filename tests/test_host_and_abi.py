"""CPU-only: the C ABI library loads, exports every symbol the header declares, the host-side helpers match
the glm/GCC-built golden vectors, and the product path refuses to run without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from niagara_b200 import host, layout, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported():
    header = open(os.path.join(ROOT, "include", "niagara_cull.h")).read()
    declared = set(re.findall(r"NVC_API\s+[\w\s\*]+?\b(nvc_\w+)\s*\(", header))
    assert len(declared) >= 19, declared
    l = ctypes.CDLL(lib.library_path())
    for name in sorted(declared):
        assert hasattr(l, name), "libniagara_cull.so does not export %s" % name
    bound = {s[0] for s in lib.SIGNATURES}
    assert declared == bound, declared ^ bound


def test_no_torch_types_in_abi():
    header = open(os.path.join(ROOT, "include", "niagara_cull.h")).read()
    code = re.sub(r"/\*.*?\*/", "", header, flags=re.S)  # strip comments
    assert "torch" not in code and "at::" not in code and "cudaStream_t" not in code and "#include <cuda" not in code


def test_header_is_plain_c(tmp_path):
    """include/niagara_cull.h compiles as strict C99 (the boundary a cgo / FFI binding would consume) and links against
    the library from a C program that calls host-only entry points."""
    import subprocess

    src = tmp_path / "abi.c"
    src.write_text(
        '#include "niagara_cull.h"\n#include <stdio.h>\n'
        "int main(void) { NvcHiZ h; if (nvc_hiz_layout(1920, 1080, &h) != NVC_OK) return 1;\n"
        '  printf("%u %u %u %s\\n", h.width, h.height, h.levels, nvc_status_string(NVC_ERROR_CORRUPT)); return sizeof(NvcMeshlet) == 24 ? 0 : 2; }\n'
    )
    exe = tmp_path / "abi"
    lib_dir = os.path.join(ROOT, "niagara_b200")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L", lib_dir, "-lniagara_cull", "-Wl,-rpath," + lib_dir], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert out[:3] == ["1024", "1024", "11"] and " ".join(out[3:]) == "corrupt scene cache"


def test_layout_sizes():
    assert layout.MESHLET_DTYPE.itemsize == 24 and layout.MESHLET_DTYPE.fields["cone_axis"][1] == 8
    assert layout.MESH_DTYPE.itemsize == 208 and layout.MESH_DTYPE.fields["lods"][1] == 48 and layout.MESH_DTYPE.fields["lodCount"][1] == 32
    assert layout.MESHDRAW_DTYPE.itemsize == 48 and layout.MESHDRAW_DTYPE.fields["meshIndex"][1] == 32
    assert layout.MESHTASKCOMMAND_DTYPE.itemsize == 20 and layout.MESHDRAWCOMMAND_DTYPE.itemsize == 24
    f = layout.CULLDATA_DTYPE.fields
    assert layout.CULLDATA_DTYPE.itemsize == 144
    assert [f[n][1] for n in ("P00", "frustum", "lodTarget", "drawCount", "clusterBackfaceEnabled", "postPass")] == [64, 80, 96, 108, 128, 132]
    assert ctypes.sizeof(layout.CullData) == 144


def test_previous_pow2_and_mips():
    # niagara.cpp:439-447: largest power of two STRICTLY below v (except v <= 2 -> 1)
    for v, want in [(1, 1), (2, 1), (3, 2), (4, 2), (5, 4), (1024, 512), (768, 512), (1920, 1024), (1080, 1024), (4096, 2048), (4097, 4096)]:
        assert host.previous_pow2(v) == want, v
    # resources.cpp:280-292
    for (w, h), want in [((1, 1), 1), ((2, 2), 2), ((512, 512), 10), ((2048, 2048), 12), ((1024, 512), 11), ((2048, 1), 12)]:
        assert host.image_mip_levels(w, h) == want
    hz = host.hiz_layout(4096, 4096)
    assert (hz.width, hz.height, hz.levels) == (2048, 2048, 12)
    assert hz.total_texels == sum((2048 >> l) ** 2 for l in range(12))  # 22.4 MB pyramid of SURVEY §8(a) a15
    hz = host.hiz_layout(1920, 1080)
    assert (hz.width, hz.height, hz.levels) == (1024, 1024, 11)
    hz = host.hiz_layout(4096, 600)
    assert (hz.width, hz.height, hz.levels) == (2048, 512, 12)
    assert hz.level_size(10) == (2, 1) and hz.level_size(11) == (1, 1)


def test_pcg32_known_answer():
    """PCG32 (XSH RR) known-answer: O'Neill's pcg32-demo seeds (42, 54) -> first outputs 0xa15c02b7 0x7b47f409 ...
    niagara.cpp:460-469 is that generator; nvc_host_random_draws must consume it identically."""

    def pcg(state, inc):
        while True:
            old = state
            state = (old * 6364136223846793005 + (inc | 1)) & ((1 << 64) - 1)
            xs = (((old >> 18) ^ old) >> 27) & 0xFFFFFFFF
            rot = old >> 59
            yield ((xs >> rot) | (xs << ((32 - rot) & 31))) & 0xFFFFFFFF

    # pcg32_srandom_r(42, 54)
    inc = (54 << 1) | 1
    state = 0
    state = (state * 6364136223846793005 + inc) & ((1 << 64) - 1)
    state = (state + 42) & ((1 << 64) - 1)
    state = (state * 6364136223846793005 + inc) & ((1 << 64) - 1)
    g = pcg(state, inc)
    assert [next(g) for _ in range(6)] == [0xA15C02B7, 0x7B47F409, 0xBA1D3330, 0x83D2F293, 0xBFA4784B, 0xCBED606E]

    # the reference's stream: PCG32_INITIALIZER inc, state = 0x42; first value feeds meshIndex, next three position
    g = pcg(0x42, 0xDA3E39CB94B95BDB)
    first = [next(g) for _ in range(4)]
    d = host.random_draws(1, 1000003)
    assert d["meshIndex"][0] == first[0] % 1000003
    for k in range(3):
        want = np.float32(np.float32(np.float32(first[1 + k] / float(1 << 32)) * np.float32(300)) * np.float32(2)) - np.float32(300)
        assert d["position"][0][k] == want


def _read_host_golden(golden_dir):
    raw = open(os.path.join(golden_dir, "host_golden.nvch"), "rb").read()
    h = np.frombuffer(raw, "<u4", 8)
    assert h[0] == 0x4843564E and h[1] == 1
    na, ma, nb, mb, ncam = (int(x) for x in h[2:7])
    off = 32
    a = np.frombuffer(raw, layout.MESHDRAW_DTYPE, na, off)
    off += na * 48
    b = np.frombuffer(raw, layout.MESHDRAW_DTYPE, nb, off)
    off += nb * 48
    cam_dt = np.dtype([("pos", "<f4", 3), ("q", "<f4", 4), ("fovY", "<f4"), ("znear", "<f4"), ("w", "<u4"), ("h", "<u4"), ("drawCount", "<u4"), ("lodStep", "<u4")])
    cams = []
    for _ in range(ncam):
        c = np.frombuffer(raw, cam_dt, 1, off)[0]
        off += cam_dt.itemsize
        g = np.frombuffer(raw, layout.CULLDATA_DTYPE, 1, off)[0]
        off += 144
        cams.append((c, g))
    return (a, ma), (b, mb), cams


def test_random_scene_matches_reference_recipe(golden_dir):
    """Golden: niagara.cpp:969-998 executed with the reference's glm (oracle/refscene/host_golden.cpp)."""
    (a, ma), (b, mb), _ = _read_host_golden(golden_dir)
    assert host.random_draws(len(a), ma).tobytes() == a.tobytes()
    assert host.random_draws(len(b), mb).tobytes() == b.tobytes()


def test_cull_data_matches_glm(golden_dir):
    """Golden: niagara.cpp:1487-1516 executed with glm; bit-exact including signed zeros."""
    _, _, cams = _read_host_golden(golden_dir)
    assert len(cams) >= 4
    for c, g in cams:
        cam = host.make_camera(tuple(c["pos"]), tuple(c["q"]), float(c["fovY"]), float(c["znear"]))
        cd = host.cull_data(cam, int(c["w"]), int(c["h"]), int(c["drawCount"]), debug_lod_step=int(c["lodStep"]))
        assert bytes(cd)[:136] == g.tobytes()[:136]


def test_visibility_offsets(golden_dir):
    meshes, meshlets, _ = layout.load_nvcg(os.path.join(golden_dir, "kitten_pirate.nvcg"))
    draws = host.random_draws(1000, len(meshes))
    draws["postPass"][7] = 1
    total, mask = host.visibility_offsets(draws, meshes)
    per = np.array([meshes["lods"]["meshletCount"][m][: meshes["lodCount"][m]].max() for m in range(len(meshes))])
    want = np.concatenate([[0], np.cumsum(per[draws["meshIndex"]])])
    assert np.array_equal(draws["meshletVisibilityOffset"], want[:-1]) and total == want[-1] and mask == 3


def test_pass_data_wiring():
    """niagara.cpp:1547-1550 vs 1595-1596: only the drawcull pass data gets clusterBackfaceEnabled (SURVEY F8)."""
    cd = host.cull_data(host.make_camera(), 1024, 768, 10)
    l = lib.load_library()
    out = layout.CullData()
    l.nvc_host_pass_data(ctypes.byref(cd), 1, 0, ctypes.byref(out))
    assert out.clusterBackfaceEnabled == 1 and out.postPass == 0
    l.nvc_host_pass_data(ctypes.byref(cd), 1, 1, ctypes.byref(out))
    assert out.clusterBackfaceEnabled == 0 and out.postPass == 1
    l.nvc_host_pass_data(ctypes.byref(cd), 0, 0, ctypes.byref(out))
    assert out.clusterBackfaceEnabled == 0


def test_product_path_fails_loudly_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    l = lib.load_library()
    ctx = ctypes.c_void_p()
    assert l.nvc_create(0, None, ctypes.byref(ctx)) == -3  # NVC_ERROR_NO_DEVICE, no CPU fallback
    from niagara_b200.path import VisibilityPath

    meshes, meshlets, _ = layout.load_nvcg(os.path.join(ROOT, "tests", "golden", "kitten.nvcg"))
    with pytest.raises(RuntimeError):
        VisibilityPath(meshes, meshlets, host.random_draws(4, 1), 64, 64)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "niagara_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "liboracle" not in src and "oracle_lib" not in src and "orc_" not in src, f


def test_cull_data_against_glm_on_random_cameras(request):
    """Property test of nvc_host_cull_data (glm-free: quaternion -> matrix, general 4x4 inverse, Z flip, projection, frustum
    planes, lodTarget, pyramid size) against the same computation through glm (oracle/refscene/host_golden.h): 3000 random
    cameras incl. non-unit and axis-aligned quaternions, extreme positions, fields of view and aspect ratios — all 136 bytes.
    Without glm its results are the pinned ones (reference_pins), one pin per 300 cameras."""
    import ctypes

    import reference_pins
    from test_scene_cache import load_glm

    glm = load_glm()
    if glm is not None:
        glm.cull_data_ref.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_float, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p]
    rng = np.random.default_rng(31)
    want = np.zeros(144, np.uint8)
    chunk = []
    with reference_pins.pinned(request, glm is not None):
        for i in range(3000):
            _random_camera_case(glm, rng, i, want, chunk)
            if len(chunk) == 300:
                reference_pins.check("cameras %d-%d" % (i - 299, i), np.concatenate(chunk))
                chunk.clear()


def _random_camera_case(glm, rng, i, want, chunk):
    pos = (rng.standard_normal(3) * 10.0 ** rng.integers(-2, 5)).astype(np.float32)
    q = rng.standard_normal(4)
    kind = i % 5
    if kind == 0:
        q /= np.linalg.norm(q)
    elif kind == 1:
        q = np.eye(4)[rng.integers(0, 4)] * rng.choice([-1.0, 1.0])  # axis aligned: exact zeros and signed zeros in the matrix
    elif kind == 2:
        q = q / np.linalg.norm(q) * rng.uniform(0.5, 2.0)  # not normalised
    elif kind == 3:
        q = np.array([0, 0, 0, 1.0]) + rng.standard_normal(4) * 1e-4
    q = q.astype(np.float32)
    fov = float(np.float32(rng.uniform(0.05, 3.0)))
    znear = float(np.float32(10.0 ** rng.uniform(-3, 1)))
    w, h = int(rng.integers(1, 8192)), int(rng.integers(1, 8192))
    n, step = int(rng.integers(0, 1 << 31)), int(rng.integers(0, 8))
    cam = host.make_camera(tuple(float(x) for x in pos), tuple(float(x) for x in q), fov, znear)
    cd = host.cull_data(cam, w, h, n, debug_lod_step=step)
    if glm is None:
        chunk.append(np.frombuffer(bytes(cd)[:136], np.uint8))
        return
    glm.cull_data_ref(pos.ctypes.data, q.ctypes.data, fov, znear, w, h, n, step, want.ctypes.data)
    assert bytes(cd)[:136] == want.tobytes()[:136], (i, kind, pos, q, fov, znear, w, h)
    chunk.append(want[:136].copy())
