"""CPU-only: the scene-cache reader (nvc_scene_cache_*, SURVEY §8(f) N2) and the keyframe evaluation
(nvc_host_animate, N3) against fixtures written by the REFERENCE's own code — importer, saveSceneCache, loadSceneCache,
glm (tests/golden/make_scene_cache_fixtures.py, oracle/refscene/write_cache.cpp)."""
import ctypes
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

from niagara_b200 import host, layout, scene_cache
from niagara_b200.lib import NvcError, load_library

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def meaningful_bytes(meshlets, words):
    """uint8 mask over meshletdata: 1 for the reference words / triangle bytes a meshlet owns, 0 for alignment padding
    (the odd uint16 of a short-ref list, the bytes after triangleCount * 3 — the reference's SIMD decoder leaves junk there)."""
    mask = np.zeros(words * 4, dtype=np.uint8)
    for m in meshlets:
        off, vc, tc = int(m["dataOffset"]) * 4, int(m["vertexCount"]), int(m["triangleCount"])
        if m["shortRefs"]:
            mask[off : off + vc * 2] = 1
            off += (vc + 1) // 2 * 4
        else:
            mask[off : off + vc * 4] = 1
            off += vc * 4
        mask[off : off + tc * 3] = 1
    return mask


def test_header_and_sections_of_reference_written_caches():
    raw = scene_cache.SceneCache(os.path.join(GOLDEN, "animated.raw.cache"))
    z = scene_cache.SceneCache(os.path.join(GOLDEN, "animated.z.cache"))
    for c, compressed in ((raw, 0), (z, 1)):
        h = c.header
        assert (h.magic, h.version, h.hashMeta, h.compressed, h.clrtMode) == (0x434E4353, 7, 0x0123456789ABCDEF, compressed, 0)
        assert (h.meshletMaxVertices, h.meshletMaxTriangles) == (64, 96)  # config.h MESH_MAXVTX / MESH_MAXTRI
        assert (h.meshCount, h.drawCount, h.animationCount, h.keyframeCount, h.materialCount) == (2, 14, 3, 18, 3)
        assert abs(h.camera.fovY - 0.9) < 1e-6 and abs(h.camera.znear - 0.1) < 1e-7  # fovY from the glTF camera (scene.cpp keeps its own znear)
        end = max(s.offset + s.stored_bytes for s in c.info.sections)
        assert end == c.size
    # every raw-stored section is byte-identical between the two files
    for name in ("meshlets", "meshes", "materials", "draws", "lights", "animations", "keyframes", "omm_descs"):
        assert np.array_equal(raw.section(name).view(np.uint8), z.section(name).view(np.uint8)), name
    assert z.section_info("meshletdata").compressed == 1 and z.section_info("meshletdata").stored_bytes < raw.section_info("meshletdata").stored_bytes
    assert z.section_info("vertices").stored_bytes == z.header.compressedVertexBytes
    assert len(raw.section("vertices")) == raw.header.vertexCount * 16


def test_vertex_and_index_codecs():
    """The vertex codec is lossless: decode(compressed cache) == the uncompressed cache's bytes.  The index codec keeps
    every triangle but rotates its corners, so the golden is the digest of what the reference's loadSceneCache returns."""
    want = json.load(open(os.path.join(GOLDEN, "scene_cache_expected.json")))
    raw = scene_cache.SceneCache(os.path.join(GOLDEN, "animated.raw.cache"))
    z = scene_cache.SceneCache(os.path.join(GOLDEN, "animated.z.cache"))
    assert np.array_equal(z.section("vertices"), raw.section("vertices")) and len(z.section("vertices")) == 722 * 16
    assert np.array_equal(z.section("meshletvtx0"), raw.section("meshletvtx0"))
    zi, ri = z.section("indices").reshape(-1, 3), raw.section("indices").reshape(-1, 3)
    assert hashlib.sha256(zi.tobytes()).hexdigest() == want["animated"]["indices_sha256"]
    assert ((zi == ri).all(1) | (np.roll(ri, 1, 1) == zi).all(1) | (np.roll(ri, 2, 1) == zi).all(1)).all() and not (zi == ri).all()
    k = scene_cache.SceneCache(os.path.join(GOLDEN, "kitten.z.cache"))
    assert hashlib.sha256(k.section("vertices").tobytes()).hexdigest() == want["kitten"]["vertices_sha256"]
    assert hashlib.sha256(k.section("indices").tobytes()).hexdigest() == want["kitten"]["indices_sha256"]
    # the decoded positions are the ones the cooked meshlets were built from (kitten_cook.npz)
    cook = np.load(os.path.join(GOLDEN, "kitten_cook.npz"))
    assert np.array_equal(k.section("vertices").view(np.uint16).reshape(-1, 8)[:, :3], cook["positions"])


def test_meshlet_codec_matches_reference_decoder():
    """decode(animated.z.cache) == what the reference's loadSceneCache produced; against the raw cache the vertex
    references are identical and every triangle is the same up to the rotation the codec applies when encoding."""
    z = scene_cache.SceneCache(os.path.join(GOLDEN, "animated.z.cache"))
    raw = scene_cache.SceneCache(os.path.join(GOLDEN, "animated.raw.cache"))
    ml = z.section("meshlets")
    got = z.section("meshletdata")
    ref = np.fromfile(os.path.join(GOLDEN, "animated.z.meshletdata"), dtype="<u4")
    mask = meaningful_bytes(ml, len(ref))
    assert mask.sum() > 8000
    assert np.array_equal(got.view(np.uint8) * mask, ref.view(np.uint8) * mask)
    orig = raw.section("meshletdata")
    rotated = 0
    for m in ml:
        off, vc, tc = int(m["dataOffset"]), int(m["vertexCount"]), int(m["triangleCount"])
        rw = (vc + 1) // 2 if m["shortRefs"] else vc
        refs_a = orig[off : off + rw].view(np.uint16 if m["shortRefs"] else np.uint32)[:vc]
        refs_b = got[off : off + rw].view(np.uint16 if m["shortRefs"] else np.uint32)[:vc]
        assert np.array_equal(refs_a, refs_b)
        ta = orig[off + rw : off + rw + (tc * 3 + 3) // 4].view(np.uint8)[: tc * 3].reshape(tc, 3)
        tb = got[off + rw : off + rw + (tc * 3 + 3) // 4].view(np.uint8)[: tc * 3].reshape(tc, 3)
        same = (ta == tb).all(1) | (np.roll(ta, 1, 1) == tb).all(1) | (np.roll(ta, 2, 1) == tb).all(1)
        assert same.all()
        rotated += int((~(ta == tb).all(1)).sum())
        assert tb.max() < vc
    assert rotated > 0


def test_kitten_cache_against_reference_geometry_and_digest():
    """data/kitten.obj through the reference's cache writer: Mesh[] / Meshlet[] equal the arrays dumped by the
    reference's scene.cpp (kitten.nvcg); 792 meshlet blocks decode to the digest of the reference decoder's output."""
    c = scene_cache.SceneCache(os.path.join(GOLDEN, "kitten.z.cache"))
    want = json.load(open(os.path.join(GOLDEN, "scene_cache_expected.json")))["kitten"]
    meshes, meshlets, _ = layout.load_nvcg(os.path.join(GOLDEN, "kitten.nvcg"))
    assert np.array_equal(c.section("meshes"), meshes) and np.array_equal(c.section("meshlets"), meshlets)
    assert (c.header.meshletCount, c.header.vertexCount, c.header.indexCount) == (want["meshlets"], want["vertices"], want["indices"])
    md = c.section("meshletdata")
    assert len(md) == want["meshletdata_words"]
    mask = meaningful_bytes(meshlets, len(md))
    assert hashlib.sha256((md.view(np.uint8) * mask).tobytes()).hexdigest() == want["meshletdata_sha256_masked"]


def test_fresh_reference_output_full_compare(tmp_path, request):
    """kitten.obj and pirate.glb (the glTF importer: several meshes and materials) through the reference's writer + loader:
    where the reference is present it runs now and its compressed caches must equal the stored ones; every section the
    product's decoders read from those caches equals what the reference's loader decodes (meshletdata, padding bytes
    masked; indices) and what its uncompressed cache holds (Meshlet[], vertices).  Elsewhere the reference's sections are
    the pinned ones (reference_pins)."""
    import reference_pins
    from refshader_lib import REFERENCE

    live = os.path.isdir(os.path.join(REFERENCE, "src"))
    if live:
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + REFERENCE], check=True)
    with reference_pins.pinned(request, live):
        for name, model, stored in (("kitten", "data/kitten.obj", "kitten.z.cache"), ("pirate_glb", "extern/meshoptimizer/demo/pirate.glb", "pirate_glb.z.cache")):
            c = scene_cache.SceneCache(os.path.join(GOLDEN, stored))
            md = c.section("meshletdata")
            ours = {"meshletdata": md.view(np.uint8) * meaningful_bytes(c.section("meshlets"), len(md)), "meshlets": c.section("meshlets"), "vertices": c.section("vertices"), "indices": c.section("indices").astype("<u4")}
            if live:
                prefix = str(tmp_path / name)
                subprocess.run([os.path.join(ROOT, "oracle", "_ref", "write_cache"), prefix, os.path.join(REFERENCE, model)], check=True, stdout=subprocess.DEVNULL)
                assert open(prefix + ".z.cache", "rb").read() == open(os.path.join(GOLDEN, stored), "rb").read(), name
                ref = np.fromfile(prefix + ".z.meshletdata", dtype="<u4")
                r = scene_cache.SceneCache(prefix + ".raw.cache")
                assert len(r.section("indices")) == r.header.indexCount
                want = {"meshletdata": ref.view(np.uint8) * meaningful_bytes(c.section("meshlets"), len(ref)), "meshlets": r.section("meshlets"), "vertices": r.section("vertices"), "indices": np.fromfile(prefix + ".z.indices", dtype="<u4")}
                for k in ours:
                    assert np.array_equal(ours[k], want[k]), (name, k)
            for k in ours:
                reference_pins.check("%s %s" % (name, k), want[k] if live else ours[k])


def test_corrupt_and_truncated_files_are_rejected(tmp_path):
    lib = load_library()
    data = bytearray(open(os.path.join(GOLDEN, "animated.z.cache"), "rb").read())
    info = layout.SceneCacheInfo()

    def parse(b):
        buf = (ctypes.c_char * len(b)).from_buffer_copy(bytes(b))
        return lib.nvc_scene_cache_parse(ctypes.addressof(buf), len(b), ctypes.byref(info)), buf

    assert parse(data)[0] == 0
    assert parse(data[:100])[0] == -7  # NVC_ERROR_CORRUPT: shorter than the header
    assert parse(data[:-1])[0] == -7 and parse(data + b"\0")[0] == -7
    bad = bytearray(data)
    bad[0] ^= 1
    assert parse(bad)[0] == -7
    bad = bytearray(data)
    bad[4] = 6  # version
    assert parse(bad)[0] == -6  # NVC_ERROR_UNSUPPORTED
    # flip bytes inside the compressed meshlet stream: parse may pass (sizes intact) but the decode must fail cleanly or
    # produce in-range output — never crash, never write outside dst
    status, buf = parse(data)
    rng = np.random.default_rng(3)
    for name in ("meshletdata", "vertices", "indices"):
        idx = layout.CACHE_SECTIONS.index(name)
        sec = info.sections[idx]
        offset, stored, decoded = int(sec.offset), int(sec.stored_bytes), int(sec.decoded_bytes)
        rejected = 0
        for trial in range(200):
            bad = bytearray(data)
            for _ in range(3):
                bad[offset + int(rng.integers(0, stored))] = int(rng.integers(0, 256))
            st, b2 = parse(bad)
            if st != 0:
                rejected += 1
                continue
            out = np.zeros(decoded + 64, dtype=np.uint8)
            out[-64:] = 0xAB
            st = lib.nvc_scene_cache_read(ctypes.addressof(b2), len(bad), ctypes.byref(info), idx, out.ctypes.data, decoded)
            assert st in (0, -6, -7), (name, st)
            rejected += st != 0
            assert (out[-64:] == 0xAB).all(), name
        assert rejected > 20, (name, rejected)
        # truncated streams (the section shortened by moving bytes out of it is caught by parse; here: zeroed tail)
        bad = bytearray(data)
        bad[offset + stored - 8 : offset + stored] = bytes(8)
        st, b2 = parse(bad)
        if st == 0:
            out = np.zeros(decoded, dtype=np.uint8)
            assert lib.nvc_scene_cache_read(ctypes.addressof(b2), len(bad), ctypes.byref(info), idx, out.ctypes.data, decoded) in (0, -6, -7)


def _load_nvca(path):
    raw = open(path, "rb").read()
    h = np.frombuffer(raw, dtype="<u4", count=8)
    assert h[0] == 0x4143564E and h[1] == 1
    na, nk, nd, nt = int(h[2]), int(h[3]), int(h[4]), int(h[5])
    off = 32
    anims = np.frombuffer(raw, dtype=layout.ANIMATION_DTYPE, count=na, offset=off).copy()
    off += na * 24
    keys = np.frombuffer(raw, dtype=layout.KEYFRAME_DTYPE, count=nk, offset=off).copy()
    off += nk * 32
    draws0 = np.frombuffer(raw, dtype=layout.MESHDRAW_DTYPE, count=nd, offset=off).copy()
    off += nd * 48
    frames = []
    for _ in range(nt):
        t = float(np.frombuffer(raw, dtype="<f8", count=1, offset=off)[0])
        off += 8
        frames.append((t, np.frombuffer(raw, dtype=layout.MESHDRAW_DTYPE, count=nd, offset=off).copy()))
        off += nd * 48
    assert off == len(raw)
    return anims, keys, draws0, frames


def test_animation_matches_glm_frame_loop():
    """nvc_host_animate == the reference's frame-loop update (glm::mix / glm::slerp), bit for bit, at 44 times: before
    the first keyframe, across wrap-arounds, exactly on keyframes, far in the future."""
    anims, keys, draws0, frames = _load_nvca(os.path.join(GOLDEN, "animated.nvca"))
    c = scene_cache.SceneCache(os.path.join(GOLDEN, "animated.z.cache"))
    assert np.array_equal(c.section("animations"), anims) and np.array_equal(c.section("keyframes"), keys) and np.array_equal(c.section("draws"), draws0)
    assert len(anims) == 3 and (anims["keyframeCount"] == 6).all() and (anims["drawIndex"] >= 0).all()
    draws = draws0.copy()
    moved = 0
    for t, want in frames:
        before = draws.copy()
        idx, val = host.animate(anims, keys, t, draws)
        assert np.array_equal(draws.view(np.uint8), want.view(np.uint8)), t
        changed = np.nonzero((before.view(np.uint8).reshape(len(draws), 48) != draws.view(np.uint8).reshape(len(draws), 48)).any(1))[0]
        assert set(changed) <= set(idx.tolist()) and np.array_equal(val, draws[idx])
        assert len(idx) in (0, 3)
        moved += len(idx)
    assert moved >= 3 * 40
    # unit quaternions stay unit (slerp), scale and position stay inside the keyframe hull
    q = draws["orientation"][anims["drawIndex"]]
    assert np.allclose(np.linalg.norm(q, axis=1), 1.0, atol=1e-5)


def test_animate_rejects_bad_tracks():
    anims = np.zeros(1, dtype=layout.ANIMATION_DTYPE)
    keys = np.zeros(2, dtype=layout.KEYFRAME_DTYPE)
    draws = np.zeros(2, dtype=layout.MESHDRAW_DTYPE)
    anims["period"] = 1.0
    anims["keyframeCount"] = 0
    with pytest.raises(NvcError):
        host.animate(anims, keys, 0.5, draws)
    anims["keyframeCount"] = 3  # past the end of keyframes[]
    with pytest.raises(NvcError):
        host.animate(anims, keys, 0.5, draws)
    anims["keyframeCount"] = 2
    anims["drawIndex"] = 5
    with pytest.raises(NvcError):
        host.animate(anims, keys, 0.5, draws)
    anims["drawIndex"] = -1  # light-only track: ignored
    idx, _ = host.animate(anims, keys, 0.5, draws)
    assert len(idx) == 0


def test_cache_scene_runs_through_the_oracle():
    """load_scene(cache) gives the path what it needs: two frames over the cache's own draws and camera, animated between them."""
    import oracle_lib

    s = scene_cache.load_scene(os.path.join(GOLDEN, "animated.z.cache"), screen=(640, 480))
    again = s.draws.copy()
    bits, _ = host.visibility_offsets(again, s.meshes)  # niagara.cpp:1003-1020 re-derived: same offsets as stored
    assert s.visibility_bits == bits and np.array_equal(again, s.draws)
    assert (s.draws["postPass"] == np.tile([0, 1], 7)).all()  # the BLEND material -> postPass 1 (scene.cpp:584-585)
    o = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *s.screen)
    o.set_visibility_bits(s.visibility_bits)
    cd = s.cull_data(occlusion=False, cluster_occlusion=False)
    o.frame(cd, s.depth, post_passes=True)
    first = o.dvb.copy()
    assert first.sum() > 0
    host.animate(s.animations, s.keyframes, 1.7, s.draws)
    o.draws[...] = s.draws
    o.frame(cd, s.depth, post_passes=True)


def test_cpp_host_example_reads_the_same(tmp_path):
    """examples/scene_cache_info.cpp (plain g++, host only): the C ABI used from C++ the way niagara's main() uses
    loadSceneCache and its animation block — same meshlet data digest and same animated transforms as through ctypes."""
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "examples"), "scene_cache_info"], check=True)
    path = os.path.join(GOLDEN, "animated.z.cache")
    out = subprocess.run([os.path.join(ROOT, "examples", "scene_cache_info"), path, "0.2", "1.7"], check=True, capture_output=True, text=True).stdout
    c = scene_cache.SceneCache(path)
    digest = 1469598103934665603
    for w in c.section("meshletdata").tolist():
        digest = ((digest ^ w) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    assert "meshletdata: ok, %d words, fnv %016x" % (c.header.meshletdataCount, digest) in out
    assert "t = 0.2: 0 draws move" in out
    draws = c.section("draws").copy()
    idx, val = host.animate(c.section("animations"), c.section("keyframes"), 1.7, draws)
    line = [l for l in out.splitlines() if l.startswith("t = 1.7")][0]
    assert line.startswith("t = 1.7: %d draws move" % len(idx))
    for i, v in zip(idx, val):
        assert "[%d] -> (%.9g %.9g %.9g) scale %.9g" % (i, v["position"][0], v["position"][1], v["position"][2], v["scale"]) in line


def test_decoders_under_address_and_ub_sanitizers(tmp_path):
    """tests/fuzz_scene_cache.cpp: the host decoders compiled from the product sources with ASan + UBSan, 3000 mutated
    caches (byte flips, truncations, edited counts): no invalid access, only the documented status codes."""
    exe = str(tmp_path / "fuzz_scene_cache")
    srcs = [os.path.join(ROOT, "tests", "fuzz_scene_cache.cpp"), os.path.join(ROOT, "niagara_b200", "csrc", "nvc_scene_cache.cpp"), os.path.join(ROOT, "niagara_b200", "csrc", "nvc_meshopt_decode.cpp")]
    build = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-o", exe] + srcs, capture_output=True, text=True)
    if build.returncode != 0 and "sanitize" in build.stderr:
        pytest.skip("this toolchain has no sanitizer runtime: " + build.stderr.splitlines()[0])
    assert build.returncode == 0, build.stderr
    for cache in ("animated.z.cache", "animated.raw.cache"):
        run = subprocess.run([exe, os.path.join(GOLDEN, cache), "1500"], capture_output=True, text=True)
        assert run.returncode == 0, run.stderr[-2000:]
        assert "mutations 1500" in run.stdout


def load_glm():
    """oracle/_ref/libanim_ref.so (glm of the reference, see oracle/refscene/anim_ref.cpp), or None where it is neither built
    nor buildable"""
    from refshader_lib import REFERENCE

    if os.path.isdir(os.path.join(REFERENCE, "src")):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + REFERENCE], check=True)
    so = os.path.join(ROOT, "oracle", "_ref", "libanim_ref.so")
    return ctypes.CDLL(so) if os.path.exists(so) else None


def test_animation_blend_against_glm_on_random_keyframes(request):
    """Property test of nvc_host_animate's blend against glm::mix / glm::slerp themselves (oracle/refscene/anim_ref.cpp):
    random unit and non-unit quaternions, nearly identical ones (glm's lerp shortcut), opposite ones (sign flip), exact 0 / 1
    and tiny blend factors — bit for bit.  Without glm its results are the pinned ones (reference_pins), one pin per factor."""
    import reference_pins

    glm = load_glm()
    with reference_pins.pinned(request, glm is not None):
        _animation_blend(glm)


def _animation_blend(glm):
    import reference_pins

    if glm is not None:
        glm.anim_ref_blend.argtypes = [ctypes.c_void_p, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_void_p, ctypes.c_float, ctypes.c_void_p]
    rng = np.random.default_rng(8)
    n = 4000
    keys = np.zeros(2 * n, dtype=layout.KEYFRAME_DTYPE)
    keys["translation"] = rng.uniform(-50, 50, (2 * n, 3)).astype(np.float32)
    keys["scale"] = rng.uniform(0.1, 5, 2 * n).astype(np.float32)
    q = rng.standard_normal((2 * n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[1::8] = q[0::8] + rng.standard_normal((len(q[0::8]), 4)) * 1e-5  # nearly the same rotation -> dot > 1 - eps
    q[3::8] = -q[2::8] + rng.standard_normal((len(q[2::8]), 4)) * 0.3  # far side of the sphere -> dot < 0
    q[5::8] = q[4::8]  # identical
    q[7::16] *= 3.0  # not normalised
    keys["rotation"] = q.astype(np.float32)
    anims = np.zeros(n, dtype=layout.ANIMATION_DTYPE)
    anims["drawIndex"] = np.arange(n)
    anims["lightIndex"] = -1
    anims["startTime"] = 0.0
    anims["period"] = 1.0
    anims["keyframeOffset"] = 2 * np.arange(n)
    anims["keyframeCount"] = 2
    out = np.zeros(8, np.float32)
    for t in (0.0, 1.0 / 3.0, 0.5, 0.999999, 1e-7, 0.25):
        draws = np.zeros(n, dtype=layout.MESHDRAW_DTYPE)
        idx, val = host.animate(anims, keys, t, draws)  # index = t in [0, 1): keyframe 0 -> 1, blend factor float(t)
        assert len(idx) == n
        a = np.float32(t - np.floor(t))
        got = np.concatenate([draws["position"], draws["scale"][:, None], draws["orientation"]], 1).astype(np.float32)
        if glm is None:
            reference_pins.check("t = %r" % t, got)
            continue
        want = np.zeros_like(got)
        for i in range(0, n, 1):
            k0, k1 = keys[2 * i], keys[2 * i + 1]
            glm.anim_ref_blend(k0["translation"].ctypes.data, float(k0["scale"]), k0["rotation"].ctypes.data, k1["translation"].ctypes.data, float(k1["scale"]), k1["rotation"].ctypes.data, float(a), out.ctypes.data)
            want[i] = out
            same = (got[i].view(np.uint32) == out.view(np.uint32)) | (np.isnan(got[i]) & np.isnan(out))
            assert same.all(), (t, i, got[i], out)
        reference_pins.check("t = %r" % t, want)
