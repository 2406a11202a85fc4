"""CPU-only: the oracle against the reference's OWN shaders executed on the host (oracle/refshader: the GLSL text of
src/shaders/*.glsl compiled by g++ through a GLSL shim — see oracle/refshader/glsl_shim.h for what the shim has to
assume).  This pins the oracle to the reference's source text instead of to our reading of it: every pass runs in
lock step on both sides from identical inputs, outputs are compared bit for bit (as sets where the GLSL's atomics
make the order arbitrary)."""
import ctypes
import os

import numpy as np
import pytest

import oracle_lib
import reference_pins
import refshader_lib
from niagara_b200 import host, layout, scenes

SOURCES = ["drawcull.comp.glsl", "tasksubmit.comp.glsl", "clustercull.comp.glsl", "clustersubmit.comp.glsl", "depthreduce.comp.glsl", "meshlet.task.glsl", "meshlet.mesh.glsl", "mesh.vert.glsl"]


@pytest.fixture(autouse=True)
def _reference_pins(request):
    with reference_pins.pinned(request, refshader_lib.available()):
        yield

F = np.float32
SPECIAL = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-38, 1.0, -1.0, 0.5, 2.0, 3.4e38, -3.4e38, np.inf, -np.inf, np.nan], dtype=np.float32)


def _mixed(rng, n, scale):
    v = (rng.standard_normal(n) * scale).astype(np.float32)
    idx = rng.integers(0, n, n // 25)
    v[idx] = SPECIAL[rng.integers(0, len(SPECIAL), len(idx))]
    return v


def _bits_equal(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    nan = np.isnan(a) & np.isnan(b)
    return np.array_equal(a.view(np.uint32)[~nan], b.view(np.uint32)[~nan]) and np.array_equal(np.isnan(a), np.isnan(b))


def test_library_is_built_from_the_reference_shaders():
    """Where the library exists: it was generated from exactly these shader files.  Without it there is no library to ask;
    what is left to check is the provenance of the pins, whose recorded entry for this test is the digest of the file names
    the library reported when they were recorded, so it must equal the digest of this list."""
    names = refshader_lib.load().rs_sources().decode().split() if refshader_lib.available() else SOURCES
    assert names == SOURCES
    reference_pins.check("shader files", np.frombuffer(" ".join(names).encode(), np.uint8))


def test_math_h_functions_random():
    """math.h:1-49 as written (projectSphere, getOcclusionMip, coneCull, rotateQuat) == the oracle's restatement,
    on random inputs with zeros / denormals / huge / inf / NaN mixed in and power-of-two box sizes."""
    rs, orc = (refshader_lib.load() if refshader_lib.available() else None), oracle_lib.load()
    rng = np.random.default_rng(7)
    n = 20000
    cx, cy, cz, r = _mixed(rng, n, 30), _mixed(rng, n, 30), np.abs(_mixed(rng, n, 60)), np.abs(_mixed(rng, n, 3))
    a = np.zeros(4, np.float32)
    ok, aabb = np.zeros(n, np.int32), np.zeros((n, 4), np.float32)  # what the reference computes (the oracle's values where it is absent)
    for i in range(n):
        c = np.array([cx[i], cy[i], cz[i]], np.float32)
        ok[i] = orc.orc_project_sphere(c.ctypes.data, float(r[i]), 0.1, float(F(1.07)), float(F(1.43)), aabb[i].ctypes.data)
        if rs:
            ok_r = rs.rs_project_sphere(c.ctypes.data, float(r[i]), 0.1, float(F(1.07)), float(F(1.43)), a.ctypes.data)
            assert ok_r == ok[i], i
            if ok_r:
                assert _bits_equal(a, aabb[i]), (i, a, aabb[i])
    aabb[ok == 0] = 0
    reference_pins.check("projectSphere", ok, aabb)

    x0, y0 = _mixed(rng, n, 0.6), _mixed(rng, n, 0.6)
    w, h = np.abs(_mixed(rng, n, 0.05)), np.abs(_mixed(rng, n, 0.05))
    k = rng.integers(0, n, n // 5)  # exactly / almost a power-of-two number of texels wide: the ceil(log2) boundary
    w[k] = (2.0 ** rng.integers(-3, 11, len(k)) / 2048.0).astype(np.float32)
    k2 = k[: len(k) // 2]
    w[k2] = np.nextafter(w[k2], np.where(rng.integers(0, 2, len(k2)) == 1, F(np.inf), F(-np.inf)).astype(np.float32))
    x0[k] = 0
    with np.errstate(all="ignore"):
        x1, y1 = (x0 + w).astype(np.float32), (y0 + h).astype(np.float32)
    mip = np.zeros(n, np.float32)
    for i in range(n):
        box = np.array([x0[i], y0[i], x1[i], y1[i]], np.float32)
        mip[i] = lo = orc.orc_occlusion_mip(box.ctypes.data, 2048.0, 1024.0)
        if rs:
            lr = rs.rs_occlusion_mip(box.ctypes.data, 2048.0, 1024.0)
            # an infinite box: the GLSL yields +inf, the oracle a huge finite level; the sampler clamps both to the last mip
            assert lr == lo or (lr >= 1e8 and lo >= 1e8), (i, lr, lo, box)
    reference_pins.check("getOcclusionMip, levels >= 1e8 as 1e8", np.where(mip >= 1e8, F(1e8), mip))

    ax = np.stack([_mixed(rng, n, 1), _mixed(rng, n, 1), _mixed(rng, n, 1)], 1)
    q = rng.standard_normal((n, 4)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True).astype(np.float32)
    cut = rng.uniform(-1, 1, n).astype(np.float32)
    cone, rot = np.zeros(n // 4, np.int32), np.zeros((n // 4, 4), np.float32)
    for j, i in enumerate(range(0, n, 4)):
        c = np.array([cx[i], cy[i], cz[i]], np.float32)
        cone[j] = orc.orc_cone_cull(c.ctypes.data, float(r[i]), ax[i].ctypes.data, float(cut[i]))
        orc.orc_rotate_quat(ax[i].ctypes.data, q[i].ctypes.data, rot[j].ctypes.data)
        if rs:
            assert rs.rs_cone_cull(c.ctypes.data, float(r[i]), ax[i].ctypes.data, float(cut[i])) == cone[j], i
            rs.rs_rotate_quat(ax[i].ctypes.data, q[i].ctypes.data, a.ctypes.data)
            assert _bits_equal(a[:3], rot[j, :3]), i
    reference_pins.check("coneCull, rotateQuat", cone, rot[:, :3])


@pytest.mark.parametrize("size", [(64, 64), (100, 60), (30, 17), (129, 257), (2, 2), (1, 1), (256, 8), (640, 480), (1000, 3)])
def test_depthreduce_chain(size):
    """depthreduce.comp.glsl dispatched mip by mip as niagara.cpp:1703-1733 does == orc_depth_pyramid, every texel."""
    w, h = size
    rng = np.random.default_rng(w * 1000 + h)
    depth = rng.random((h, w), dtype=np.float32)
    depth[rng.random((h, w)) < 0.2] = 0.0
    paths = []
    for cls in (oracle_lib.OraclePath, refshader_lib.RefShaderPath):
        p = cls(np.zeros(1, layout.MESH_DTYPE), np.zeros(1, layout.MESHLET_DTYPE), np.zeros(1, layout.MESHDRAW_DTYPE), w, h, threads=3)
        p.pyramid(depth)
        paths.append(p)
    assert np.array_equal(paths[0].pyramid_texels, paths[1].pyramid_texels)


def _sync(dst, src):
    """Makes dst's buffers identical to src's (inputs of the next pass)."""
    for name in ("dvb", "dcb", "dccb", "cib", "ccb", "mvb", "pyramid_texels"):
        getattr(dst, name)[...] = getattr(src, name)


def _compare_cull(o, r, task, n_draws):
    assert np.array_equal(o.dvb, r.dvb)
    if task:
        assert np.array_equal(o.dccb, r.dccb)
        total = int(o.dccb[1]) * 64
        oc, rc = o.read_task_commands(total), r.read_task_commands(total)
        count = min(int(o.dccb[0]), total)
        assert np.array_equal(oracle_lib.sorted_commands(oc[:count]), oracle_lib.sorted_commands(rc[:count]))
        assert np.array_equal(oc[count:], rc[count:])  # tasksubmit's zero padding
        # commands of one draw are contiguous and ordered (drawcull.comp.glsl:132-139)
        d = rc["drawId"][:count]
        assert len(np.unique(d)) == (np.r_[True, d[1:] != d[:-1]].sum() if count else 0)
    else:
        assert o.dccb[0] == r.dccb[0]
        count = int(o.dccb[0])
        assert np.array_equal(oracle_lib.sorted_commands(o.read_draw_commands(count)), oracle_lib.sorted_commands(r.read_draw_commands(count)))


def _compare_clusters(o, r):
    assert np.array_equal(o.ccb, r.ccb)
    assert np.array_equal(o.mvb, r.mvb)
    count = int(o.ccb[0])
    # same dcb on both sides, so the raw indices (commandId | mgi << 24) must agree as sets
    assert np.array_equal(np.sort(o.read_cluster_indices(count)), np.sort(r.read_cluster_indices(count)))
    pad = (count + 255) // 256 * 256
    assert (r.cib[count:pad] == 0xFFFFFFFF).all() and np.array_equal(o.cib[count:pad], r.cib[count:pad])


def _lockstep(s, cd, frames=2, task=True, threads=4, post_passes=False, cluster_backface=True, history=True):
    o = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *s.screen, mesh_shading=task)
    r = refshader_lib.RefShaderPath(s.meshes, s.meshlets, s.draws, *s.screen, mesh_shading=task, threads=threads)
    for p in (o, r):
        p.set_visibility_bits(s.visibility_bits)
    if history:
        o.dvb[: len(s.draws) // 2] = 1
        o.mvb[:] = np.random.default_rng(5).integers(0, 1 << 32, len(o.mvb), dtype=np.uint64).astype(np.uint32)
    emitted = 0
    for _ in range(frames):
        passes = [(False, 0), (True, 0)] + ([(True, 1)] if post_passes else [])
        for late, post in passes:
            if late and post == 0:
                _sync(r, o)
                o.pyramid(s.depth)
                r.pyramid(s.depth)
                assert np.array_equal(o.pyramid_texels, r.pyramid_texels)
            _sync(r, o)
            o.cull(cd, late, post_pass=post)
            r.cull(cd, late, post_pass=post)
            _compare_cull(o, r, task, len(s.draws))
            if task:
                _sync(r, o)
                o.render_clusters(cd, late, post_pass=post, cluster_backface=cluster_backface)
                r.render_clusters(cd, late, post_pass=post, cluster_backface=cluster_backface)
                _compare_clusters(o, r)
                emitted += int(o.ccb[0])
            else:
                emitted += int(o.dccb[0])
    return emitted


def _kitten_pirate(golden_dir, n=3000, screen=(640, 480)):
    return scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), n, screen=screen)


@pytest.mark.parametrize("toggles", [dict(), dict(lod=False), dict(culling=False), dict(occlusion=False), dict(cluster_occlusion=False)])
def test_frames_in_lockstep_with_reference_shaders(golden_dir, toggles):
    s = _kitten_pirate(golden_dir)
    assert _lockstep(s, s.cull_data(**toggles)) > 1000


def test_reference_wiring_of_cluster_backface(golden_dir):
    """cluster_backface=None: clusterBackfaceEnabled exactly as the render lambda passes it (niagara.cpp:1595-1596)."""
    s = _kitten_pirate(golden_dir, n=2000)
    assert _lockstep(s, s.cull_data(), cluster_backface=None) > 1000
    assert _lockstep(s, s.cull_data(), cluster_backface=False) > 1000


def test_draw_path_and_post_pass(golden_dir):
    """TASK=false specialisation (MeshDrawCommand output) and the postPass=1 variant."""
    s = _kitten_pirate(golden_dir, n=4000)
    s.draws["postPass"][::7] = 1
    assert _lockstep(s, s.cull_data(), task=False, post_passes=True) > 300
    assert _lockstep(s, s.cull_data(), task=True, post_passes=True) > 500


def test_moving_camera_cold_start(golden_dir):
    s = _kitten_pirate(golden_dir, n=5000, screen=(800, 600))
    o = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *s.screen)
    r = refshader_lib.RefShaderPath(s.meshes, s.meshlets, s.draws, *s.screen, threads=6)
    for p in (o, r):
        p.set_visibility_bits(s.visibility_bits)
    cams = [host.make_camera((0, 0, 0)), host.make_camera((12, -4, 9), host.quat_from_axis_angle((0, 1, 0), 0.35)), host.make_camera((25, 3, -14), host.quat_from_axis_angle((0.1, 1, 0), 0.9))]
    for f in range(3):
        s.camera = cams[f]
        cd = s.cull_data()
        o.frame(cd, s.depth, cluster_backface=True)
        r.frame(cd, s.depth, cluster_backface=True)
        # free-running (no per-pass sync): command order differs, so compare what the consumers decode
        assert np.array_equal(o.dvb, r.dvb) and np.array_equal(o.mvb, r.mvb)
        assert np.array_equal(o.dccb, r.dccb) and np.array_equal(o.ccb, r.ccb)
        oc, rc = o.read_task_commands(int(o.dccb[1]) * 64), r.read_task_commands(int(r.dccb[1]) * 64)
        assert np.array_equal(oracle_lib.cluster_pairs(o.read_cluster_indices(int(o.ccb[0])), oc), oracle_lib.cluster_pairs(r.read_cluster_indices(int(r.ccb[0])), rc))


def test_synthetic_scene_with_many_lods_and_groups():
    """meshes with up to 8 LODs and several task groups per draw (taskCount < 64 tails, padded commands)."""
    s = scenes.config2_scene(draw_count=20000, num_meshes=64, screen=(512, 512))
    assert _lockstep(s, s.cull_data(), frames=2) > 100


def test_task_shader_payloads(golden_dir):
    """meshlet.task.glsl (shared counter + barrier, run as fibers) == orc_taskcull: same survivors per command; the
    oracle's payload order (ascending lane) is the order a serial execution of the workgroup produces."""
    s = _kitten_pirate(golden_dir, n=3000)
    cd = s.cull_data()
    o = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *s.screen)
    r = refshader_lib.RefShaderPath(s.meshes, s.meshlets, s.draws, *s.screen, threads=4)
    for p in (o, r):
        p.set_visibility_bits(s.visibility_bits)
    total_emitted = 0
    for f in range(2):
        for late in (False, True):
            if late:
                o.pyramid(s.depth)
            o.cull(cd, late)
            _sync(r, o)
            n = int(o.dccb[1]) * 64
            op, oe = np.zeros((max(n, 1), 64), np.uint32), np.zeros(max(n, 1), np.uint32)
            rp, re_ = np.full((max(n, 1), 64), 0xDEADBEEF, np.uint32), np.zeros(max(n, 1), np.uint32)
            o.task_shading(cd, late, op, oe, cluster_backface=True)
            r.task_shading(cd, late, rp, re_, cluster_backface=True)
            assert np.array_equal(oe, re_)
            for i in range(n):
                assert np.array_equal(op[i, : oe[i]], rp[i, : oe[i]]), i
            assert np.array_equal(o.mvb, r.mvb)
            total_emitted += int(oe.sum())
    assert total_emitted > 1000


def test_tiny_and_empty_inputs(golden_dir):
    s = _kitten_pirate(golden_dir, n=1)
    _lockstep(s, s.cull_data(), history=False)
    s3 = _kitten_pirate(golden_dir, n=3)
    cd = s3.cull_data()
    cd.drawCount = 0  # nothing dispatched: counters zero, padding written
    _lockstep(s3, cd, history=False)


def test_hostile_inputs_against_reference_shaders(golden_dir):
    """The fuzz scene of the GPU suite (NaN / inf / zero / huge transforms, fp16 specials in meshlet bounds, extreme cone
    bytes, inf and denormal depth texels): the oracle must follow the reference's shader text there too.  Where the shim
    has to pick a behaviour GLSL/Vulkan leave undefined (NaN texture coordinates, NaN in min/max) it picks what the
    oracle and the CUDA path document; everything else is the shader's own arithmetic."""
    import warnings

    import hostile

    s = hostile.hostile_scene(golden_dir, 12000)
    cams = [host.make_camera((0, 0, 0)), host.make_camera((5, 2, -3), host.quat_from_axis_angle((0.3, 1, 0), 0.9))]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        total = 0
        for cam in cams:
            s.camera = cam
            total += _lockstep(s, s.cull_data(), frames=2)
        # culling off: draws with NaN / inf centres pass the frustum stage and reach projectSphere and the sampler
        total += _lockstep(s, s.cull_data(culling=False), frames=2)
    assert total > 1000


def test_full_size_c4_against_reference_shaders():
    """BASELINE configs[3] at FULL size (1M draws x 10 unique meshlets, 4096^2 depth): two frames in lock step, the oracle
    (the checker of the GPU suite's full-size run) against the reference's own shaders — 28M meshlet tests, bit for bit."""
    s = scenes.config4_scene()
    threads = os.cpu_count() or 8
    o = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *s.screen, threads=threads, cmd_capacity=2 * len(s.draws))
    r = refshader_lib.RefShaderPath(s.meshes, s.meshlets, s.draws, *s.screen, threads=threads, cmd_capacity=2 * len(s.draws))
    for p in (o, r):
        p.set_visibility_bits(s.visibility_bits)
    cd = s.cull_data()
    tested = 0
    for f in range(2):
        for late in (False, True):
            if late:
                o.pyramid(s.depth)
                r.pyramid(s.depth)
                assert np.array_equal(o.pyramid_texels, r.pyramid_texels)
            _sync(r, o)
            o.cull(cd, late)
            r.cull(cd, late)
            assert np.array_equal(o.dvb, r.dvb) and np.array_equal(o.dccb, r.dccb)
            n = int(o.dccb[1]) * 64
            assert np.array_equal(oracle_lib.sorted_commands(o.read_task_commands(n)), oracle_lib.sorted_commands(r.read_task_commands(n)))
            _sync(r, o)
            o.render_clusters(cd, late, cluster_backface=True)
            r.render_clusters(cd, late, cluster_backface=True)
            assert np.array_equal(o.ccb, r.ccb) and np.array_equal(o.mvb, r.mvb)
            count = int(o.ccb[0])
            assert np.array_equal(np.sort(o.read_cluster_indices(count)), np.sort(r.read_cluster_indices(count)))
            tested += int(o.read_task_commands(n)["taskCount"].sum())
    assert tested > 25_000_000
