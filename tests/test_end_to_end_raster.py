"""CPU-only end-to-end check on REAL geometry: the two-phase visibility path (oracle), the reference's own mesh shader
(meshlet.mesh.glsl compiled through oracle/refshader) as the consumer of cib / ccb / dcb, and a small rasteriser that
turns its output into the depth buffer the next pass culls against — no synthetic depth anywhere.

Properties checked every frame, with a moving camera (SURVEY §3.3: why the two-phase scheme is correct):
  * the mesh stage decodes exactly what nvc_decode_clusters / the oracle say is in cib (N1), and nothing else;
  * no cluster is drawn twice (early and late sets are disjoint);
  * the image rendered from early + late clusters equals the brute-force image of ALL clusters of the selected LODs
    (nothing visible was culled), up to the reference's own fp16 rounding of meshlet bounds — the tolerance is stated;
  * every cluster owning a pixel of the brute-force image was emitted."""
import os

import numpy as np
import pytest

import emu_lib
import oracle_lib
import reference_pins
import refshader_lib
from niagara_b200 import host, layout, scenes

CULLERS = ["oracle", "reference-shaders", "cuda-kernels-emulated"]


def _culler(name):
    """who runs drawcull / clustercull / taskcull / the pyramid: our oracle, the reference's own shaders (oracle/refshader), or the
    PRODUCT's CUDA kernels under the CPU SIMT emulation (tests/cuda_emu)"""
    return {"oracle": oracle_lib.OraclePath, "reference-shaders": refshader_lib.RefShaderPath, "cuda-kernels-emulated": emu_lib.EmuPath}[name]



@pytest.fixture(autouse=True)
def _reference_pins(request):
    """where the reference's shaders cannot run, its passes, mesh and vertex stages are stood in for and held to its pinned outputs"""
    with reference_pins.pinned(request, refshader_lib.available()):
        yield


def _kitten_scene(golden_dir, n, screen):
    meshes, meshlets, _ = layout.load_nvcg(os.path.join(golden_dir, "kitten.nvcg"))
    z = np.load(os.path.join(golden_dir, "kitten_cook.npz"))
    positions, meshletdata = z["positions"], z["meshletdata"]
    vertices = np.zeros((len(positions), 8), dtype=np.uint16)
    vertices[:, :3] = positions
    rng = np.random.default_rng(4)
    draws = np.zeros(n, dtype=layout.MESHDRAW_DTYPE)
    draws["position"] = np.stack([rng.uniform(-14, 14, n), rng.uniform(-9, 9, n), -rng.uniform(6, 60, n)], 1)  # the camera looks down -Z (niagara.cpp:1492).astype(np.float32)
    draws["scale"] = rng.uniform(1.5, 4.5, n).astype(np.float32)
    q = rng.standard_normal((n, 4))
    draws["orientation"] = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    bits, _ = host.visibility_offsets(draws, meshes)
    cam = host.make_camera()
    s = scenes.Scene("kitten-field", meshes, meshlets, draws, np.zeros((screen[1], screen[0]), np.float32), cam, screen, bits)
    return s, vertices.view(np.uint8).reshape(-1), meshletdata


def _all_clusters(cmds, count):
    """cib / ccb listing every (command, lane) of the first `count` task commands — the brute-force draw list."""
    live = np.nonzero(cmds["taskCount"][:count] > 0)[0]
    tc = cmds["taskCount"][live].astype(np.int64)
    cid = np.repeat(live, tc)
    lane = np.arange(int(tc.sum())) - np.repeat(np.cumsum(tc) - tc, tc)
    ci = (cid | (lane << 24)).astype(np.uint32)
    pad = (len(ci) + 255) // 256 * 256
    cib = np.full(max(pad, 256), 0xFFFFFFFF, np.uint32)
    cib[: len(ci)] = ci
    return cib, np.array([len(ci), 16, max(pad // 256, 0), 16], np.uint32), ci


@pytest.mark.parametrize("culler", CULLERS)
def test_two_phase_frames_on_rasterised_depth(golden_dir, culler):
    """culler = who runs drawcull / clustercull / depthreduce: our oracle, or the reference's own shaders."""
    screen = (512, 384)
    s, vertices, meshletdata = _kitten_scene(golden_dir, 300, screen)
    o = _culler(culler)(s.meshes, s.meshlets, s.draws, *screen, threads=8)
    o.set_visibility_bits(s.visibility_bits)
    # brute-force lister: the early drawcull with every draw marked visible and every test but LOD selection switched off
    gt = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *screen, threads=8)
    gt.set_visibility_bits(s.visibility_bits)
    cams = [
        host.make_camera((0, 0, 0)),
        host.make_camera((0, 0, 0)),
        host.make_camera((3.5, -1.0, 2.0), host.quat_from_axis_angle((0, 1, 0), 0.18)),
        host.make_camera((7.0, 1.5, 5.0), host.quat_from_axis_angle((0.1, 1, 0), 0.42)),
        host.make_camera((7.0, 1.5, 5.0), host.quat_from_axis_angle((0.1, 1, 0), 0.42)),
    ]
    late_added, mismatching_pixels, total_pixels, missed_owners, owners_total = 0, 0, 0, 0, 0
    for f, cam in enumerate(cams):
        s.camera = cam
        cd = s.cull_data()
        ms = refshader_lib.MeshStage(o, vertices, meshletdata, host.projection(cam, *screen))
        depth = np.zeros((screen[1], screen[0]), np.float32)  # reverse Z: cleared to 0 = infinitely far (niagara.cpp:1744)

        def draw_pass(late):
            o.cull(cd, late)
            o.render_clusters(cd, late)  # the reference's own wiring of clusterBackfaceEnabled
            n = int(o.ccb[0])
            rec, pos, tri = ms.run(cd)
            # N1: the reference's mesh shader sees exactly the clusters the decoder reports
            drec, dstats = o.decode_clusters()
            assert int(dstats[0]) == n and int(dstats[2]) == 0
            live = rec[:, 0] > 0
            assert live.sum() == n and np.array_equal(live, drec[:, 0] != 0xFFFFFFFF)
            assert np.array_equal(rec[live, 2], drec[live, 0]) and np.array_equal(rec[live, 0], drec[live, 2]) and np.array_equal(rec[live, 1], drec[live, 3])
            ms.rasterize(rec, pos, tri, depth)
            cmds = o.read_task_commands(int(o.dccb[1]) * 64)
            return oracle_lib.cluster_pairs(o.read_cluster_indices(n), cmds), cmds

        early, _ = draw_pass(False)
        o.pyramid(depth)
        late, cmds = draw_pass(True)
        assert len(np.intersect1d(early, late)) == 0
        late_added += len(late)

        # brute force: every meshlet of the LOD drawcull selects for every draw, no culling at all
        gt.dvb[:] = 1
        gt.cull(s.cull_data(culling=False, occlusion=False, cluster_occlusion=False), late=False)
        assert int(gt.dccb[0]) >= len(s.draws)
        all_cmds = gt.read_task_commands(int(gt.dccb[1]) * 64)
        cib, ccb, ci = _all_clusters(all_cmds, int(gt.dccb[0]))
        rec, pos, tri = ms.run(cd, cib=cib, ccb=ccb, dcb=gt.dcb)
        truth = np.zeros_like(depth)
        ms.rasterize(rec, pos, tri, truth)
        diff = truth != depth
        mismatching_pixels += int(diff.sum())
        total_pixels += diff.size
        assert (truth >= depth).all()  # the path can only lose pixels, never invent them
        # owners of the brute-force image must have been emitted
        own = ms.owners(rec, pos, tri, truth)
        owner_pairs = oracle_lib.cluster_pairs(ci[own[: len(ci)]], all_cmds)
        emitted = np.union1d(early, late)
        missed = ~np.isin(owner_pairs, emitted)
        missed_owners += int(missed.sum())
        owners_total += len(owner_pairs)
        print("frame %d: early %d late %d clusters, brute force %d; coverage %.2f; pixels differing %d; owners %d missed %d" % (f, len(early), len(late), len(ci), (truth > 0).mean(), int(diff.sum()), len(owner_pairs), int(missed.sum())))
        assert (truth > 0).mean() > 0.2, "the scene should cover a good part of the screen"
    assert late_added > 0 and owners_total > 5000
    # In general exactness is not guaranteed by the reference (meshlet spheres are stored rounded to nearest fp16,
    # scene.cpp:71-74, cones quantised to 8 bits); on this scene the result IS exact, and the run is deterministic.
    print("frames %d: %d/%d pixels differ from brute force, %d/%d pixel-owning clusters not emitted" % (len(cams), mismatching_pixels, total_pixels, missed_owners, owners_total))
    assert mismatching_pixels == 0 and missed_owners == 0

    # sensitivity of the check itself: cull against a vertically flipped depth (the wrong viewport convention) and the late
    # pass rejects clusters that own pixels
    s.camera = cams[-1]
    cd = s.cull_data()
    o.pyramid(np.ascontiguousarray(truth[::-1]))
    o.cull(cd, True)
    o.render_clusters(cd, True)
    cmds = o.read_task_commands(int(o.dccb[1]) * 64)
    live = cmds[cmds["taskCount"] > 0]
    rejected = 0
    for c in live:
        mvi = int(c["meshletVisibilityOffset"]) + np.arange(int(c["taskCount"]))
        bits = (o.mvb[mvi >> 5] >> (mvi & 31).astype(np.uint32)) & 1
        pairs = (np.uint64(c["drawId"]) << np.uint64(32)) | (int(c["taskOffset"]) + np.nonzero(bits == 0)[0]).astype(np.uint64)
        rejected += int(np.isin(pairs, owner_pairs).sum())
    assert rejected > 20


@pytest.mark.parametrize("culler", CULLERS)
def test_task_shading_mode_on_rasterised_depth(golden_dir, culler):
    """The other submission mode (niagara.cpp:1666-1679): drawcull -> meshlet.task (payload + emit count per command, the
    contract of nvc_taskcull) -> the reference's mesh shader with TASK = true reading the payloads.  Same closed loop, same
    properties: disjoint early / late sets, image == brute force, every pixel owner emitted."""
    screen = (512, 384)
    s, vertices, meshletdata = _kitten_scene(golden_dir, 200, screen)
    o = _culler(culler)(s.meshes, s.meshlets, s.draws, *screen, threads=8)
    o.set_visibility_bits(s.visibility_bits)
    gt = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *screen, threads=8)
    gt.set_visibility_bits(s.visibility_bits)
    cams = [host.make_camera((0, 0, 0)), host.make_camera((0, 0, 0)), host.make_camera((4.0, 0.5, 3.0), host.quat_from_axis_angle((0, 1, 0), 0.25)), host.make_camera((4.0, 0.5, 3.0), host.quat_from_axis_angle((0, 1, 0), 0.25))]
    owners_total, late_total = 0, 0
    for cam in cams:
        s.camera = cam
        cd = s.cull_data()
        ms = refshader_lib.MeshStage(o, vertices, meshletdata, host.projection(cam, *screen))
        depth = np.zeros((screen[1], screen[0]), np.float32)

        def draw_pass(late):
            o.cull(cd, late)
            n = int(o.dccb[1]) * 64
            payloads, emit = np.zeros((max(n, 1), 64), np.uint32), np.zeros(max(n, 1), np.uint32)
            o.task_shading(cd, late, payloads, emit)
            cmds = o.read_task_commands(n)
            rec, pos, tri = ms.run_payloads(cd, payloads[:n], emit[:n])
            assert len(rec) == int(emit[:n].sum()) and (rec[:, 0] > 0).all()
            # what the mesh stage decoded == what the payloads say: (drawId, meshlet) per slot
            ci = np.concatenate([payloads[c, : emit[c]] for c in range(n)]) if n else np.zeros(0, np.uint32)
            assert np.array_equal(ci & 0xFFFFFF, rec[:, 3])
            assert np.array_equal(rec[:, 2], cmds["drawId"][ci & 0xFFFFFF])
            assert np.array_equal(rec[:, 1], s.meshlets["triangleCount"][cmds["taskOffset"][ci & 0xFFFFFF] + (ci >> 24)])
            ms.rasterize(rec, pos, tri, depth)
            return oracle_lib.cluster_pairs(ci, cmds)

        early = draw_pass(False)
        o.pyramid(depth)
        late = draw_pass(True)
        assert len(np.intersect1d(early, late)) == 0
        late_total += len(late)
        gt.dvb[:] = 1
        gt.cull(s.cull_data(culling=False, occlusion=False, cluster_occlusion=False), late=False)
        all_cmds = gt.read_task_commands(int(gt.dccb[1]) * 64)
        cib, ccb, ci = _all_clusters(all_cmds, int(gt.dccb[0]))
        rec, pos, tri = ms.run(cd, cib=cib, ccb=ccb, dcb=gt.dcb)
        truth = np.zeros_like(depth)
        ms.rasterize(rec, pos, tri, truth)
        assert np.array_equal(truth, depth)
        own = ms.owners(rec, pos, tri, truth)
        owner_pairs = oracle_lib.cluster_pairs(ci[own[: len(ci)]], all_cmds)
        assert np.isin(owner_pairs, np.union1d(early, late)).all()
        owners_total += len(owner_pairs)
    assert owners_total > 3000 and late_total > 0


@pytest.mark.parametrize("culler", CULLERS)
def test_draw_path_on_rasterised_depth(golden_dir, culler):
    """The third submission mode (mesh shading off, niagara.cpp:1680-1694): drawcull writes MeshDrawCommand[] + a count, consumed by
    vkCmdDrawIndexedIndirectCount with mesh.vert.glsl.  Geometry comes out of the reference-written compressed cache through OUR
    codecs (vertices + indices of kitten.z.cache).  Closed loop as above: early / late draw sets disjoint, image == brute force of
    every draw at its selected LOD, every pixel-owning draw emitted."""
    from niagara_b200 import scene_cache

    screen = (512, 384)
    cache = scene_cache.SceneCache(os.path.join(golden_dir, "kitten.z.cache"))
    vertices, indices, meshes, meshlets = cache.section("vertices"), cache.section("indices"), cache.section("meshes"), cache.section("meshlets")
    s, _, _ = _kitten_scene(golden_dir, 160, screen)
    assert np.array_equal(s.meshes, meshes)
    o = _culler(culler)(meshes, meshlets, s.draws, *screen, mesh_shading=False, threads=8)
    gt = oracle_lib.OraclePath(meshes, meshlets, s.draws, *screen, mesh_shading=False, threads=8)
    cams = [host.make_camera((0, 0, 0)), host.make_camera((0, 0, 0)), host.make_camera((4.0, 0.5, 3.0), host.quat_from_axis_angle((0, 1, 0), 0.25)), host.make_camera((4.0, 0.5, 3.0), host.quat_from_axis_angle((0, 1, 0), 0.25))]
    toggles = dict(mesh_shading=False, cluster_occlusion=False)
    owners_total, late_total, lods = 0, 0, set()
    for cam in cams:
        s.camera = cam
        cd = s.cull_data(**toggles)
        vs = refshader_lib.VertexStage(o, vertices, indices, host.projection(cam, *screen))
        depth = np.zeros((screen[1], screen[0]), np.float32)

        def draw_pass(late):
            o.cull(cd, late, task=False)
            n = int(o.dccb[0])
            vs.draw(cd, depth)
            cmds = o.read_draw_commands(n)
            lods.update(cmds["indexCount"].tolist())
            return np.sort(cmds["drawId"])

        early = draw_pass(False)
        o.pyramid(depth)
        late = draw_pass(True)
        assert len(np.intersect1d(early, late)) == 0 and len(np.unique(early)) == len(early)
        late_total += len(late)
        gt.dvb[:] = 1
        gt.cull(s.cull_data(culling=False, occlusion=False, **toggles), late=False, task=False)
        assert int(gt.dccb[0]) == len(s.draws)
        vg = refshader_lib.VertexStage(gt, vertices, indices, host.projection(cam, *screen))
        truth = np.zeros_like(depth)
        vg.draw(cd, truth)
        assert np.array_equal(truth, depth)
        own = vg.draw(cd, truth, owners=True)
        owner_draws = gt.read_draw_commands(len(s.draws))["drawId"][own]
        assert np.isin(owner_draws, np.union1d(early, late)).all()
        owners_total += len(owner_draws)
        assert (truth > 0).mean() > 0.2
    assert owners_total > 200 and late_total > 0 and len(lods) >= 2


def test_animated_cache_scene_with_post_pass(golden_dir):
    """Everything at once on the scene the reference's importer made from tests/golden/animated.gltf: cache reader (N2) -> keyframe
    animation between frames (N3) -> early / late / POST passes (postPass = 1 draws: the alpha-blended primitives) -> the reference's
    mesh shader -> rasteriser -> pyramid.  Image == brute force of all 14 draws, every pixel-owning cluster emitted by exactly one pass."""
    from niagara_b200 import scene_cache

    screen = (512, 384)
    path = os.path.join(golden_dir, "animated.z.cache")
    s = scene_cache.load_scene(path, screen=screen)
    cache = scene_cache.SceneCache(path)
    vertices, meshletdata = cache.section("vertices"), cache.section("meshletdata")
    assert set(s.draws["postPass"].tolist()) == {0, 1}
    o = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *screen, threads=4)
    o.set_visibility_bits(s.visibility_bits)
    gt = oracle_lib.OraclePath(s.meshes, s.meshlets, s.draws, *screen, threads=4)
    gt.set_visibility_bits(s.visibility_bits)
    s.camera = host.make_camera((0.0, 1.0, 16.0), (0.0, 0.0, 0.0, 1.0), s.camera.fovY, s.camera.znear)
    owners_total, post_total, moved = 0, 0, 0
    for t in (0.0, 0.0, 0.7, 0.95, 1.6, 1.6):
        idx, _ = host.animate(s.animations, s.keyframes, t, s.draws)
        moved += len(idx)
        o.draws[...] = s.draws
        gt.draws[...] = s.draws
        cd = s.cull_data()
        ms = refshader_lib.MeshStage(o, vertices, meshletdata, host.projection(s.camera, *screen), threads=4)
        depth = np.zeros((screen[1], screen[0]), np.float32)

        def draw_pass(late, post):
            o.cull(cd, late, post_pass=post)
            o.render_clusters(cd, late, post_pass=post)
            n = int(o.ccb[0])
            rec, pos, tri = ms.run(cd)
            assert int((rec[:, 0] > 0).sum()) == n
            ms.rasterize(rec, pos, tri, depth)
            return oracle_lib.cluster_pairs(o.read_cluster_indices(n), o.read_task_commands(int(o.dccb[1]) * 64))

        early = draw_pass(False, 0)
        o.pyramid(depth)
        late = draw_pass(True, 0)
        post = draw_pass(True, 1)
        assert len(np.intersect1d(early, late)) == 0 and len(np.intersect1d(np.union1d(early, late), post)) == 0
        post_total += len(post)

        truth = np.zeros_like(depth)
        everything = []
        for pp in (0, 1):
            gt.dvb[:] = 1
            gt.cull(s.cull_data(culling=False, occlusion=False, cluster_occlusion=False), late=False, post_pass=pp)
            cmds = gt.read_task_commands(int(gt.dccb[1]) * 64)
            cib, ccb, ci = _all_clusters(cmds, int(gt.dccb[0]))
            mg = refshader_lib.MeshStage(gt, vertices, meshletdata, host.projection(s.camera, *screen), threads=4)
            rec, pos, tri = mg.run(cd, cib=cib, ccb=ccb)
            mg.rasterize(rec, pos, tri, truth)
            everything.append((mg, rec, pos, tri, ci, cmds.copy()))
        assert np.array_equal(truth, depth)
        emitted = np.union1d(np.union1d(early, late), post)
        for mg, rec, pos, tri, ci, cmds in everything:
            own = mg.owners(rec, pos, tri, truth)
            owner_pairs = oracle_lib.cluster_pairs(ci[own[: len(ci)]], cmds)
            assert np.isin(owner_pairs, emitted).all()
            owners_total += len(owner_pairs)
        assert (truth > 0).mean() > 0.02
    assert moved >= 9 and post_total > 0 and owners_total > 100


def test_device_rasteriser_matches_the_test_rasteriser(golden_dir):
    """nvc_raster_depth (the product's kernel, under the CPU emulation) against the reference's mesh shader + the sequential test
    rasteriser on the same cib / ccb / dcb: identical depth images bit for bit, early and late pass, moving camera."""
    screen = (320, 240)
    s, vertices, meshletdata = _kitten_scene(golden_dir, 120, screen)
    o = emu_lib.EmuPath(s.meshes, s.meshlets, s.draws, *screen, threads=4)
    o.set_visibility_bits(s.visibility_bits)
    cams = [host.make_camera((0, 0, 0)), host.make_camera((2.5, -1.0, 2.0), host.quat_from_axis_angle((0, 1, 0), 0.2))]
    drawn_total = 0
    for cam in cams:
        s.camera = cam
        cd = s.cull_data()
        proj = host.projection(cam, *screen)
        ms = refshader_lib.MeshStage(o, vertices, meshletdata, proj)
        want = np.zeros((screen[1], screen[0]), np.float32)
        got = np.zeros_like(want)
        for late in (False, True):
            if late:
                o.pyramid(want)
            o.cull(cd, late)
            o.render_clusters(cd, late)
            rec, pos, tri = ms.run(cd)
            ms.rasterize(rec, pos, tri, want)
            stats = o.raster_depth(cd, proj, vertices, meshletdata, got)
            assert int(stats[0]) == int(o.ccb[0]) and int(stats[2]) == 0
            drawn_total += int(stats[0])
            assert np.array_equal(want.view(np.uint32), got.view(np.uint32)), (late, int((want != got).sum()))
    assert drawn_total > 300 and (want > 0).mean() > 0.05
    # hostile geometry references are skipped and counted, never read
    bad = o.meshlets.copy()
    bad["dataOffset"][:] = 0x7FFFFFF0
    good, o.meshlets = o.meshlets, bad
    depth = np.zeros_like(want)
    stats = o.raster_depth(cd, proj, vertices, meshletdata, depth)
    assert int(stats[0]) == 0 and int(stats[2]) == int(o.ccb[0]) and not depth.any()
    o.meshlets = good
    o.close()
