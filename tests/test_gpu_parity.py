"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle on the same inputs.
Bar: bit-exact — identical visible sets, lod selection, counters, padding, dvb / mvb words, every pyramid texel.
Only ORDER inside dcb / cib may differ (atomics), exactly as in the reference (SURVEY §8(b))."""
import os

import numpy as np
import pytest

import oracle_lib
from niagara_b200 import host, layout, scenes

pytestmark = pytest.mark.gpu


def _torch():
    import torch

    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


def _paths(s, hiz_stage_texels=None, prepare_meshes=True, checker=None, **kw):
    from niagara_b200.path import VisibilityPath

    torch = _torch()
    g = VisibilityPath(s.meshes, s.meshlets, s.draws, *s.screen, hiz_stage_texels=hiz_stage_texels, prepare_meshes=prepare_meshes, **kw)
    o = (checker or oracle_lib.OraclePath)(s.meshes, s.meshlets, s.draws, *s.screen, threads=8, **kw)
    g.set_visibility_bits(s.visibility_bits)
    o.set_visibility_bits(s.visibility_bits)
    depth = torch.from_numpy(s.depth).cuda()
    return g, o, depth


def _compare_draw_pass(g, o, task, what):
    torch = _torch()
    torch.cuda.synchronize()
    gd, _ = g.read_counts()
    od, _ = o.read_counts()
    assert np.array_equal(gd, od), (what, gd, od)
    if task:
        n = int(gd[1]) * 64  # includes the zero padding written by the tasksubmit epilogue
        assert np.array_equal(oracle_lib.sorted_commands(g.read_task_commands(n)), oracle_lib.sorted_commands(o.read_task_commands(n))), what
    else:
        n = int(gd[0])
        assert np.array_equal(oracle_lib.sorted_commands(g.read_draw_commands(n)), oracle_lib.sorted_commands(o.read_draw_commands(n))), what
    assert np.array_equal(g.dvb.cpu().numpy().astype(np.uint32)[: len(o.dvb)], o.dvb), what


def _compare_cluster_pass(g, o, what):
    torch = _torch()
    torch.cuda.synchronize()
    gd, gc = g.read_counts()
    od, oc = o.read_counts()
    assert np.array_equal(gc, oc), (what, gc, oc)
    n = int(gc[0])
    gt, ot = g.read_task_commands(int(gd[1]) * 64), o.read_task_commands(int(od[1]) * 64)
    assert np.array_equal(oracle_lib.cluster_pairs(g.read_cluster_indices(n), gt), oracle_lib.cluster_pairs(o.read_cluster_indices(n), ot)), what
    pad = (n + 255) // 256 * 256
    assert (g.read_cluster_indices(pad)[n:] == 0xFFFFFFFF).all(), what
    assert np.array_equal(g.mvb.cpu().numpy().astype(np.uint32), o.mvb), what


def _compare_pyramid(g, o, what):
    _torch().cuda.synchronize()
    assert np.array_equal(g.depthPyramid.cpu().numpy().view(np.uint32), o.pyramid_texels.view(np.uint32)), what


def _run_frames(s, frames=2, cameras=None, toggles=None, cluster_backface=True, **kw):
    g, o, depth = _paths(s, **kw)
    for f in range(frames):
        if cameras:
            s.camera = cameras[f % len(cameras)]
        cd = s.cull_data(**(toggles or {}))
        for late in (False, True):
            if late:
                g.pyramid(depth)
                o.pyramid(s.depth)
                _compare_pyramid(g, o, ("pyramid", f))
            g.cull(cd, late)
            o.cull(cd, late)
            _compare_draw_pass(g, o, g.mesh_shading, ("cull", f, late))
            if g.mesh_shading:
                g.render_clusters(cd, late, cluster_backface=cluster_backface)
                o.render_clusters(cd, late, cluster_backface=cluster_backface)
                _compare_cluster_pass(g, o, ("clusters", f, late))
    return g, o


def test_kitten_4096_two_phase(golden_dir):
    """BASELINE configs[0] geometry (kitten.obj cooked by the reference's scene.cpp), 4096 instanced draws."""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten.nvcg"), 4096)
    g, o = _run_frames(s, frames=3)
    assert o.read_counts()[0][0] > 0


def test_cuda_reproduces_committed_vectors(golden_dir):
    """The CUDA path against the COMMITTED expected outputs of BASELINE configs[0] + its two-phase variant
    (tests/golden/c1_kitten_expected.npz, reproduced byte for byte by the oracle and by the reference's own shaders on the
    CPU side): counters, dvb, mvb, pyramid digest exactly; command lists and cluster indices as sets."""
    torch = _torch()
    from niagara_b200.path import VisibilityPath

    want = np.load(os.path.join(golden_dir, "c1_kitten_expected.npz"))
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten.nvcg"), 4096)

    # (a) frustum + LOD only, draw-command path, every draw visible last frame
    cd = s.cull_data(occlusion=False, cluster_occlusion=False, mesh_shading=False)
    g = VisibilityPath(s.meshes, s.meshlets, s.draws, *s.screen, mesh_shading=False)
    g.dvb.fill_(1)
    g.cull(cd, late=False, task=False)
    torch.cuda.synchronize()
    n = int(g.read_counts()[0][0])
    assert n == int(want["a_count"])
    got = g.read_draw_commands(n).view(np.uint32).reshape(n, 6)
    order = lambda a: a[np.lexsort(a.T[::-1])]
    assert np.array_equal(order(got), order(want["a_commands"]))

    # (b) two frames of the full two-phase path with cone culling
    cd = s.cull_data()
    g = VisibilityPath(s.meshes, s.meshlets, s.draws, *s.screen)
    g.set_visibility_bits(s.visibility_bits)
    depth = torch.from_numpy(s.depth).cuda()
    crc = lambda v: np.uint64(int(np.bitwise_xor.reduce(v.astype(np.uint64) * np.arange(1, len(v) + 1, dtype=np.uint64)))) if len(v) else np.uint64(0)
    for f in range(2):
        g.frame(cd, depth, cluster_backface=True)
        torch.cuda.synchronize()
        dccb, ccb = g.read_counts()
        assert np.array_equal(dccb, want["b%d_dccb" % f]) and np.array_equal(ccb, want["b%d_ccb" % f])
        assert np.array_equal(np.packbits(g.dvb.cpu().numpy()[: len(s.draws)].astype(np.uint8)), want["b%d_dvb" % f])
        assert np.array_equal(g.mvb.cpu().numpy().astype(np.uint32), want["b%d_mvb" % f])
        cmds = g.read_task_commands(int(dccb[1]) * 64).view(np.uint32).reshape(-1, 5)
        assert np.array_equal(order(cmds), order(want["b%d_commands" % f]))
    pyr = g.depthPyramid.cpu().numpy()
    assert np.array_equal(pyr[-341:].view(np.uint32), want["b_pyramid_top"].view(np.uint32))
    assert crc(pyr.view(np.uint32)) == want["b_pyramid_crc"]


def test_cuda_vs_reference_shaders(golden_dir, request):
    """The CUDA path against the reference's OWN GLSL shaders run on the host (oracle/_ref/librefshader.so: the text of
    src/shaders/*.glsl compiled through oracle/refshader/glsl_shim.h).  Same bar as against the oracle: bit-exact, order
    inside dcb / cib aside.  Without the library the oracle runs in its place, held to the reference's pinned outputs."""
    import reference_pins
    import refshader_lib

    with reference_pins.pinned(request, refshader_lib.available()):
        s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 20000, screen=(1280, 720))
        g, r = _run_frames(s, frames=2, checker=refshader_lib.RefShaderPath)
        assert r.read_counts()[0][0] > 0
        s = scenes.config2_scene(draw_count=50000, num_meshes=256, screen=(1024, 1024))
        _run_frames(s, frames=2, checker=refshader_lib.RefShaderPath)
        s = scenes.instanced_scene(os.path.join(golden_dir, "kitten.nvcg"), 3000)
        _run_frames(s, frames=2, checker=refshader_lib.RefShaderPath, toggles=dict(mesh_shading=False, cluster_occlusion=False), mesh_shading=False)


def test_scene_cache_and_animated_draws(golden_dir):
    """Widening N2 + N3: a scene read from a reference-written compressed cache (nvc_scene_cache_*), animated with
    nvc_host_animate, the changed draws scattered into the device buffer by nvc_update_draws; every frame bit-exact
    against the oracle fed with the same host arrays."""
    from niagara_b200 import scene_cache

    torch = _torch()
    s = scene_cache.load_scene(os.path.join(golden_dir, "animated.z.cache"), screen=(640, 480))
    g, o, depth = _paths(s)
    for f, t in enumerate((0.0, 0.9, 1.7, 2.05, 7.3)):
        idx, val = host.animate(s.animations, s.keyframes, t, s.draws)
        assert len(idx) == (0 if t < 0.5 else 3)
        g.scatter_draws(idx, val)
        o.draws[...] = s.draws
        torch.cuda.synchronize()
        assert np.array_equal(g.db.cpu().numpy().view(layout.MESHDRAW_DTYPE), s.draws)
        cd = s.cull_data()
        for late in (False, True):
            if late:
                g.pyramid(depth)
                o.pyramid(s.depth)
            for post in (0, 1):
                if post and not late:
                    continue
                g.cull(cd, late, post_pass=post)
                o.cull(cd, late, post_pass=post)
                _compare_draw_pass(g, o, True, ("cull", f, late, post))
                g.render_clusters(cd, late, post_pass=post)
                o.render_clusters(cd, late, post_pass=post)
                _compare_cluster_pass(g, o, ("clusters", f, late, post))
    # out-of-range indices are ignored, nothing else is touched
    before = g.db.cpu().numpy().copy()
    g.scatter_draws(np.array([len(s.draws) + 5], np.uint32), s.draws[:1])
    torch.cuda.synchronize()
    assert np.array_equal(g.db.cpu().numpy(), before)


@pytest.mark.parametrize(
    "toggles",
    [dict(lod=False), dict(culling=False), dict(occlusion=False), dict(cluster_occlusion=False), dict(debug_lod_step=3)],
)
def test_toggles(golden_dir, toggles):
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 20000, screen=(1280, 720))
    _run_frames(s, frames=2, toggles=toggles)


@pytest.mark.parametrize("backface", [False, True, None])
def test_cluster_backface_flag(golden_dir, backface):
    """clusterBackfaceEnabled 0 / 1 / reference wiring (never set for the cluster pass, SURVEY F8)."""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 15000, screen=(1024, 768))
    _run_frames(s, frames=2, cluster_backface=backface)


def test_moving_camera_multi_frame(golden_dir):
    """Early/late interplay: the camera moves and turns every frame so draws and meshlets change visibility state."""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 60000, screen=(1920, 1080))
    cams = [
        host.make_camera((0, 0, 0)),
        host.make_camera((30, -10, 20), host.quat_from_axis_angle((0, 1, 0), 0.4)),
        host.make_camera((60, 5, -40), host.quat_from_axis_angle((0.2, 1, 0.1), 1.3)),
        host.make_camera((-20, 40, 10), host.quat_from_axis_angle((1, 0.3, 0), -0.7)),
    ]
    _run_frames(s, frames=5, cameras=cams)


@pytest.mark.parametrize("texels", [6144, 11264, 87, 5])
def test_tma_staged_hiz(golden_dir, texels):
    """coarse Hi-Z mips staged into shared memory by one TMA bulk copy per CTA (nvc_set_hiz_staging): same results.
    Close-up draws so that many lookups land in the staged mips."""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 30000, screen=(1920, 1080))
    s.draws["position"][:, 2] = -np.abs(s.draws["position"][:, 2]) * 0.1 - 3
    s.draws["position"][:, :2] *= 0.03
    cams = [host.make_camera((0, 0, 0)), host.make_camera((1, -0.5, 2), host.quat_from_axis_angle((0, 1, 0), 0.2))]
    _run_frames(s, frames=3, cameras=cams, hiz_stage_texels=texels)


@pytest.mark.parametrize("mesh_shading", [True, False])
def test_without_prepared_mesh_view(golden_dir, mesh_shading):
    """nvc_prepare_meshes is optional: the plain AoS Mesh[] path must give the same results (task and draw commands)"""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 30000, screen=(1024, 768))
    toggles = None if mesh_shading else dict(mesh_shading=False, cluster_occlusion=False)
    _run_frames(s, frames=2, toggles=toggles, mesh_shading=mesh_shading, prepare_meshes=False)


def test_draw_path_without_mesh_shading(golden_dir):
    """TASK = 0 variants: MeshDrawCommand output for vkCmdDrawIndexedIndirectCount (niagara.cpp:1680-1694)."""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 50000, screen=(1024, 768))
    _run_frames(s, frames=3, toggles=dict(mesh_shading=False, cluster_occlusion=False), mesh_shading=False)


def test_post_pass_draws(golden_dir):
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 8000)
    s.draws["postPass"][::3] = 1
    g, o, depth = _paths(s)
    cd = s.cull_data()
    for f in range(2):
        g.frame(cd, depth, post_passes=True, cluster_backface=True)
        o.frame(cd, s.depth, post_passes=True, cluster_backface=True)
        _compare_draw_pass(g, o, True, ("post", f))
        _compare_cluster_pass(g, o, ("post", f))


def test_empty_and_tiny_inputs(golden_dir):
    meshes, meshlets, _ = layout.load_nvcg(os.path.join(golden_dir, "kitten.nvcg"))
    for n in (0, 1, 31, 33, 257):
        s = scenes.reference_random_scene(meshes, meshlets, max(n, 1), screen=(64, 48))
        s.draws["position"][:] = (0, 0, -20)  # in front of the default camera (view z = -world z)
        s.draws = s.draws[:n] if n else s.draws[:1]
        g, o, depth = _paths(s)
        cd = s.cull_data()
        if n == 0:
            cd.drawCount = 0
        for f in range(2):
            g.frame(cd, depth, cluster_backface=True)
            o.frame(cd, s.depth, cluster_backface=True)
            _compare_draw_pass(g, o, True, ("tiny", n, f))
            _compare_cluster_pass(g, o, ("tiny", n, f))


@pytest.mark.parametrize("size", [(64, 64), (128, 128), (100, 60), (1920, 1080), (4096, 4096), (2048, 256), (30, 17), (3, 2), (1, 1), (4096, 600), (16384, 4), (4, 16384), (8192, 130), (512, 512)])
def test_pyramid_sizes(size):
    torch = _torch()
    from niagara_b200.path import VisibilityPath

    w, h = size
    rng = np.random.default_rng(w + 7 * h)
    depth = rng.random((h, w), dtype=np.float32)
    dummy = (np.zeros(1, layout.MESH_DTYPE), np.zeros(1, layout.MESHLET_DTYPE), np.zeros(1, layout.MESHDRAW_DTYPE))
    g = VisibilityPath(*dummy, w, h, task_wglimit=64, cluster_limit=256)
    o = oracle_lib.OraclePath(*dummy, w, h, threads=8)
    for rep in range(2):  # second run checks that the ticket counter was left reset
        g.depthPyramid.zero_()
        g.pyramid(torch.from_numpy(depth).cuda())
        o.pyramid(depth)
        _compare_pyramid(g, o, size)


def test_pyramid_unaligned_depth_pointer():
    """the 16-byte-load fast path must not be taken for a depth pointer that is only 4-byte aligned"""
    torch = _torch()
    from niagara_b200.path import VisibilityPath

    w = h = 256
    rng = np.random.default_rng(3)
    depth = rng.random((h, w), dtype=np.float32)
    dummy = (np.zeros(1, layout.MESH_DTYPE), np.zeros(1, layout.MESHLET_DTYPE), np.zeros(1, layout.MESHDRAW_DTYPE))
    g = VisibilityPath(*dummy, w, h, task_wglimit=64, cluster_limit=256)
    o = oracle_lib.OraclePath(*dummy, w, h)
    buf = torch.zeros(w * h + 1, dtype=torch.float32, device="cuda")
    view = buf[1:].view(h, w)
    view.copy_(torch.from_numpy(depth))
    assert view.data_ptr() % 16 != 0
    g.pyramid(view)
    o.pyramid(depth)
    _compare_pyramid(g, o, "unaligned")


def test_big_meshes_many_groups_per_draw(golden_dir):
    """draws with hundreds of meshlets (several task commands per draw, blocks that exceed the command staging
    buffer take the direct write path)"""
    meshes, nmeshlets = scenes.synthetic_meshes(40, 3, 700, seed=5)
    meshlets = scenes.synthetic_meshlets(nmeshlets, seed=6)
    s = scenes.reference_random_scene(meshes, meshlets, 30000, screen=(1024, 1024))
    s.draws["position"][:, 2] = -np.abs(s.draws["position"][:, 2]) * 0.4 - 10
    s.draws["position"][:, :2] *= 0.2
    _run_frames(s, frames=2)


def test_overflow_limits(golden_dir):
    """TASK_WGLIMIT / CLUSTER_LIMIT overflow (drawcull.comp.glsl:129, clustercull.comp.glsl:137, the submit clamps):
    counters keep counting, writes are dropped, dispatch sizes clamp.  WHICH draws are dropped depends on atomic
    order, so compare counters, clamps, padding and that everything written is a subset of the unlimited result."""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten.nvcg"), 30000, screen=(800, 600))
    s.draws["position"][:, 2] = -np.abs(s.draws["position"][:, 2]) * 0.3 - 5
    s.draws["position"][:, :2] *= 0.05
    cd = s.cull_data()
    full_g, full_o = _run_frames(s, frames=1)
    fd, fc = full_o.read_counts()
    assert fd[0] > 1000 and fc[0] > 5000
    wg, cl = 640, 2048
    g, o, depth = _paths(s, task_wglimit=wg, cluster_limit=cl)
    g.dcb.zero_()
    for late in (False, True):
        g.pyramid(depth)
        o.pyramid(s.depth)
        g.cull(cd, late)
        o.cull(cd, late)
        _torch().cuda.synchronize()
        gd, _ = g.read_counts()
        od, _ = o.read_counts()
        assert np.array_equal(gd, od)  # count unclamped, X clamped identically
        g.render_clusters(cd, late, cluster_backface=True)
        _torch().cuda.synchronize()
        _, gc = g.read_counts()
        if late:
            assert gd[0] == fd[0] and gd[0] > wg and gd[1] == wg // 64
            written = g.read_task_commands(wg)
            live = written[written["taskCount"] > 0]
            allowed = set(map(tuple, full_o.read_task_commands(int(fd[0])).tolist()))
            assert all(tuple(c) in allowed for c in live.tolist())
            assert gc[0] > cl and gc[2] == cl // 256 and gc[1] == 16 and gc[3] == 16


def test_taskcull_payloads(golden_dir):
    """meshlet.task.glsl path: per-command payload + emit count."""
    torch = _torch()
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 12000)
    g, o, depth = _paths(s)
    cd = s.cull_data()
    for f in range(2):
        for late in (False, True):
            if late:
                g.pyramid(depth)
                o.pyramid(s.depth)
            g.cull(cd, late)
            o.cull(cd, late)
            torch.cuda.synchronize()
            n = int(o.read_counts()[0][1]) * 64
            gp = torch.zeros((max(n, 1), 64), dtype=torch.int32, device="cuda")
            ge = torch.zeros(max(n, 1), dtype=torch.int32, device="cuda")
            op = np.zeros((max(n, 1), 64), dtype=np.uint32)
            oe = np.zeros(max(n, 1), dtype=np.uint32)
            g.task_shading(cd, late, gp, ge, cluster_backface=True)
            o.task_shading(cd, late, op, oe, cluster_backface=True)
            torch.cuda.synchronize()
            # commands are in a different order on the two sides: key by command contents
            gt, ot = g.read_task_commands(n), o.read_task_commands(n)
            gp, ge = gp.cpu().numpy().astype(np.uint32), ge.cpu().numpy().astype(np.uint32)

            def table(cmds, payloads, counts):
                out = {}
                for i in range(n):
                    if cmds["taskCount"][i]:
                        out[tuple(cmds[i].tolist())] = tuple(sorted(int(v) >> 24 for v in payloads[i][: counts[i]]))  # order inside a payload is unspecified (atomicAdd, meshlet.task.glsl:137)
                        assert all((int(v) & 0xFFFFFF) == i for v in payloads[i][: counts[i]])
                return out

            assert table(gt, gp, ge) == table(ot, op, oe)
            assert np.array_equal(g.mvb.cpu().numpy().astype(np.uint32), o.mvb)


def test_c4_full_size_bit_exact():
    """BASELINE configs[3] at FULL size (1M draws x 10 unique meshlets = 10M meshlet instances, 4096^2 depth): two
    frames of the whole path, CUDA vs the multi-threaded oracle, bit-exact (counters, dvb, mvb, pyramid, command and
    cluster sets) — plus size-independent properties: steady-state idempotence and conservation between passes."""
    torch = _torch()
    s = scenes.config4_scene()
    g, o, depth = _paths(s)
    o.threads = os.cpu_count() or 8
    cd = s.cull_data()
    for f in range(2):
        for late in (False, True):
            if late:
                g.pyramid(depth)
                o.pyramid(s.depth)
                _compare_pyramid(g, o, ("c4 pyramid", f))
            g.cull(cd, late)
            o.cull(cd, late)
            _compare_draw_pass(g, o, True, ("c4 cull", f, late))
            g.render_clusters(cd, late, cluster_backface=True)
            o.render_clusters(cd, late, cluster_backface=True)
            _compare_cluster_pass(g, o, ("c4 clusters", f, late))
    # properties that hold at any size
    dvb1 = g.dvb.clone()
    mvb1 = g.mvb.clone()
    gd1, gc1 = g.read_counts()
    g.frame(cd, depth, cluster_backface=True)
    torch.cuda.synchronize()
    gd2, gc2 = g.read_counts()
    assert torch.equal(g.dvb, dvb1) and torch.equal(g.mvb, mvb1)  # static camera: the visibility state is a fixed point
    assert np.array_equal(gd1, gd2) and gc2[0] == 0  # everything visible was already drawn by the early pass
    vis_draws = int((g.dvb != 0).sum().item())
    assert gd2[0] == vis_draws  # one task command per visible draw (10 meshlets < 64)
    bits = int(sum(bin(int(x) & 0xFFFFFFFF).count("1") for x in g.mvb.cpu().numpy()[:: 997]))  # sampled popcount is finite
    assert bits >= 0
    # early pass of the next frame emits exactly the meshlets whose bit is set among visible draws
    g.cull(cd, late=False)
    g.render_clusters(cd, late=False, cluster_backface=True)
    torch.cuda.synchronize()
    _, gce = g.read_counts()
    mv = g.mvb.cpu().numpy().astype(np.uint32)
    assert int(gce[0]) == int(np.unpackbits(mv.view(np.uint8)).sum())


def test_hostile_inputs_fuzz(golden_dir):
    """non-finite / degenerate inputs: zero, negative and huge scales, NaN / inf positions, un-normalised and zero
    quaternions, fp16 inf / NaN / subnormal meshlet bounds, extreme cone bytes.  IEEE semantics are the contract, so the
    CUDA path must still equal the oracle bit for bit (and neither may crash)."""
    import hostile

    s = hostile.hostile_scene(golden_dir, 40000)
    cams = [host.make_camera((0, 0, 0)), host.make_camera((5, 2, -3), host.quat_from_axis_angle((0.3, 1, 0), 0.9))]
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _run_frames(s, frames=3, cameras=cams)


def test_decode_clusters_consumer_walk(golden_dir):
    """nvc_decode_clusters (what meshlet.mesh would read) vs the oracle's decode of ITS buffers: same multiset of
    (drawId, meshlet, vertexCount, triangleCount), same statistics, no invalid slot"""
    s = scenes.instanced_scene(os.path.join(golden_dir, "kitten_pirate.nvcg"), 25000, screen=(1280, 720))
    g, o, depth = _paths(s)
    cd = s.cull_data()
    for f in range(2):
        for late in (False, True):
            if late:
                g.pyramid(depth)
                o.pyramid(s.depth)
            g.cull(cd, late)
            o.cull(cd, late)
            g.render_clusters(cd, late, cluster_backface=True)
            o.render_clusters(cd, late, cluster_backface=True)
            grec, gstats = g.decode_clusters()
            orec, ostats = o.decode_clusters()
            assert np.array_equal(gstats, ostats) and gstats[2] == 0, (f, late, gstats, ostats)
            n = int(gstats[0])
            key = lambda r: np.sort((r[:, 0].astype(np.uint64) << 32) | r[:, 1])
            gv, ov = grec[grec[:, 0] != 0xFFFFFFFF], orec[orec[:, 0] != 0xFFFFFFFF]
            assert len(gv) == n and np.array_equal(key(gv), key(ov))
    assert n >= 0


def test_c3_bistro_standin_two_pass(golden_dir):
    """BASELINE configs[2] stand-in (bistro.gltf is not shipped with the reference, SURVEY F7): kitten + pirate geometry
    cooked by the reference's scene.cpp, instanced with its PCG32 recipe to ~3M LOD-0 meshlets, packed around the
    camera; full two-pass Hi-Z occlusion + meshlet cone cull over three frames with a moving camera, bit-exact, plus the
    two-phase invariants (no meshlet emitted twice in a frame, every late-visible meshlet emitted once)."""
    torch = _torch()
    meshes, meshlets, _ = layout.load_nvcg(os.path.join(golden_dir, "kitten_pirate.nvcg"))
    n = 16500
    s = scenes.reference_random_scene(meshes, meshlets, n, screen=(1920, 1080), occluders=80)
    s.draws["position"] *= 0.3  # +-90 around the origin: most of the scene is inside the 200 draw distance
    lod0 = int(meshes["lods"]["meshletCount"][s.draws["meshIndex"], 0].sum())
    assert 2.8e6 < lod0 < 3.3e6
    g, o, depth = _paths(s)
    cams = [host.make_camera((0, 0, 0)), host.make_camera((8, -2, 15), host.quat_from_axis_angle((0, 1, 0), 0.5)), host.make_camera((-20, 6, 30), host.quat_from_axis_angle((0.2, 1, 0), 2.2))]
    for f in range(3):
        s.camera = cams[f]
        cd = s.cull_data()
        g.cull(cd, False)
        o.cull(cd, False)
        _compare_draw_pass(g, o, True, ("c3 cull early", f))
        g.render_clusters(cd, False, cluster_backface=True)
        o.render_clusters(cd, False, cluster_backface=True)
        _compare_cluster_pass(g, o, ("c3 clusters early", f))
        gd, gc = g.read_counts()
        early = oracle_lib.cluster_pairs(g.read_cluster_indices(int(gc[0])), g.read_task_commands(int(gd[1]) * 64))
        g.pyramid(depth)
        o.pyramid(s.depth)
        g.cull(cd, True)
        o.cull(cd, True)
        _compare_draw_pass(g, o, True, ("c3 cull late", f))
        g.render_clusters(cd, True, cluster_backface=True)
        o.render_clusters(cd, True, cluster_backface=True)
        _compare_cluster_pass(g, o, ("c3 clusters late", f))
        gd, gc = g.read_counts()
        late = oracle_lib.cluster_pairs(g.read_cluster_indices(int(gc[0])), g.read_task_commands(int(gd[1]) * 64))
        assert len(np.intersect1d(early, late)) == 0
        rec, stats = g.decode_clusters()
        assert stats[2] == 0 and stats[0] == gc[0]
    assert int(o.read_counts()[1][0]) >= 0 and len(early) + len(late) > 10000


def test_two_phase_on_device_produced_depth(golden_dir, request):
    """The whole loop on the device with NO synthetic depth: early cull -> nvc_raster_depth -> pyramid of that depth -> late cull ->
    nvc_raster_depth, over a moving camera — against the oracle culling + the reference's mesh shader + the sequential test
    rasteriser (oracle/refshader) doing the same on the CPU.  Depth images, cluster sets and visibility state must be identical.
    Without the reference's shaders their mesh stage is stood in for and held to its pinned outputs."""
    import reference_pins
    import refshader_lib

    with reference_pins.pinned(request, refshader_lib.available()):
        _two_phase_on_device_produced_depth(golden_dir)


def _two_phase_on_device_produced_depth(golden_dir):
    import refshader_lib

    torch = _torch()
    from test_end_to_end_raster import _kitten_scene

    screen = (512, 384)
    s, vertices, meshletdata = _kitten_scene(golden_dir, 300, screen)
    g, o, _ = _paths(s)
    vb = torch.from_numpy(np.ascontiguousarray(vertices)).cuda()
    md = torch.from_numpy(np.ascontiguousarray(meshletdata, dtype=np.uint32).view(np.int32)).cuda()
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    cams = [host.make_camera((0, 0, 0)), host.make_camera((0, 0, 0)), host.make_camera((3.5, -1.0, 2.0), host.quat_from_axis_angle((0, 1, 0), 0.18)),
            host.make_camera((7.0, 1.5, 5.0), host.quat_from_axis_angle((0.1, 1, 0), 0.42))]
    late_total = 0
    for f, cam in enumerate(cams):
        s.camera = cam
        cd = s.cull_data()
        proj = host.projection(cam, *screen)
        ms = refshader_lib.MeshStage(o, vertices, meshletdata, proj)
        want = np.zeros((screen[1], screen[0]), np.float32)
        got = torch.zeros((screen[1], screen[0]), dtype=torch.float32, device="cuda")
        for late in (False, True):
            if late:
                g.pyramid(got)
                o.pyramid(want)
                _compare_pyramid(g, o, ("pyramid of produced depth", f))
            g.cull(cd, late)
            o.cull(cd, late)
            _compare_draw_pass(g, o, True, ("cull", f, late))
            g.render_clusters(cd, late)
            o.render_clusters(cd, late)
            _compare_cluster_pass(g, o, ("clusters", f, late))
            rec, pos, tri = ms.run(cd)
            ms.rasterize(rec, pos, tri, want)
            g.raster_depth(cd, proj, vb, md, got, stats)
            torch.cuda.synchronize()
            st = stats.cpu().numpy()
            assert int(st[0]) == int(o.ccb[0]) and int(st[2]) == 0, (f, late, st)
            assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32)), ("depth image", f, late)
            if late:
                late_total += int(o.ccb[0])
    assert late_total > 0 and (want > 0).mean() > 0.2


@pytest.mark.parametrize("num_meshes,lod0", [(1024, 64), (1_000_000, 8)])
def test_c2_full_size_bit_exact(num_meshes, lod0):
    """BASELINE configs[1] at FULL size: the reference's own PCG32 scene with 1M draws over 4-LOD meshes, 4096^2 depth, both
    settings of SURVEY §8(d)'s mesh-count knob (1024 = L2-resident mesh table, 1 000 000 = one Mesh gather per draw) — two frames,
    CUDA vs the multi-threaded oracle, bit-exact incl. the selected LOD of every surviving draw (carried by the task commands)."""
    s = scenes.config2_scene(draw_count=1_000_000, num_meshes=num_meshes, lod0_meshlets=lod0)
    g, o, depth = _paths(s)
    o.threads = os.cpu_count() or 8
    cd = s.cull_data()
    survivors = 0
    for f in range(2):
        for late in (False, True):
            if late:
                g.pyramid(depth)
                o.pyramid(s.depth)
            g.cull(cd, late)
            o.cull(cd, late)
            _compare_draw_pass(g, o, True, ("c2 cull", num_meshes, f, late))
            g.render_clusters(cd, late, cluster_backface=True)
            o.render_clusters(cd, late, cluster_backface=True)
            _compare_cluster_pass(g, o, ("c2 clusters", num_meshes, f, late))
            survivors += int(o.read_counts()[0][0])
    assert survivors > 1000
