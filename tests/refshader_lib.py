"""ctypes wrapper of oracle/_ref/librefshader.so — the reference's OWN GLSL shaders compiled for the host through
oracle/refshader/glsl_shim.h (see oracle/refshader/gen.py).  Test infrastructure only: it is the third, strongest
checker of the oracle (the shader text itself instead of a restatement) and, transitively, of the CUDA path.

The library is built from the reference checkout named by NIAGARA_REFERENCE where that exists, or a prebuilt
oracle/_ref/librefshader.so is used.  Without either, RefShaderPath runs the oracle in its place and every pass checks its
outputs against the reference's, pinned by tests/reference_pins.py."""
import ctypes
import os
import subprocess

import numpy as np

from niagara_b200 import layout

import oracle_lib
import reference_pins

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "_ref", "librefshader.so")
REFERENCE = os.environ.get("NIAGARA_REFERENCE", "/root/reference")
_LIB = None

vp = ctypes.c_void_p
sz = ctypes.c_size_t


def available():
    return os.path.exists(SO) or os.path.isdir(os.path.join(REFERENCE, "src", "shaders"))


def _stand_in():
    """tests/mesh_stage_host.cpp: the mesh / vertex stages without the reference's shaders (built into tests/_build/)"""
    out = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libmeshstage.so")
    srcs = [os.path.join(ROOT, "tests", "mesh_stage_host.cpp"), os.path.join(ROOT, "oracle", "refshader", "raster.h"), os.path.join(ROOT, "include", "niagara_cull.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-msse2", "-mfpmath=sse", srcs[0], "-o", so], check=True)
    return ctypes.CDLL(so)


def load():
    """The reference's shaders (librefshader.so) where available(); elsewhere the stand-in of their mesh and vertex stages
    (rs_mesh_clusters, rs_mesh_payloads, rs_draw_indexed, rs_rasterize only)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not available():
        lib = _stand_in()
        _bind_stages(lib)
        _LIB = lib
        return lib
    if os.path.isdir(os.path.join(REFERENCE, "src", "shaders")):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle", "refshader"), "REF=" + REFERENCE], check=True)
    lib = ctypes.CDLL(SO)
    cd, hz = ctypes.POINTER(layout.CullData), ctypes.POINTER(layout.HiZ)
    lib.rs_sources.restype = ctypes.c_char_p
    lib.rs_drawcull.restype = ctypes.c_int
    lib.rs_drawcull.argtypes = [cd, ctypes.c_int, ctypes.c_int, vp, sz, vp, sz, vp, sz, vp, sz, vp, hz, ctypes.c_int]
    lib.rs_clustercull.restype = ctypes.c_int
    lib.rs_clustercull.argtypes = [cd, ctypes.c_int, vp, sz, vp, vp, sz, vp, sz, vp, sz, vp, sz, vp, hz, ctypes.c_int]
    lib.rs_taskcull.restype = ctypes.c_int
    lib.rs_taskcull.argtypes = [cd, ctypes.c_int, vp, sz, vp, vp, sz, vp, sz, vp, sz, vp, vp, hz, ctypes.c_int]
    lib.rs_depth_pyramid.restype = ctypes.c_int
    lib.rs_depth_pyramid.argtypes = [vp, ctypes.c_uint32, ctypes.c_uint32, hz, ctypes.c_int]
    _bind_stages(lib)
    lib.rs_project_sphere.restype = ctypes.c_int
    lib.rs_project_sphere.argtypes = [vp, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, vp]
    lib.rs_occlusion_mip.restype = ctypes.c_float
    lib.rs_occlusion_mip.argtypes = [vp, ctypes.c_float, ctypes.c_float]
    lib.rs_cone_cull.restype = ctypes.c_int
    lib.rs_cone_cull.argtypes = [vp, ctypes.c_float, vp, ctypes.c_float]
    lib.rs_rotate_quat.argtypes = [vp, vp, vp]
    _LIB = lib
    return lib


def _stand_in_allowed():
    """Without the reference the stand-ins only run inside a test that holds them to the reference's pinned outputs: anywhere
    else they would compare the oracle with itself."""
    if not available() and reference_pins.current is None:
        raise RuntimeError("the reference's shaders are not available (oracle/_ref/librefshader.so or NIAGARA_REFERENCE); their stand-ins only run inside a test pinned by reference_pins")


def _bind_stages(lib):
    cd = ctypes.POINTER(layout.CullData)
    lib.rs_mesh_clusters.restype = ctypes.c_int
    lib.rs_mesh_clusters.argtypes = [vp, cd, ctypes.c_float, ctypes.c_float, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp, ctypes.c_int]
    lib.rs_mesh_payloads.restype = ctypes.c_int
    lib.rs_mesh_payloads.argtypes = [vp, cd, ctypes.c_float, ctypes.c_float, vp, sz, ctypes.c_uint32, vp, sz, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp, vp, vp, ctypes.c_int]
    lib.rs_draw_indexed.restype = ctypes.c_int
    lib.rs_draw_indexed.argtypes = [vp, cd, ctypes.c_float, ctypes.c_float, vp, sz, ctypes.c_uint32, vp, sz, vp, sz, vp, sz, ctypes.c_uint32, ctypes.c_uint32, vp, vp, ctypes.c_int]
    lib.rs_rasterize.restype = ctypes.c_int
    lib.rs_rasterize.argtypes = [vp, vp, vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, vp, vp, ctypes.c_int]


def _p(a):
    return a.ctypes.data_as(vp) if a is not None else None


def _n(a):
    return a.nbytes if a is not None else 0


def _task_commands(p):
    return p.read_task_commands(min(int(p.dccb[1]) * 64, len(p.dcb) // layout.MESHTASKCOMMAND_DTYPE.itemsize))


class RefShaderPath(oracle_lib.OraclePath):
    """OraclePath's surface and buffers, every pass executed by the reference's shaders.  Only the reference's own
    TASK_WGLIMIT / CLUSTER_LIMIT (config.h) exist here; smaller buffers behave like robustBufferAccess.

    Every pass pins what it wrote in an order-independent form (reference_pins): sorted commands, (drawId, meshlet) pairs
    instead of command ids.  Without the reference the oracle runs the pass and must produce the pinned outputs."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        assert self.limits.task_wglimit == layout.TASK_WGLIMIT and self.limits.cluster_limit == layout.CLUSTER_LIMIT
        _stand_in_allowed()
        self.rs = load() if available() else None

    def cull(self, cull_data, late, post_pass=0, task=None):
        task = self.mesh_shading if task is None else task
        if self.rs is None:
            super().cull(cull_data, late, post_pass, task)
        else:
            pd = self._pass_data(cull_data, 1, post_pass)
            s = self.rs.rs_drawcull(ctypes.byref(pd), int(late), int(task), _p(self.draws), _n(self.draws), _p(self.meshes), _n(self.meshes), _p(self.dvb), _n(self.dvb), _p(self.dcb), _n(self.dcb), _p(self.dccb), ctypes.byref(self.hiz), self.threads)
            assert s == 0, s
        cmds = _task_commands(self) if task else self.read_draw_commands(int(self.dccb[0]))
        reference_pins.check("drawcull", self.dvb, self.dccb, oracle_lib.sorted_commands(cmds))

    def render_clusters(self, cull_data, late, post_pass=0, cluster_backface=None):
        if self.rs is None:
            super().render_clusters(cull_data, late, post_pass, cluster_backface)
        else:
            pd = self._pass_data(cull_data, 0, post_pass)
            if cluster_backface is not None:
                pd.clusterBackfaceEnabled = int(cluster_backface)
            s = self.rs.rs_clustercull(ctypes.byref(pd), int(late), _p(self.dcb), _n(self.dcb), _p(self.dccb), _p(self.draws), _n(self.draws), _p(self.meshlets), _n(self.meshlets), _p(self.mvb), _n(self.mvb), _p(self.cib), _n(self.cib), _p(self.ccb), ctypes.byref(self.hiz), self.threads)
            assert s == 0, s
        count = min(int(self.ccb[0]), len(self.cib))
        pad = min((count + 255) // 256 * 256, len(self.cib))
        reference_pins.check("clustercull", self.ccb, self.mvb, oracle_lib.cluster_pairs(self.cib[:count], _task_commands(self)), self.cib[count:pad])

    def task_shading(self, cull_data, late, payloads, emit_counts, post_pass=0, cluster_backface=None):
        if self.rs is None:
            super().task_shading(cull_data, late, payloads, emit_counts, post_pass, cluster_backface)
        else:
            pd = self._pass_data(cull_data, 0, post_pass)
            if cluster_backface is not None:
                pd.clusterBackfaceEnabled = int(cluster_backface)
            s = self.rs.rs_taskcull(ctypes.byref(pd), int(late), _p(self.dcb), _n(self.dcb), _p(self.dccb), _p(self.draws), _n(self.draws), _p(self.meshlets), _n(self.meshlets), _p(self.mvb), _n(self.mvb), _p(payloads), _p(emit_counts), ctypes.byref(self.hiz), self.threads)
            assert s == 0, s
        # one row per command: its fields, its emit count, the meshlet lanes of its payload (command ids are positions in dcb)
        cmds = _task_commands(self)
        n = min(len(cmds), len(emit_counts))
        emit = np.asarray(emit_counts, np.uint32)[:n]
        lanes = np.asarray(payloads, np.uint32).reshape(len(emit_counts), 64)[:n] >> 24
        lanes[np.arange(64)[None, :] >= emit[:, None]] = 0
        rows = np.concatenate([cmds[:n].view(np.uint32).reshape(n, layout.MESHTASKCOMMAND_DTYPE.itemsize // 4), emit[:, None], lanes], 1)
        reference_pins.check("taskcull", self.mvb, rows[np.lexsort(rows.T[::-1])] if n else rows)

    def pyramid(self, depth):
        if self.rs is None:
            super().pyramid(depth)
        else:
            depth = np.ascontiguousarray(depth, dtype=np.float32)
            s = self.rs.rs_depth_pyramid(_p(depth), self.depth_width, self.depth_height, ctypes.byref(self.hiz), self.threads)
            assert s == 0, s
        reference_pins.check("depthreduce", self.pyramid_texels)


def _pin_mesh_outputs(what, cluster_indices, dcb, rec, pos, tri):
    """records (first three words), positions and triangles of the mesh workgroups, in (drawId, meshlet) order of their
    cluster indices: the slot order follows the order of cib / dcb, which the culler's atomics choose"""
    ci = np.asarray(cluster_indices, np.uint32)
    cmds = np.asarray(dcb).view(np.uint8)[: len(dcb) // 20 * 20].view(layout.MESHTASKCOMMAND_DTYPE)
    keys = np.full(len(ci), np.iinfo(np.uint64).max, np.uint64)
    live = ci != 0xFFFFFFFF
    cmd = cmds[ci[live] & 0xFFFFFF]
    keys[live] = (cmd["drawId"].astype(np.uint64) << np.uint64(32)) | (cmd["taskOffset"].astype(np.uint64) + (ci[live] >> 24))
    order = np.argsort(keys, kind="stable")
    reference_pins.check(what, rec[order, :3], pos[order], tri[order])


class MeshStage:
    """meshlet.mesh.glsl (the reference's consumer of cib / ccb / dcb) + a small rasteriser, for end-to-end tests."""

    def __init__(self, path, vertices, meshletdata, projection16, threads=8):
        _stand_in_allowed()
        self.p, self.rs, self.threads = path, load(), threads
        self.vertices = np.ascontiguousarray(vertices)
        self.meshletdata = np.ascontiguousarray(meshletdata, dtype=np.uint32)
        self.projection = np.ascontiguousarray(projection16, dtype=np.float32)

    def run(self, cull_data, cib=None, ccb=None, dcb=None):
        """Runs the mesh stage over (cib, ccb) (default: the path's own buffers).  Returns records[slots, 4]
        (vertexCount, triangleCount, drawId or ~0, 0), positions[slots, 64, 4], triangles[slots, 96, 3]."""
        p = self.p
        cib = p.cib if cib is None else np.ascontiguousarray(cib, dtype=np.uint32)
        ccb = p.ccb if ccb is None else np.ascontiguousarray(ccb, dtype=np.uint32)
        dcb = p.dcb if dcb is None else dcb
        slots = int(ccb[1]) * int(ccb[2]) * int(ccb[3])
        rec = np.zeros((max(slots, 1), 4), np.uint32)
        pos = np.zeros((max(slots, 1), 64, 4), np.float32)
        tri = np.zeros((max(slots, 1), 96, 3), np.uint8)
        pd = p._pass_data(cull_data, 0, 0)
        w, h = p.depth_width, p.depth_height
        s = self.rs.rs_mesh_clusters(_p(self.projection), ctypes.byref(pd), float(w), float(h), _p(dcb), _n(dcb), _p(p.draws), _n(p.draws), _p(p.meshlets), _n(p.meshlets), _p(self.meshletdata), _n(self.meshletdata), _p(self.vertices), _n(self.vertices), _p(cib), _n(cib), _p(ccb), _p(rec), _p(pos), _p(tri), self.threads)
        assert s == 0, s
        _pin_mesh_outputs("mesh stage", cib[:slots], dcb, rec[:slots], pos[:slots], tri[:slots])
        return rec[:slots], pos[:slots], tri[:slots]

    def run_payloads(self, cull_data, payloads, emit_counts, dcb=None):
        """Task-shading mode: the mesh stage (TASK = true) over task payloads.  Returns records (…, command id in column 3),
        positions, triangles with one slot per emitted mesh workgroup, in command order."""
        p = self.p
        dcb = p.dcb if dcb is None else dcb
        ncmd = len(emit_counts)
        emit = np.minimum(np.ascontiguousarray(emit_counts, dtype=np.uint32), 64)
        first = (np.cumsum(emit) - emit).astype(np.uint32)
        slots = int(emit.sum())
        rec = np.zeros((max(slots, 1), 4), np.uint32)
        pos = np.zeros((max(slots, 1), 64, 4), np.float32)
        tri = np.zeros((max(slots, 1), 96, 3), np.uint8)
        payloads = np.ascontiguousarray(payloads, dtype=np.uint32)
        pd = p._pass_data(cull_data, 0, 0)
        s = self.rs.rs_mesh_payloads(_p(self.projection), ctypes.byref(pd), float(p.depth_width), float(p.depth_height), _p(dcb), _n(dcb), ncmd, _p(p.draws), _n(p.draws), _p(p.meshlets), _n(p.meshlets), _p(self.meshletdata), _n(self.meshletdata), _p(self.vertices), _n(self.vertices), _p(payloads), _p(emit), _p(first), _p(rec), _p(pos), _p(tri), self.threads)
        assert s == 0, s
        ci = np.concatenate([payloads[c, : emit[c]] for c in range(ncmd)]) if ncmd else np.zeros(0, np.uint32)
        _pin_mesh_outputs("mesh stage (task payloads)", ci, dcb, rec[:slots], pos[:slots], tri[:slots])
        return rec[:slots], pos[:slots], tri[:slots]

    def rasterize(self, rec, pos, tri, depth):
        s = self.rs.rs_rasterize(_p(pos), _p(tri), _p(rec), len(rec), depth.shape[1], depth.shape[0], _p(depth), None, 0)
        assert s == 0, s

    def owners(self, rec, pos, tri, depth):
        hit = np.zeros(max(len(rec), 1), np.uint8)
        s = self.rs.rs_rasterize(_p(pos), _p(tri), _p(rec), len(rec), depth.shape[1], depth.shape[0], _p(depth), _p(hit), 1)
        assert s == 0, s
        return hit[: len(rec)].astype(bool)


class VertexStage:
    """mesh.vert.glsl (the draw path's consumer of dcb / dccb under vkCmdDrawIndexedIndirectCount) + the same rasteriser."""

    def __init__(self, path, vertices, indices, projection16):
        _stand_in_allowed()
        self.p, self.rs = path, load()
        self.vertices = np.ascontiguousarray(vertices)
        self.indices = np.ascontiguousarray(indices, dtype=np.uint32)
        self.projection = np.ascontiguousarray(projection16, dtype=np.float32)

    def draw(self, cull_data, depth, dcb=None, count=None, owners=False):
        p = self.p
        dcb = p.dcb if dcb is None else dcb
        count = int(p.dccb[0]) if count is None else int(count)
        hit = np.zeros(max(count, 1), np.uint8)
        pd = p._pass_data(cull_data, 0, 0)
        s = self.rs.rs_draw_indexed(_p(self.projection), ctypes.byref(pd), float(p.depth_width), float(p.depth_height), _p(dcb), _n(dcb), count, _p(p.draws), _n(p.draws), _p(self.vertices), _n(self.vertices), _p(self.indices), len(self.indices), depth.shape[1], depth.shape[0], _p(depth), _p(hit), 1 if owners else 0)
        assert s == 0, s
        if owners:  # the draws whose commands own a pixel
            reference_pins.check("vertex stage owners", np.sort(dcb[: count * 24].view(layout.MESHDRAWCOMMAND_DTYPE)["drawId"][hit[:count] != 0]))
        else:
            reference_pins.check("vertex stage depth", depth)
        return hit[:count].astype(bool)
