"""CPU-only property tests of the three meshopt stream decoders (nvc_decode_vertex_stream / _index_stream /
_meshlet_stream, csrc/nvc_meshopt_decode.cpp + nvc_scene_cache.cpp) against the REFERENCE's vendored codec library
(oracle/_ref/libmeshopt_ref.so: extern/meshoptimizer/src/{vertex,index,meshlet}codec.cpp compiled where they lie):
random and structured inputs are encoded by the reference's encoders (both codec versions, all compression levels)
and decoded by both sides; results must be identical, byte for byte.

Without the reference library the decoders run on a fixed sample of the same cases: the streams the reference's encoders
wrote for them (tests/golden/meshopt_streams.npz, made by tests/golden/make_meshopt_streams.py) and the reference decoder's
outputs, pinned by reference_pins."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import reference_pins
from niagara_b200.lib import load_library
from refshader_lib import REFERENCE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libmeshopt_ref.so")
STREAMS = os.path.join(ROOT, "tests", "golden", "meshopt_streams.npz")

vp, sz = ctypes.c_void_p, ctypes.c_size_t


def load_ref():
    """The reference's codec library, or None where it is neither built nor buildable."""
    if os.path.isdir(os.path.join(REFERENCE, "src")):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + REFERENCE], check=True)
    if not os.path.exists(REF_SO):
        return None
    lib = ctypes.CDLL(REF_SO)
    lib.meshopt_encodeVertexBufferBound.restype = sz
    lib.meshopt_encodeVertexBufferBound.argtypes = [sz, sz]
    lib.meshopt_encodeVertexBufferLevel.restype = sz
    lib.meshopt_encodeVertexBufferLevel.argtypes = [vp, sz, vp, sz, sz, ctypes.c_int, ctypes.c_int]
    lib.meshopt_decodeVertexBuffer.restype = ctypes.c_int
    lib.meshopt_decodeVertexBuffer.argtypes = [vp, sz, sz, vp, sz]
    lib.meshopt_encodeIndexBufferBound.restype = sz
    lib.meshopt_encodeIndexBufferBound.argtypes = [sz, sz]
    lib.meshopt_encodeIndexBuffer.restype = sz
    lib.meshopt_encodeIndexBuffer.argtypes = [vp, sz, vp, sz]
    lib.meshopt_encodeIndexVersion.argtypes = [ctypes.c_int]
    lib.meshopt_decodeIndexBuffer.restype = ctypes.c_int
    lib.meshopt_decodeIndexBuffer.argtypes = [vp, sz, sz, vp, sz]
    lib.meshopt_encodeMeshletBound.restype = sz
    lib.meshopt_encodeMeshletBound.argtypes = [sz, sz]
    lib.meshopt_encodeMeshlet.restype = sz
    lib.meshopt_encodeMeshlet.argtypes = [vp, sz, vp, sz, vp, sz]
    lib.meshopt_decodeMeshlet.restype = ctypes.c_int
    lib.meshopt_decodeMeshlet.argtypes = [vp, sz, sz, vp, sz, sz, vp, sz]
    return lib


@pytest.fixture(scope="module")
def ref():
    return load_ref()


@pytest.fixture(scope="module")
def stored():
    z = np.load(STREAMS)
    ends = np.cumsum(z["sizes"].astype(np.int64))
    return {str(k): z["streams"][e - n : e] for k, n, e in zip(z["keys"], z["sizes"], ends)}


@pytest.fixture(autouse=True)
def _reference_pins(request, ref):
    with reference_pins.pinned(request, ref is not None):
        yield


def _stream(ref, stored, key, encode):
    """The reference's stream for case `key`: encoded now (and equal to the stored copy, if any), or the stored copy;
    None when the reference is absent and the case is not in the stored sample."""
    if ref is None:
        return stored.get(key)
    stream = encode()
    if key in stored:
        assert np.array_equal(stored[key], stream), key
    return stream


def _p(a):
    return a.ctypes.data_as(vp)


def _vertex_data(rng, count, stride, kind):
    if kind == "random":
        return rng.integers(0, 256, (count, stride), dtype=np.uint8)
    if kind == "zeros":
        return np.zeros((count, stride), np.uint8)
    if kind == "smooth16":  # slowly varying 16-bit fields (positions, uvs): 16-bit delta channels
        base = np.cumsum(rng.integers(-40, 41, (count, stride // 2)), axis=0).astype(np.int64) + 30000
        return (base & 0xFFFF).astype("<u2").view(np.uint8).reshape(count, stride)
    if kind == "floats":  # float32 fields with shared exponents: the rotating 32-bit xor channel
        f = (rng.standard_normal((count, stride // 4)) * 0.01 + np.linspace(1, 2, stride // 4)).astype("<f4")
        return f.view(np.uint8).reshape(count, stride)
    if kind == "sparse":  # mostly constant bytes with rare spikes: 1/2/4-bit groups with escapes
        d = np.full((count, stride), 7, np.uint8)
        idx = rng.integers(0, count, max(1, count // 9))
        d[idx, rng.integers(0, stride, len(idx))] = rng.integers(0, 256, len(idx))
        return np.cumsum(d, axis=0).astype(np.uint8)
    raise ValueError(kind)


def vertex_cases(version):
    """(key, data, level) of every vertex codec case, in the order the random inputs are drawn"""
    rng = np.random.default_rng(100 + version)
    for stride in (4, 8, 12, 16, 20, 32, 48, 64, 256):
        for count in (1, 2, 15, 16, 17, 255, 256, 257, 1000, 3000):
            for kind in ("random", "zeros", "smooth16", "floats", "sparse"):
                if stride > 64 and count > 300:
                    continue
                data = np.ascontiguousarray(_vertex_data(rng, count, stride, kind))
                for level in ((0, 1, 2, 3) if version == 1 else (2,)):
                    yield "vertex_v%d_%d_%d_%s_%d" % (version, stride, count, kind, level), data, level


def encode_vertex(ref, data, level, version):
    count, stride = data.shape
    buf = np.zeros(ref.meshopt_encodeVertexBufferBound(count, stride), np.uint8)
    n = ref.meshopt_encodeVertexBufferLevel(_p(buf), len(buf), _p(data), count, stride, level, version)
    assert n > 0
    stream = np.ascontiguousarray(buf[:n])
    want = np.zeros_like(data)
    assert ref.meshopt_decodeVertexBuffer(_p(want), count, stride, _p(stream), n) == 0
    assert np.array_equal(want, data)  # the codec is lossless
    return stream


@pytest.mark.parametrize("version", [0, 1])
def test_vertex_codec_against_reference(ref, stored, version):
    ours = load_library()
    cases = 0
    for key, data, level in vertex_cases(version):
        count, stride = data.shape
        stream = _stream(ref, stored, key, lambda: encode_vertex(ref, data, level, version))
        if stream is None:
            continue
        n = len(stream)
        got = np.full((count + 1, stride), 0xEE, np.uint8)
        assert ours.nvc_decode_vertex_stream(_p(got), count, stride, _p(stream), n) == 0, key
        assert np.array_equal(got[:count], data), key
        assert (got[count] == 0xEE).all()
        # a truncated or extended stream is rejected by both
        assert ours.nvc_decode_vertex_stream(_p(got), count, stride, _p(stream), n - 1) != 0
        cases += 1
    assert cases > (400 if ref is not None else 40)


def _index_data(rng, triangles, kind):
    if kind == "random":
        return rng.integers(0, max(3, triangles), triangles * 3, dtype=np.uint32)
    if kind == "strip":  # cache-friendly strip-like order: edge and vertex FIFO hits, sequential new vertices
        i = np.arange(triangles, dtype=np.uint32)
        return np.stack([i, i + 1, i + 2], 1).reshape(-1)
    if kind == "grid":
        w = 17
        q = np.arange(triangles // 2 + 1, dtype=np.uint32)
        x, y = q % (w - 1), q // (w - 1)
        a, b, c, d = y * w + x, y * w + x + 1, (y + 1) * w + x, (y + 1) * w + x + 1
        return np.stack([a, b, c, c, b, d], 1).reshape(-1)[: triangles * 3].astype(np.uint32)
    if kind == "jumps":  # large index deltas: 5-byte varints, +-1 shortcuts
        base = rng.integers(0, 1 << 31, triangles, dtype=np.int64)
        return np.stack([base, base + rng.integers(-1, 2, triangles), base ^ 0x40000000], 1).reshape(-1).astype(np.uint32)
    raise ValueError(kind)


def index_cases(version):
    rng = np.random.default_rng(200 + version)
    for triangles in (1, 2, 3, 16, 17, 100, 1000, 5000):
        for kind in ("random", "strip", "grid", "jumps"):
            yield "index_v%d_%d_%s" % (version, triangles, kind), np.ascontiguousarray(_index_data(rng, triangles, kind), dtype=np.uint32)


def encode_index(ref, idx, version):
    ref.meshopt_encodeIndexVersion(version)
    try:
        buf = np.zeros(ref.meshopt_encodeIndexBufferBound(len(idx), 0xFFFFFFFF), np.uint8)
        n = ref.meshopt_encodeIndexBuffer(_p(buf), len(buf), _p(idx), len(idx))
    finally:
        ref.meshopt_encodeIndexVersion(1)
    assert n > 0
    return np.ascontiguousarray(buf[:n])


@pytest.mark.parametrize("version", [0, 1])
def test_index_codec_against_reference(ref, stored, version):
    ours = load_library()
    cases = 0
    for key, idx in index_cases(version):
        stream = _stream(ref, stored, key, lambda: encode_index(ref, idx, version))
        if stream is None:
            continue
        n = len(stream)
        assert stream[0] == (0xE0 | version)
        got = np.full(len(idx) + 3, 0xEEEEEEEE, np.uint32)
        assert ours.nvc_decode_index_stream(_p(got), len(idx), _p(stream), n) == 0, key
        if ref is not None:
            want = np.zeros_like(idx)
            assert ref.meshopt_decodeIndexBuffer(_p(want), len(idx), 4, _p(stream), n) == 0
            assert np.array_equal(got[: len(idx)], want), key
        if key in stored:
            reference_pins.check(key, want if ref is not None else got[: len(idx)])
        assert (got[len(idx) :] == 0xEEEEEEEE).all()
        # same triangles as the input, corners possibly rotated
        a, b = idx.reshape(-1, 3), got[: len(idx)].reshape(-1, 3)
        assert ((a == b).all(1) | (np.roll(a, 1, 1) == b).all(1) | (np.roll(a, 2, 1) == b).all(1)).all()
        assert ours.nvc_decode_index_stream(_p(got), len(idx), _p(stream), n - 1) != 0
        cases += 1
    assert cases == (32 if ref is not None else len([k for k in stored if k.startswith("index_v%d_" % version)]))


def meshlet_cases():
    rng = np.random.default_rng(300)
    for case in range(600):
        vc = int(rng.integers(3, 257)) if rng.random() < 0.3 else int(rng.integers(3, 65))
        tc = int(rng.integers(1, 257)) if rng.random() < 0.3 else int(rng.integers(1, 97))
        style = rng.integers(0, 4)
        if style == 0:  # arbitrary references, arbitrary triangles
            refs = rng.integers(0, 1 << 32, vc, dtype=np.uint64).astype(np.uint32)
            tris = rng.integers(0, vc, (tc, 3)).astype(np.uint8)
        elif style == 1:  # ascending references with small gaps, strip-like triangles (edge reuse, next-vertex codes)
            refs = (np.cumsum(rng.integers(1, 4, vc)) + 1000).astype(np.uint32)
            i = np.arange(tc) % max(1, vc - 2)
            tris = np.stack([i, i + 1, i + 2], 1).astype(np.uint8)
        elif style == 2:  # 16-bit references (shortRefs), fans
            refs = rng.integers(0, 1 << 16, vc).astype(np.uint32)
            i = 1 + np.arange(tc) % max(1, vc - 2)
            tris = np.stack([np.zeros(tc, np.int64), i, i + 1], 1).astype(np.uint8)
        else:  # large deltas: 3- and 4-byte groups
            refs = (rng.integers(0, 1 << 24, vc) * rng.integers(1, 200, vc)).astype(np.uint32)
            tris = rng.integers(0, vc, (tc, 3)).astype(np.uint8)
        yield "meshlet_%d" % case, np.ascontiguousarray(refs), np.ascontiguousarray(tris), style


def encode_meshlet(ref, refs, tris):
    buf = np.zeros(ref.meshopt_encodeMeshletBound(256, 256), np.uint8)
    n = ref.meshopt_encodeMeshlet(_p(buf), len(buf), _p(refs), len(refs), _p(tris), len(tris))
    assert n > 0
    return np.ascontiguousarray(buf[:n])


def test_meshlet_codec_against_reference(ref, stored):
    ours = load_library()
    cases = 0
    for key, refs, tris, style in meshlet_cases():
        vc, tc = len(refs), len(tris)
        stream = _stream(ref, stored, key, lambda: encode_meshlet(ref, refs, tris))
        if stream is None:
            continue
        n = len(stream)
        for ref_size in ((2, 4) if int(refs.max()) < (1 << 16) else (4,)):
            got_r = np.full(vc + 2, 0xEE, np.uint16 if ref_size == 2 else np.uint32)
            got_t = np.full((tc + 2) * 3 + 4, 0xEE, np.uint8)
            assert ours.nvc_decode_meshlet_stream(_p(got_r), vc, ref_size, _p(got_t), tc, _p(stream), n) == 0, (vc, tc, style)
            if ref is not None:
                want_r = np.zeros(vc + 2, got_r.dtype)
                want_t = np.zeros((tc + 2) * 3 + 4, np.uint8)
                assert ref.meshopt_decodeMeshlet(_p(want_r), vc, ref_size, _p(want_t), tc, 3, _p(stream), n) == 0
                assert np.array_equal(got_r[:vc], want_r[:vc])
                assert np.array_equal(got_t[: tc * 3], want_t[: tc * 3]), (vc, tc, style)
            if key in stored:
                reference_pins.check("%s ref_size %d" % (key, ref_size), *((want_r[:vc], want_t[: tc * 3]) if ref is not None else (got_r[:vc], got_t[: tc * 3])))
            assert np.array_equal(got_r[:vc].astype(np.uint32), refs.astype(got_r.dtype).astype(np.uint32))
            assert (got_t[tc * 3 :] == 0xEE).all() and (got_r[vc:] == 0xEE).all()  # nothing written past the outputs
            a, b = tris.reshape(-1, 3), got_t[: tc * 3].reshape(-1, 3)
            assert ((a == b).all(1) | (np.roll(a, 1, 1) == b).all(1) | (np.roll(a, 2, 1) == b).all(1)).all()
            cases += 1
        # (a meshlet block carries no length of its own — it is parsed from its end — so a truncated block may still be a valid one)
        assert ours.nvc_decode_meshlet_stream(_p(got_r), vc, 4 if got_r.dtype == np.uint32 else 2, _p(got_t), tc, _p(stream), n - 1) in (0, -7)
    assert cases >= (600 if ref is not None else 100)
