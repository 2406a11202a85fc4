#!/usr/bin/env python
"""Regenerates tests/golden/meshopt_streams.npz: the streams the reference's vendored meshoptimizer encoders write for a
fixed sample of the cases of tests/test_meshopt_decoders.py, so that the product's decoders are checked against them where
the reference is absent.  The sample takes, per codec and version, the cases whose streams are at most LIMIT bytes (every
input kind and shape up to that size).  Needs the reference (oracle/_ref/libmeshopt_ref.so, built by `make -C oracle ref`).

    python tests/golden/make_meshopt_streams.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LIMIT = {"vertex": 256, "index": 1024, "meshlet": 160}


def main():
    import test_meshopt_decoders as t

    ref = t.load_ref()
    assert ref is not None, "needs the reference's codecs (make -C oracle ref)"
    out = {}
    for version in (0, 1):
        for key, data, level in t.vertex_cases(version):
            out[key] = t.encode_vertex(ref, data, level, version)
        for key, idx in t.index_cases(version):
            out[key] = t.encode_index(ref, idx, version)
    for key, refs, tris, _ in t.meshlet_cases():
        out[key] = t.encode_meshlet(ref, refs, tris)
    keep = {k: v for k, v in out.items() if len(v) <= LIMIT[k.split("_")[0]]}
    path = os.path.join(ROOT, "tests", "golden", "meshopt_streams.npz")
    keys = sorted(keep)
    np.savez_compressed(path, keys=np.array(keys), sizes=np.array([len(keep[k]) for k in keys], np.uint32), streams=np.concatenate([keep[k] for k in keys]))
    for codec in LIMIT:
        n = [k for k in keep if k.startswith(codec)]
        print(codec, "%d of %d cases, %d bytes" % (len(n), len([k for k in out if k.startswith(codec)]), sum(len(keep[k]) for k in n)))
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
