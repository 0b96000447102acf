#!/usr/bin/env python
"""Converter: the reference checkout's operator fixtures -> the pickle-free tests/golden/smpl_topology.*.npz.

The reference ships its fixed mesh hierarchy as pickled scipy CSC matrices
(<CAPE checkout>/data/transform_matrices/{for_demo,ds2}/{A,D,U}.npy, loaded at lib/load_data.py:7-32 with
encoding='latin1').  The files written here are the copy `cape_b200.topology` reads; they come from the reference's
data/ directory and fall under the reference's licence.  They hold the operators as plain CSR arrays
(indptr/indices/data/shape), the SMPL edge table (data/edges_smpl.npy, used by lib/losses.py:9-25; = upper triangle
of A[0], checked against the reference file), the per-vertex normalisation statistics
(data/demo_data/trainset_stats.npz, demos.py:155), the clothing-vertex index list, the template mesh and the demo
poses (demos.py:349-357), split in the parts of `topology.DATA_PARTS` (each well under 1 MB).

    python -m cape_b200.pack_topology --reference /path/to/CAPE        (default: $CAPE_REFERENCE)
"""
import argparse
import os
import sys
import numpy as np
import scipy.sparse as sp

from cape_b200 import topology


def pack(REF, out_dir=topology.DATA_DIR):
    def _load(kind, name):
        path = os.path.join(REF, "data", "transform_matrices", kind, name + ".npy")
        return list(np.load(path, encoding="latin1", allow_pickle=True))

    out = {}
    for kind in ("for_demo", "ds2"):
        for name in ("A", "D", "U"):
            mats = _load(kind, name)
            out[f"{kind}.{name}.count"] = np.int64(len(mats))
            for i, m in enumerate(mats):
                m = sp.csr_matrix(m)
                m.sort_indices()
                key = f"{kind}.{name}.{i}"
                out[key + ".indptr"] = m.indptr.astype(np.int32)
                out[key + ".indices"] = m.indices.astype(np.int32)
                out[key + ".data"] = m.data  # dtype kept (for_demo fp32, ds2 fp64)
                out[key + ".shape"] = np.asarray(m.shape, np.int64)
    a0 = sp.coo_matrix(_load("for_demo", "A")[0])
    keep = a0.row < a0.col
    edges = np.stack([a0.row[keep], a0.col[keep]], 1).astype(np.int32)
    edges = edges[np.lexsort((edges[:, 1], edges[:, 0]))]
    ref_edges = np.load(os.path.join(REF, "data", "edges_smpl.npy"))
    assert set(map(tuple, edges.tolist())) == set(map(tuple, np.sort(ref_edges, 1).tolist()))
    out["edges"] = edges
    st = np.load(os.path.join(REF, "data", "demo_data", "trainset_stats.npz"))
    out["stats.mean"] = st["mean"].astype(np.float32)
    out["stats.std"] = st["std"].astype(np.float32)
    out["clothing_verts_idx"] = np.load(os.path.join(REF, "data", "clothing_verts_idx.npy")).astype(np.int32)
    # demo assets (demos.py:351-357): template mesh (minimal body shape + faces) and the demo poses
    v, f = [], []
    for ln in open(os.path.join(REF, "data", "template_mesh.obj")):
        t = ln.split()
        if t and t[0] == "v":
            v.append([float(x) for x in t[1:4]])
        elif t and t[0] == "f":
            f.append([int(x.split("/")[0]) - 1 for x in t[1:4]])
    out["template.v"], out["template.f"] = np.asarray(v, np.float64), np.asarray(f, np.int32)
    dp = np.load(os.path.join(REF, "data", "demo_data", "demo_pose_params.npz"))
    out["demo.rot"], out["demo.pose"] = dp["rot"], dp["pose"]
    os.makedirs(out_dir, exist_ok=True)
    part_of = lambda key: key.split(".")[0] if key.split(".")[0] in ("for_demo", "ds2") else "assets"
    files = topology.data_files(out_dir)
    for part, fn in zip(topology.DATA_PARTS, files):
        np.savez_compressed(fn, **{k: v for k, v in out.items() if part_of(k) == part})
    return files


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reference", default=os.environ.get("CAPE_REFERENCE"), help="checkout of qianlim/CAPE")
    ap.add_argument("--out-dir", default=topology.DATA_DIR)
    a = ap.parse_args(argv)
    if not a.reference:
        ap.error("no reference checkout given: pass --reference or set CAPE_REFERENCE")
    for fn in pack(a.reference, a.out_dir):
        print("wrote", os.path.abspath(fn), os.path.getsize(fn), "bytes")


if __name__ == "__main__":
    sys.exit(main())
