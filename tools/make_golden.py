#!/usr/bin/env python
"""Generates tests/golden/ikd_*.npz from the REFERENCE's own ikd-Tree (oracle/_ref/libref_ikd.so, built from
include/ikd-Tree of an ImMesh checkout by oracle/Makefile.ref):

    python tools/make_golden.py <path to an ImMesh checkout> [output directory, default tests/golden]

Fixtures (inputs + reference outputs), consumed by tests/test_ref_ikd.py (oracle, CPU) and tests/test_mesh_gpu.py (CUDA):
  ikd_knn.npz          vertices (insertion order), queries, Nearest_Search results for (k, max_dist) in CASES
  ikd_append.npz       three world-frame frames (sub-sampled) and the vertex list produced by the reference's append loop
                       (pointcloud_rgbd.cpp:411-552: xi-grid test, ikd-Tree 1-NN test, Add_Point) driven with the real tree
  ikd_incremental.npz  the tree grown frame by frame with the oracle mesher's new vertices (Add_Point, the tree re-balances
                       itself): per frame the vertex count and Nearest_Search results for every sixteenth of the random queries
  ikd_loop.npz         the vertex list of the append loop driven with the real tree on a second stream
  ikd_mesh_knn.npz     Nearest_Search over the vertices of three meshed frames (the same on the oracle and the CUDA mesher),
                       every sixteenth of the random queries
The streams are regenerated from their seeds by immesh_b200.synth; the vertex counts stored with them pin that they are the
streams the reference tree saw.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_ikd  # noqa: E402
from immesh_b200 import api, synth  # noqa: E402

CASES = [(20, float("inf")), (1, 0.1), (20, 1.0), (5, 0.3), (32, 0.75)]
INCREMENTAL_CASES = [(20, float("inf")), (1, 0.1), (20, 1.0), (5, 0.3)]
MESH_KNN_CASES = [(20, float("inf")), (1, 0.1), (20, 1.0)]


def world_frames(scans):
    return [(s["body_full"].astype(np.float64) @ s["R_true"].T + s["t_true"]).astype(np.float32) for s in scans]


def append_with_tree(frames, xi, target, tree=None):
    """Global_map::append_points_to_global_map (pointcloud_rgbd.cpp:411-552) with the kd-tree queries answered by `tree`."""
    tree = tree or ref_ikd.RefIkdTree()
    verts, grid = [], set()
    for pts in frames:
        step = max(1, round(len(pts) // target))
        for i in range(0, len(pts), step):
            p = pts[i]
            g = tuple(int(np.round(np.float64(p[j]) / xi)) for j in range(3))
            if g in grid:
                continue
            if verts:
                idx, d2, cnt = tree.knn(p[None, :], 1)
                if cnt[0] and np.sqrt(d2[0, 0]) < xi:
                    continue
            grid.add(g)
            verts.append(p.copy())
            tree.add(p[None, :])
    return np.asarray(verts, dtype=np.float32)


def incremental_fixture():
    import oracle_api as oa
    sensor, scans = synth.make_stream("avia", 4, seed=11, n_points=12000)
    o, t, n_prev = oa.OracleMesh(api.MeshConfig()), ref_ikd.RefIkdTree(), 0
    rng = np.random.default_rng(5)
    d = {"cases": np.array(INCREMENTAL_CASES)}
    for k, f in enumerate(world_frames(scans)):
        o.push_frame(f, scans[k]["t_true"], k)
        v, _, _ = o.snapshot()
        t.add(v[n_prev:])            # Add_Point per accepted vertex, as pointcloud_rgbd.cpp:540
        n_prev = len(v)
        q = (v[rng.integers(0, len(v), 1500)] + rng.normal(0, 0.15, (1500, 3))).astype(np.float32)[::16]
        d[f"n_vertices{k}"], d[f"queries{k}"] = np.int64(n_prev), q
        for c, (kk, md) in enumerate(INCREMENTAL_CASES):
            idx, d2, _ = t.knn(q, kk, md)
            d[f"idx{k}_{c}"], d[f"d2{k}_{c}"] = idx.astype(np.int32), d2
    return d


def loop_fixture():
    cfg = api.MeshConfig()
    sensor, scans = synth.make_stream("avia", 3, seed=4, n_points=4000)
    return {"verts": append_with_tree(world_frames(scans), cfg.points_minimum_scale, cfg.number_of_pts_append_to_map)}


def mesh_knn_fixture():
    import oracle_api as oa
    from mesh_common import SMALL, world_scans
    o = oa.OracleMesh(api.MeshConfig(**SMALL))
    for k, (world, t) in enumerate(world_scans("avia", 3, 9)):
        o.push_frame(world, t, k)
    v = o.snapshot()[0]
    tree = ref_ikd.RefIkdTree()
    tree.add(v)
    rng = np.random.default_rng(1)
    q = (v[rng.integers(0, len(v), 4000)] + rng.normal(0, 0.2, (4000, 3))).astype(np.float32)[::16]
    d = {"n_vertices": np.int64(len(v)), "queries": q, "cases": np.array(MESH_KNN_CASES)}
    for c, (k, md) in enumerate(MESH_KNN_CASES):
        idx, d2, _ = tree.knn(q, k, md)
        d[f"idx{c}"], d[f"d2{c}"] = idx.astype(np.int32), d2
    return d


def main(ref_dir, out):
    ref_ikd.build(ref_dir)
    os.makedirs(out, exist_ok=True)
    cfg = api.MeshConfig()
    sensor, scans = synth.make_stream("avia", 3, seed=21, n_points=5000)
    frames = world_frames(scans)
    tree = ref_ikd.RefIkdTree()
    verts = append_with_tree(frames, cfg.points_minimum_scale, cfg.number_of_pts_append_to_map, tree)
    np.savez_compressed(os.path.join(out, "ikd_append.npz"), **{f"frame{k}": f for k, f in enumerate(frames)},
                        pose_t=np.stack([s["t_true"] for s in scans]), verts=verts, xi=cfg.points_minimum_scale,
                        res=cfg.voxel_resolution, target=cfg.number_of_pts_append_to_map)
    rng = np.random.default_rng(3)
    q = (verts[rng.integers(0, len(verts), 192)] + rng.normal(0, 0.15, (192, 3))).astype(np.float32)
    q = np.concatenate([q, verts[:32], (verts[:32] + np.float32(50.0))]).astype(np.float32)   # exact hits and far misses
    d = {"verts": verts, "queries": q, "cases": np.array(CASES)}
    for c, (k, md) in enumerate(CASES):
        idx, d2, cnt = tree.knn(q, k, md)
        d[f"idx{c}"], d[f"d2{c}"], d[f"cnt{c}"] = idx.astype(np.int32), d2, cnt
    np.savez_compressed(os.path.join(out, "ikd_knn.npz"), **d)
    np.savez_compressed(os.path.join(out, "ikd_incremental.npz"), **incremental_fixture())
    np.savez_compressed(os.path.join(out, "ikd_loop.npz"), **loop_fixture())
    np.savez_compressed(os.path.join(out, "ikd_mesh_knn.npz"), **mesh_knn_fixture())
    print("wrote", sorted(os.listdir(out)), "to", out)


if __name__ == "__main__":
    if len(sys.argv) not in (2, 3):
        sys.exit(__doc__)
    main(sys.argv[1], sys.argv[2] if len(sys.argv) == 3 else os.path.join(ROOT, "tests", "golden"))
