"""Pins the kNN / vertex-append rows of the oracle (SURVEY 8a a13-a15) to the REFERENCE's own ikd-Tree: the oracle against
tests/golden/ikd_*.npz, generated from include/ikd-Tree/ikd_Tree.cpp compiled unmodified (oracle/Makefile.ref) by
tools/make_golden.py.  The CUDA path is checked against the same fixtures in tests/test_mesh_gpu.py."""
import os

import numpy as np

import oracle_api as oa
import ref_ikd
from immesh_b200 import api, synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _oracle_with_frames(frames, pose_t, cfg):
    o = oa.OracleMesh(cfg)
    for k, f in enumerate(frames):
        o.push_frame(f, pose_t[k], k)
    return o


def test_golden_append_matches_oracle():
    g = np.load(os.path.join(GOLD, "ikd_append.npz"))
    cfg = api.MeshConfig()
    assert float(g["xi"]) == cfg.points_minimum_scale and float(g["res"]) == cfg.voxel_resolution
    frames = [g[f"frame{k}"] for k in range(3)]
    o = _oracle_with_frames(frames, g["pose_t"], cfg)
    v, _, _ = o.snapshot()
    assert v.shape == g["verts"].shape and np.array_equal(v, g["verts"])        # ids = append order, positions bit-exact


def test_golden_knn_matches_oracle():
    g = np.load(os.path.join(GOLD, "ikd_knn.npz"))
    ga = np.load(os.path.join(GOLD, "ikd_append.npz"))
    o = _oracle_with_frames([ga[f"frame{k}"] for k in range(3)], ga["pose_t"], api.MeshConfig())
    for c, (k, md) in enumerate(g["cases"]):
        idx, d2 = o.knn(g["queries"], int(k), float(md))
        assert ref_ikd.same_knn(idx.astype(np.int64), d2, g[f"idx{c}"].astype(np.int64), g[f"d2{c}"]), (k, md)


def test_oracle_knn_matches_reference_ikdtree_incremental():
    """The tree grown frame by frame with the oracle's new vertices, queried after every frame."""
    g = np.load(os.path.join(GOLD, "ikd_incremental.npz"))
    sensor, scans = synth.make_stream("avia", 4, seed=11, n_points=12000)
    frames = [(s["body_full"].astype(np.float64) @ s["R_true"].T + s["t_true"]).astype(np.float32) for s in scans]
    o = oa.OracleMesh(api.MeshConfig())
    for k, f in enumerate(frames):
        o.push_frame(f, scans[k]["t_true"], k)
        v, _, _ = o.snapshot()
        assert len(v) == int(g[f"n_vertices{k}"]), k       # the vertex set the reference tree was grown with
        for c, (kk, md) in enumerate(g["cases"]):
            io, do = o.knn(g[f"queries{k}"], int(kk), float(md))
            assert ref_ikd.same_knn(io.astype(np.int64), do, g[f"idx{k}_{c}"].astype(np.int64), g[f"d2{k}_{c}"]), (k, kk, md)


def test_oracle_append_matches_reference_ikdtree_driven_loop():
    """The append loop with the reference tree answering its 1-NN queries (tools/make_golden.py append_with_tree)."""
    ref = np.load(os.path.join(GOLD, "ikd_loop.npz"))["verts"]
    cfg = api.MeshConfig()
    sensor, scans = synth.make_stream("avia", 3, seed=4, n_points=4000)
    frames = [(s["body_full"].astype(np.float64) @ s["R_true"].T + s["t_true"]).astype(np.float32) for s in scans]
    o = _oracle_with_frames(frames, [s["t_true"] for s in scans], cfg)
    v, _, _ = o.snapshot()
    assert v.shape == ref.shape and np.array_equal(v, ref)
