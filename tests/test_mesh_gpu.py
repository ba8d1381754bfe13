"""GPU tier: the CUDA mesher through the C ABI against the oracle (vertex ids, facet connectivity, flags: bit-exact)."""
import numpy as np
import pytest

from immesh_b200 import api
from mesh_common import run_mesh_parity, world_scans, SMALL
from oracle_api import OracleMesh

pytestmark = pytest.mark.gpu


def test_avia_frames_bit_exact(cuda_lib):
    g, o, stats = run_mesh_parity(cuda_lib, "avia", 8, seed=0)
    assert stats[-1]["n_triangles"] > 10000 and stats[-1]["frame_removed"] > 0


def test_hdl64_frames_bit_exact(cuda_lib):
    run_mesh_parity(cuda_lib, "hdl64", 4, seed=2)


def test_step_one_dense_append(cuda_lib):
    run_mesh_parity(cuda_lib, "avia", 3, seed=4, n_points=9000)


def test_knn_matches_oracle(cuda_lib):
    g, o, _ = run_mesh_parity(cuda_lib, "avia", 3, seed=6)
    v, _, _ = o.snapshot()
    rng = np.random.default_rng(0)
    q = np.concatenate([v[rng.integers(0, len(v), 300)] + rng.normal(0, 0.05, (300, 3)).astype(np.float32),
                        v[:100], rng.uniform(-50, 50, (50, 3)).astype(np.float32)]).astype(np.float32)
    for k, md in ((1, np.inf), (20, np.inf), (20, 1.0), (5, 0.3)):
        ig, dg = g.knn(q, k, md)
        io, do = o.knn(q, k, md)
        assert np.array_equal(ig, io), (k, md)
        assert np.array_equal(dg, do), (k, md)


def _golden(name):
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name))


def test_golden_reference_ikdtree_append_and_knn(cuda_lib):
    """CUDA vertex append + kNN against fixtures produced by the REFERENCE's own ikd-Tree (tools/make_golden.py)."""
    import ref_ikd
    ga, gk = _golden("ikd_append.npz"), _golden("ikd_knn.npz")
    g = api.Mesh(api.MeshConfig(), lib=cuda_lib)
    for k in range(3):
        g.push_frame(ga[f"frame{k}"], ga["pose_t"][k], k)
    v = g.snapshot()[0]
    assert v.shape == ga["verts"].shape and np.array_equal(v, ga["verts"])
    for c, (k, md) in enumerate(gk["cases"]):
        idx, d2 = g.knn(gk["queries"], int(k), float(md))
        assert ref_ikd.same_knn(idx.astype(np.int64), d2, gk[f"idx{c}"].astype(np.int64), gk[f"d2{c}"]), (k, md)


def test_knn_matches_reference_ikdtree_live(cuda_lib):
    """CUDA kNN over the vertices of three meshed frames against the reference ikd-Tree built on the same vertices
    (tests/golden/ikd_mesh_knn.npz, tools/make_golden.py)."""
    import ref_ikd
    gk = _golden("ikd_mesh_knn.npz")
    g, o, _ = run_mesh_parity(cuda_lib, "avia", 3, seed=9)
    assert g.counts()["n_vertices"] == int(gk["n_vertices"])
    for c, (k, md) in enumerate(gk["cases"]):
        ig, dg = g.knn(gk["queries"], int(k), float(md))
        assert ref_ikd.same_knn(ig.astype(np.int64), dg, gk[f"idx{c}"].astype(np.int64), gk[f"d2{c}"]), (k, md)


def test_empty_frame_and_restart(cuda_lib):
    cfg = api.MeshConfig(**SMALL)
    g = api.Mesh(cfg, lib=cuda_lib)
    g.push_frame(np.zeros((0, 3), np.float32), np.zeros(3), 0)
    assert g.counts()["n_vertices"] == 0
    pts = np.array([[1.0, 0, 0], [1.1, 0.1, 0], [1.0, 0.15, 0.05]], np.float32)   # one 0.4 m voxel, three xi-cells
    g.push_frame(pts, np.zeros(3), 1)
    c = g.counts()
    assert c["n_vertices"] == 3 and c["n_triangles"] == 1


def test_pipelined_equals_sequential(cuda_lib):
    """LIO(k+1) overlapped with mesh(k) on two streams must give exactly the results of the blocking calls."""
    from immesh_b200 import synth
    from lio_common import init_velocity
    cfg = api.AVIA
    sensor, scans = synth.make_stream("avia", 7, seed=8, ext_T=cfg.ext_T)
    res = []
    for mode in ("sync", "async"):
        lio, mesh = api.Lio(cfg, lib=cuda_lib), api.Mesh(api.MeshConfig(**SMALL), lib=cuda_lib)
        lio.set_pose(scans[0]["R_true"], scans[0]["t_true"])
        init_velocity(lio, sensor, scans)
        lio.voxel_map_init(scans[0]["body_full"])
        for k in range(1, 7):
            if mode == "sync":
                lio.step(scans[k]["body_ds"], scans[k]["dt"])
                mesh.push_frame_from_lio(lio, scans[k]["body_full"])
            else:
                lio.step_async(scans[k]["body_ds"], dt=scans[k]["dt"])
                mesh.push_frame_from_lio_async(lio, scans[k]["body_full"])
        if mode == "async":
            lio.wait()
            mesh.wait()
        res.append((lio.get_state(), lio.dump_map(), mesh.snapshot()))
    assert np.array_equal(res[0][0], res[1][0])
    assert np.array_equal(res[0][1], res[1][1])
    for a, b in zip(res[0][2], res[1][2]):
        assert np.array_equal(a, b)
    assert len(res[0][2][1]) > 1000


def test_smooth_all_pts_and_region_stream(cuda_lib):
    """smooth_all_pts (mesh_rec_geometry.cpp:60-69 -> Global_map::smooth_pts, pointcloud_rgbd.cpp:932-958) and the viewer's
    region-bucketed triangle sets (triangle.cpp:35-53) on the device against the oracle."""
    g, o, _ = run_mesh_parity(cuda_lib, "avia", 4, seed=14)
    for sf, k in ((0.1, 20), (0.5, 8)):
        sg, so = g.smooth_all(sf, k), o.smooth_all(sf, k)
        assert sg.shape == so.shape and len(sg) > 3000
        same = (sg == so) | (np.isnan(sg) & np.isnan(so))      # a vertex without a neighbour inside the limit divides by zero on both sides
        assert same.all()
    keys, offs, tris = g.region_stream(10.0)
    _, to, _ = o.snapshot()
    ko = o.region_keys(10.0)
    assert len(ko) == len(to) == len(tris)
    order = np.lexsort((to[:, 2], to[:, 1], to[:, 0], ko[:, 2], ko[:, 1], ko[:, 0]))
    assert np.array_equal(tris, to[order])
    ref_keys, first = np.unique(ko[order], axis=0, return_index=True)
    assert np.array_equal(keys, ref_keys) and np.array_equal(offs[:-1], np.sort(first)) and offs[-1] == len(to)
    assert len(keys) >= 2
    # a finer region size
    keys2, offs2, tris2 = g.region_stream(2.0)
    assert len(keys2) > len(keys) and offs2[-1] == len(to)


def test_offline_reconstruct_from_pointcloud(cuda_lib):
    """reconstruct_mesh_from_pointcloud (ImMesh_mesh_reconstruction.cpp:328-345): whole cloud -> VoxelGrid(minimum_pts_distance) -> one frame,
    identity pose, against the same two oracle steps."""
    import oracle_api as oa
    from oracle_api import OracleMesh
    clouds = [w for w, _ in world_scans("avia", 3, seed=15)]
    cloud = np.concatenate(clouds, axis=0)
    cfg = api.MeshConfig(**{**SMALL, "number_of_pts_append_to_map": 1 << 30})     # offline_pointcloud.yaml: every point is an append candidate
    g, o = api.Mesh(cfg, lib=cuda_lib), OracleMesh(cfg)
    vg = api.VoxelGrid(1 << 18, lib=cuda_lib)
    m = g.reconstruct_from_pointcloud(vg, cloud, 0.1)
    ds, small, _ = oa.voxel_grid(cloud, 0.1)
    assert m == len(ds) and not small
    o.push_frame(ds, np.zeros(3), 0)
    assert g.counts() == o.counts()
    for a, b in zip(g.snapshot(), o.snapshot()):
        assert np.array_equal(a, b)
    assert g.counts()["n_triangles"] > 5000


def test_depth_rasterisation_of_the_mesh(cuda_lib):
    """immesh_mesh_render_depth (the reference's depth view of the mesh, ImMesh_node.cpp:305-329 / openGL_camera_view.cpp:316-418, as a CUDA
    rasteriser) against the oracle's rasteriser with the same sampling rule: depth image and unprojected points identical; and a
    geometric sanity check -- every unprojected point lies on the mesh surface it was rendered from (within the local facet size)."""
    from lio_common import init_velocity  # noqa: F401
    from immesh_b200 import synth
    g, o, _ = run_mesh_parity(cuda_lib, "avia", 4, seed=16)
    sensor, scans = synth.make_stream("avia", 4, seed=16)
    Rw, tw = scans[3]["R_true"], scans[3]["t_true"]
    # Cam_view convention: world = R diag(1,-1,-1) p_cam + t with p_cam in the x-right / y-down / z-forward camera frame.  The sensor looks
    # along body +x: camera z = body x, camera x = -body y, camera y = -body z.
    body_from_cam = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
    cam_R = Rw @ body_from_cam @ np.diag([1.0, -1.0, -1.0])
    K = (300.0, 300.0, 319.5, 239.5)
    dg, pg, xg = g.render_depth(K, 640, 480, 0.5, 100.0, cam_R, tw)
    do, po, xo = o.render_depth(K, 640, 480, 0.5, 100.0, cam_R, tw)
    assert np.array_equal(dg, do)
    assert np.array_equal(xg, xo) and np.array_equal(pg, po)
    valid = dg >= 0
    assert valid.sum() > 20000 and dg[valid].min() > 0.5 and dg[valid].max() < 99.0
    # unprojected points are close to mesh vertices (the facets are a few decimetres wide)
    v = g.snapshot()[0]
    idx, d2 = g.knn(pg[::50], 1)
    dist = np.sqrt(d2[:, 0])
    assert np.median(dist) < 0.3 and np.percentile(dist, 99) < 1.5
