"""Host-side mesh ingestion (sph_taichi_b200/voxelizer.py): restatement of the reference's trimesh pipeline
(particle_system.py:421-447).  trimesh is not available offline, so the checks are geometric."""
import os
import tempfile

import numpy as np

from sph_taichi_b200 import voxelizer as vx

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _box_mesh(lo, hi):
    lo, hi = np.asarray(lo, float), np.asarray(hi, float)
    v = np.array([[x, y, z] for x in (lo[0], hi[0]) for y in (lo[1], hi[1]) for z in (lo[2], hi[2])])
    f = np.array([[0, 1, 3], [0, 3, 2], [4, 6, 7], [4, 7, 5], [0, 4, 5], [0, 5, 1],
                  [2, 3, 7], [2, 7, 6], [0, 2, 6], [0, 6, 4], [1, 5, 7], [1, 7, 3]])
    return v, f


def test_box_is_filled_solid():
    pitch = 0.02
    v, f = _box_mesh([0.1, 0.2, 0.3], [0.3, 0.32, 0.5])
    idx = vx.voxelize_solid(v, f, pitch)
    want = [int(round(a / pitch)) for a in (0.1, 0.2, 0.3)], [int(round(a / pitch)) for a in (0.3, 0.32, 0.5)]
    n = [hi - lo + 1 for lo, hi in zip(*want)]
    assert idx.shape == (n[0] * n[1] * n[2], 3)            # surface + interior, every lattice site once
    assert idx.min(0).tolist() == want[0] and idx.max(0).tolist() == want[1]
    assert len(np.unique(idx, axis=0)) == len(idx)
    # the surface alone is hollow
    surf = vx.surface_lattice(v, f, pitch)
    assert len(surf) == n[0] * n[1] * n[2] - (n[0] - 2) * (n[1] - 2) * (n[2] - 2)


def test_subdivision_is_dense_enough():
    """One big triangle: every lattice site its plane passes must be hit (edge <= pitch / 2 after splitting)."""
    pitch = 0.02
    v = np.array([[0.0, 0.0, 0.1], [0.5, 0.0, 0.1], [0.0, 0.4, 0.1]])
    surf = vx.surface_lattice(v, np.array([[0, 1, 2]]), pitch)
    assert (surf[:, 2] == 5).all()
    ii, jj = np.meshgrid(np.arange(0, 26), np.arange(0, 21), indexing="ij")
    inside = (ii * pitch / 0.5 + jj * pitch / 0.4) <= 1.0 - 1e-9
    have = set(map(tuple, surf[:, :2]))
    missing = [(a, b) for a, b in zip(ii[inside], jj[inside]) if (a, b) not in have]
    assert not missing, missing[:5]


def test_transform_order_scale_rotate_about_mean_translate():
    v, _ = _box_mesh([-1, -1, -1], [1, 2, 1])
    out = vx.transform_rigid_mesh(v, [0.5, 0.5, 0.5], 180, [0, 1, 0], [4.0, 2.0, 1.2])
    c = (v * 0.5).mean(0)
    # 180 degrees about y through the vertex mean (pi taken as 3.1415926 like the reference): x, z mirrored
    want = np.stack([2 * c[0] - v[:, 0] * 0.5, v[:, 1] * 0.5, 2 * c[2] - v[:, 2] * 0.5], axis=1) + [4.0, 2.0, 1.2]
    assert np.allclose(out, want, atol=1e-6)
    R = vx.rotation_about_point(0.7, [0, 0, 2], [1, 2, 3])
    assert np.allclose(R[:3, :3] @ R[:3, :3].T, np.eye(3), atol=1e-12)
    assert np.allclose(R[:3, :3] @ [1, 2, 3] + R[:3, 3], [1, 2, 3])  # the pivot is fixed


def test_obj_reader_and_fixture_fallback():
    from sph_taichi_b200 import SimConfig, scene
    v, f = _box_mesh([0, 0, 0], [0.1, 0.1, 0.1])
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "box.obj")
        with open(path, "w") as fh:
            fh.write("# comment\nvt 0 0\n")
            for p in v:
                fh.write(f"v {p[0]} {p[1]} {p[2]}\n")
            fh.write("f 1/1 2/1 4/1 3/1\n")          # a quad with texture indices -> two triangles
            for t in f[2:]:
                fh.write(f"f {t[0] + 1} {t[1] + 1} {t[2] + 1}\n")
        rv, rf = vx.load_obj(path)
        assert rv.shape == (8, 3) and rf.shape == (12, 3) and rf.min() == 0
        sc = scene.dam_break_box([2, 2, 2], domain_end=[1, 1, 1], start=[0.1, 0.1, 0.1])
        sc["RigidBodies"] = [{"objectId": 1, "geometryFile": path, "translation": [0.5, 0.5, 0.5], "rotationAxis": [0, 1, 0],
                              "rotationAngle": 0, "scale": [1, 1, 1], "velocity": [0, 0, 0], "density": 500.0,
                              "color": [1, 2, 3], "isDynamic": True}]
        arrays, coll, rigid_ids, counts = scene.assemble_particles(SimConfig(sc), 3, 0.02)
        assert counts["fluid"] == 8 and counts["solid"] == 6 ** 3 and rigid_ids == {1}
        assert coll[1]["restPosition"].shape == (8, 3)
        solid = arrays["material"] == 0
        assert np.allclose(arrays["x"][solid].min(0), 0.5, atol=1e-6) and (arrays["density"][solid] == 500).all()
    # the committed fixture is used when the mesh file is absent (GPU box)
    arrays, coll, _, counts = scene.assemble_particles(SimConfig(scene.dragon_bath()), 3, 0.02)
    assert counts["solid"] == 18496 and "restPosition" not in coll[1]


def test_named_scenes_match_the_reference_scene_files():
    """Scene ingestion fidelity (SURVEY section 8f rank 3): every scene file the reference ships has a named
    scene with identical configuration, fluid blocks and rigid bodies (ours add `voxelizedPointsFile`, the
    committed voxel fixture used when the mesh file is not on disk).  The reference's scene files are stored
    in tests/golden/reference_scenes/ (tests/golden/make_reference_samples.py)."""
    import json
    import os
    from sph_taichi_b200 import scene
    ref = os.path.join(GOLD, "reference_scenes")
    files = sorted(f for f in os.listdir(ref) if f.endswith(".json"))
    assert len(files) >= 7
    for f in files:
        name = f[:-5]
        assert name in scene.NAMED_SCENES, name
        want = json.load(open(os.path.join(ref, f)))
        got = json.loads(json.dumps(scene.NAMED_SCENES[name]()))
        assert got["Configuration"] == want["Configuration"], name
        for key in ("FluidBlocks", "RigidBodies", "RigidBlocks"):
            a, b = want.get(key, []), got.get(key, [])
            assert len(a) == len(b), (name, key)
            for x, y in zip(a, b):
                y = {k: v for k, v in y.items() if k != "voxelizedPointsFile"}
                assert x == y, (name, key)


def test_obj_vertex_multiplicity_follows_trimesh():
    """trimesh keeps one copy of a vertex per distinct (uv, normal) value it is used with and drops unreferenced
    vertices; the rotation pivot and the rest centre of mass of the reference are the mean over THOSE vertices
    (particle_system.py:428, 436).  A seam vertex counts twice; both meshes the reference ships have weight 1
    everywhere, so for them the plain mean is the trimesh mean (and the committed fixtures stay valid)."""
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "seam.obj")
        with open(path, "w") as fh:
            fh.write("v 0 0 0\nv 1 0 0\nv 0 1 0\nv 1 1 0\nv 9 9 9\n")          # vertex 5 is unreferenced
            fh.write("vt 0 0\nvt 1 0\nvt 0 1\nvt 0.5 0.5\n")
            fh.write("f 1/1 2/2 3/3\nf 2/4 4/1 3/3\n")                           # vertex 2 is used with two uv values
        v, f, w = vx.load_obj(path, with_multiplicity=True)
        assert f.shape == (2, 3) and list(w) == [1, 2, 1, 1, 0]
        assert np.allclose(vx.vertex_mean(v, w), (v[0] + 2 * v[1] + v[2] + v[3]) / 5)
        moved = vx.transform_rigid_mesh(v, [1, 1, 1], 90, [0, 0, 1], [0, 0, 0], weights=w)
        pivot = vx.vertex_mean(v, w)
        assert np.allclose(vx.vertex_mean(moved, w), pivot)                       # the weighted mean is the fixed point
    # samples of the reference's meshes (tests/golden/make_reference_samples.py): every face using one of the first
    # 32 vertices is kept, so their weights are those of the full mesh
    for name in ("armadillo_small", "Dragon_50k"):
        v, f, w = vx.load_obj(os.path.join(GOLD, "reference_models", name + "_sample.obj"), with_multiplicity=True)
        assert len(v) > 32 and (w[:32] == 1).all() and (w >= 1).all(), name
