"""CPU: the marching-cubes case table (product side, dist-renderer_b200/mc_tables.py) against the oracle's independent
per-cube tracing, the oracle against properties of analytic shapes, and the chamfer oracle against the outputs of the
reference's own eval_func.py (tests/golden/chamfer.npz)."""
import importlib
import os

import numpy as np
import pytest

import cases  # noqa: F401  (puts the repo root on sys.path)
import mesh_cases
from oracle import mesh_oracle as O

mc_tables = importlib.import_module("dist-renderer_b200.mc_tables")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "chamfer.npz")


def test_case_table_matches_oracle_tracing():
    """Two derivations of the 256 rows (face-normal rule vs summed-normal rule for the orientation) agree."""
    for c in range(256):
        assert [tuple(t) for t in mc_tables.case_triangles(c)] == [tuple(t) for t in O.case_triangles(c)], c
    n = mc_tables.n_tris()
    assert n[0] == 0 and n[255] == 0 and max(n) == mc_tables.MAX_TRIS == 5 and sum(n) == 820


def test_case_table_rows_are_surface_patches():
    """Every row: interior edges are shared by two triangles with opposite direction; boundary edges join two cube edges
    of one face; every crossing edge is used; no other edge is."""
    for c in range(256):
        tris = mc_tables.case_triangles(c)
        crossing = {e for e in range(12)
                    if ((c >> mc_tables.edge_corners(e)[0]) ^ (c >> mc_tables.edge_corners(e)[1])) & 1}
        assert {e for t in tris for e in t} == crossing
        directed = [(t[k], t[(k + 1) % 3]) for t in tris for k in range(3)]
        assert len(set(directed)) == len(directed)
        for a, b in directed:
            if (b, a) in directed:
                continue
            shared = [(f, s) for f in range(3) for s in range(2)
                      if a in mc_tables.face_edges(f, s) and b in mc_tables.face_edges(f, s)]
            assert shared, (c, a, b)


def test_committed_header_is_current():
    path = os.path.join(ROOT, "dist-renderer_b200", "csrc", "mc_tables.inc")
    assert open(path).read() == mc_tables.as_header()


@pytest.mark.parametrize("name,euler,volume", [("sphere33", 2, 4 / 3 * np.pi * 0.6 ** 3),
                                                ("torus40", 0, 2 * np.pi ** 2 * 0.55 * 0.22 ** 2)])
def test_oracle_analytic_shapes(name, euler, volume):
    cs = mesh_cases.VOLUMES[name]
    v, f = O.marching_cubes(cs["vol"](), cs["level"], cs["spacing"], cs["origin"])
    r = O.mesh_report(v, f)
    assert r["closed"] and r["oriented"] and r["euler"] == euler and r["used_verts"] == len(v)
    assert abs(r["volume"] - volume) / volume < 0.02       # positive: normals point out of the sdf < 0 region


def test_oracle_noise_volume_is_closed_manifold():
    """White noise exercises every case, ambiguous faces included: the face rule must leave no cracks."""
    cs = mesh_cases.VOLUMES["noise_closed"]
    v, f = O.marching_cubes(cs["vol"](), cs["level"], cs["spacing"], cs["origin"])
    r = O.mesh_report(v, f)
    assert len(f) > 1000 and r["closed"] and r["oriented"] and r["used_verts"] == len(v)


def test_oracle_vertices_sit_on_sign_changes():
    cs = mesh_cases.VOLUMES["noise"]
    vol = cs["vol"]()
    v, f = O.marching_cubes(vol, cs["level"])
    frac = v - np.floor(v)
    on_edge = (frac > 0).sum(1)
    assert np.all(on_edge <= 1)
    # trilinear interpolation of the volume at a vertex returns the level
    i0 = np.floor(v).astype(int)
    i1 = np.minimum(i0 + 1, np.array(vol.shape) - 1)
    t = (v - i0).max(1)
    ax = np.argmax(v - i0, 1)
    a = vol[i0[:, 0], i0[:, 1], i0[:, 2]]
    j = i0.copy()
    j[np.arange(len(v)), ax] = i1[np.arange(len(v)), ax]
    b = vol[j[:, 0], j[:, 1], j[:, 2]]
    assert np.allclose(a + t * (b - a), cs["level"], atol=1e-5)


def test_sampling_oracle_is_area_weighted_and_on_surface():
    cs = mesh_cases.VOLUMES["sphere33"]
    v, f = O.marching_cubes(cs["vol"](), cs["level"], cs["spacing"], cs["origin"])
    u = np.random.default_rng(0).random((200000, 3), dtype=np.float32)
    pts, fi = O.sample_surface(v, f, u)
    assert abs(np.linalg.norm(pts, axis=1) - 0.6).max() < 4e-3            # on the sphere's mesh
    area = O.face_areas(v, f).astype(np.float64)
    expect = area / area.sum() * len(u)
    got = np.bincount(fi, minlength=len(f))
    z = (got - expect) / np.sqrt(expect)
    assert abs(z).max() < 6 and abs(z.std() - 1) < 0.1
    # uniform over the surface: the mean of the samples of a centred sphere is the origin
    assert np.abs(pts.mean(0)).max() < 5e-3


def _chamfer_inputs():
    rng = np.random.default_rng(7)
    a = rng.standard_normal((3000, 3)) * 0.3
    b = rng.standard_normal((2500, 3)) * 0.3 + 0.05
    return a, b


def test_chamfer_oracle_matches_reference():
    """Bit for bit: the oracle's float results equal the reference's."""
    g = np.load(GOLD)
    a, b = _chamfer_inputs()
    assert O.compute_chamfer_distance(a, b) == float(g["sq"])
    assert O.compute_chamfer_distance(a, b, False) == float(g["lin"])
    assert O.compute_chamfer_distance_separate(a, b) == tuple(float(x) for x in g["sep"])


def test_chamfer_oracle_matches_golden():
    """tests/golden/chamfer.npz = outputs of the reference's eval_func.py (oracle/make_golden.py --chamfer)."""
    g = np.load(GOLD)
    a, b = _chamfer_inputs()
    assert np.array_equal(g["a"], a) and np.array_equal(g["b"], b)
    assert np.isclose(O.compute_chamfer_distance(a, b), float(g["sq"]), rtol=1e-12)
    assert np.isclose(O.compute_chamfer_distance(a, b, False), float(g["lin"]), rtol=1e-12)
    assert np.allclose(O.compute_chamfer_distance_separate(a, b), g["sep"], rtol=1e-12)


def test_write_ply_round_trip(tmp_path):
    """evaluation.write_ply: binary little-endian, float x/y/z + uchar-counted int32 faces (create_mesh.py:180-198)."""
    import torch
    ev = importlib.import_module("dist-renderer_b200.evaluation")
    cs = mesh_cases.VOLUMES["sphere_ragged"]
    v, f = O.marching_cubes(cs["vol"](), cs["level"], cs["spacing"], cs["origin"])
    path = str(tmp_path / "m.ply")
    ev.write_ply(torch.from_numpy(v), torch.from_numpy(f), path)
    raw = open(path, "rb").read()
    head, body = raw.split(b"end_header\n", 1)
    lines = head.decode("ascii").split("\n")
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0"
    assert "element vertex %d" % len(v) in lines and "element face %d" % len(f) in lines
    assert "property list uchar int vertex_indices" in lines
    vv = np.frombuffer(body[:len(v) * 12], dtype="<f4").reshape(-1, 3)
    rec = np.frombuffer(body[len(v) * 12:], dtype=[("n", "u1"), ("idx", "<i4", (3,))])
    assert np.array_equal(vv, v) and np.all(rec["n"] == 3) and np.array_equal(rec["idx"], f)


def test_evaluation_rejects_cpu_tensors():
    """No CPU path: the mesh entry points refuse host tensors instead of computing on the host."""
    import torch
    ev = importlib.import_module("dist-renderer_b200.evaluation")
    with pytest.raises(ValueError, match="CUDA"):
        ev.marching_cubes(torch.zeros(4, 4, 4), 0.0)
    with pytest.raises(ValueError, match="CUDA"):
        ev.nearest_sqdist(torch.zeros(4, 3), torch.zeros(2, 3))
    with pytest.raises(ValueError, match="CUDA"):
        ev.sample_surface(torch.zeros(3, 3), torch.zeros(1, 3, dtype=torch.int32), 5)
