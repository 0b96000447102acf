"""Mesh hierarchy generation without psbody (cape_b200/mesh_sampling.py, SURVEY.md 8(f) row 4).

Pinned by the reference itself: `data/transform_matrices/for_demo/{A,D,U}.npy` are the output of the reference's
`generate_transform_matrices(template, [1, 2, 1, 2, 1, 2, 1, 1])` (psbody + qslim), and this restatement must
reproduce them -- adjacency and down-sampling matrices exactly, up-sampling matrices to fp32 rounding.  The
fixtures and the template are read from tests/golden/smpl_topology.*.npz (cape_b200.pack_topology), like every other
test.  The synthetic-mesh tests need none of the reference's data."""
import heapq

import numpy as np
import pytest
import scipy.sparse as sp

from cape_b200 import mesh_sampling as MS


def icosphere(levels=2):
    t = (1.0 + 5 ** 0.5) / 2.0
    v = [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t),
         (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
         (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7),
         (9, 8, 1)]
    v = [np.asarray(x, np.float64) / np.linalg.norm(x) for x in v]
    for _ in range(levels):
        mid, nf = {}, []

        def m(a, b):
            k = (min(a, b), max(a, b))
            if k not in mid:
                p = v[a] + v[b]
                v.append(p / np.linalg.norm(p))
                mid[k] = len(v) - 1
            return mid[k]

        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    rng = np.random.RandomState(0)                      # break the symmetry: no exactly tied collapse costs
    v = np.asarray(v) * (1.0 + 0.05 * rng.rand(len(v), 1)) * np.asarray([1.0, 0.8, 1.3])
    return MS.TriMesh(v=v, f=np.asarray(f))


def test_reproduces_the_reference_fixtures(hierarchy):
    """The 8-layer / ds_factor 2 hierarchy from the SMPL template == the matrices the reference ships."""
    from cape_b200 import topology as T
    v, f = T.template_mesh()
    ref_A = T._mats("for_demo", "A", np.float64)
    ref_D = T._mats("for_demo", "D", np.float64)
    ref_U = T._mats("for_demo", "U", np.float64)
    M, A, D, U, E = MS.generate_transform_matrices(MS.TriMesh(v=v, f=f), [1, 2, 1, 2, 1, 2, 1, 1])
    assert [a.shape[0] for a in A] == [6890, 6890, 3445, 3445, 1723, 1723, 862, 862, 862]
    for a, b in zip(ref_A, A):
        assert abs(sp.csr_matrix(a) - sp.csr_matrix(b)).max() == 0
    for a, b in zip(ref_D, D):
        assert abs(sp.csr_matrix(a) - sp.csr_matrix(b)).max() == 0
    for a, b in zip(ref_U, U):
        assert abs(sp.csr_matrix(a) - sp.csr_matrix(b)).max() < 1e-6          # the shipped files are fp32
    assert sorted(map(tuple, E[0].tolist())) == sorted(map(tuple, T.smpl_edges().tolist()))
    # and through the front door (main.py:31-43): the Laplacians the model is built from
    L, D2, U2, p = MS.hierarchy(MS.TriMesh(v=v, f=f), 8, 2)
    for a, b in zip(hierarchy["L"], L):
        assert abs(sp.csr_matrix(a) - sp.csr_matrix(b)).max() == 0
    assert p == hierarchy["p"]


@pytest.mark.parametrize("layers,want", [(4, [642, 642, 321, 321, 321]), (6, [642, 642, 321, 321, 161, 161, 161])])
def test_other_depths(layers, want):
    """--num_conv_layers 4 / 6 (main.py:31-34), which the reference cannot run without psbody."""
    mesh = icosphere(3)                                  # 642 vertices
    L, D, U, p = MS.hierarchy(mesh, layers, 2)
    assert p == want and [l.shape[0] for l in L] == want
    for i in range(layers):
        assert D[i].shape == (p[i + 1], p[i]) and U[i].shape == (p[i], p[i + 1])
        assert D[i].dtype == np.float32 and U[i].dtype == np.float32


def test_decimation_properties():
    mesh = icosphere(3)
    faces, D = MS.qslim_decimator_transformer(mesh, factor=0.5)
    D = sp.csr_matrix(D)
    assert D.shape == (321, 642) and D.nnz == 321 and (D.data == 1).all()
    kept = D.indices
    assert (np.diff(kept) > 0).all()                     # kept vertices in increasing order of their old index
    assert faces.min() == 0 and faces.max() == 320 and len(np.unique(faces)) == 321
    assert not ((faces[:, 0] == faces[:, 1]) | (faces[:, 1] == faces[:, 2]) | (faces[:, 0] == faces[:, 2])).any()
    coarse = MS.TriMesh(v=D.dot(mesh.v), f=faces)
    A = MS.get_vert_connectivity(coarse)
    assert abs(A - A.T).max() == 0 and set(np.unique(A.data)) <= {1.0, 2.0}
    # a closed surface stays closed: V - E + F = 2
    assert coarse.v.shape[0] - len(MS.get_vertices_per_edge(coarse)) + len(faces) == 2
    # up-sampling: kept vertices map to themselves exactly, every fine vertex lands close to its own position
    U = sp.csr_matrix(MS.setup_deformation_transfer(coarse, mesh))
    assert U.shape == (642, 321)
    back = U.dot(coarse.v)
    assert np.abs(back[kept] - mesh.v[kept]).max() < 1e-12
    edge = np.linalg.norm(mesh.v[mesh.f[:, 0]] - mesh.v[mesh.f[:, 1]], axis=1).mean()
    assert np.linalg.norm(back - mesh.v, axis=1).max() < 1.5 * edge
    # factor 1: nothing collapses
    f1, D1 = MS.qslim_decimator_transformer(mesh, factor=1.0)
    assert abs(sp.csr_matrix(D1) - sp.identity(642)).max() == 0 and (f1 == mesh.f).all()


def test_edge_heap_behaves_like_heapq():
    """_EdgeHeap must pop in exactly the order Python's heapq would, including after in-place renames that break the
    heap invariant (the reference's qslim loop depends on that order, lib/mesh_sampling.py:196-206)."""
    rng = np.random.RandomState(3)
    ref, mine = [], MS._EdgeHeap(4)
    for step in range(4000):
        op = rng.rand()
        if op < 0.55 or len(ref) < 5:
            cost, r, c = float(rng.randint(0, 40)) / 7.0, int(rng.randint(0, 30)), int(rng.randint(0, 30))
            heapq.heappush(ref, (cost, (r, c)))
            mine.push(cost, r, c)
        elif op < 0.85:
            a = heapq.heappop(ref)
            b = mine.pop()
            assert (a[0], a[1][0], a[1][1]) == (float(b[0]), int(b[1]), int(b[2]))
        else:
            old, new = int(rng.randint(0, 30)), int(rng.randint(0, 30))
            for k in range(len(ref)):
                if ref[k][1][0] == old:
                    ref[k] = (ref[k][0], (new, ref[k][1][1]))
            for k in range(len(ref)):
                if ref[k][1][1] == old:
                    ref[k] = (ref[k][0], (ref[k][1][0], new))
            mine.rename(old, new)
        assert mine.n == len(ref)
    assert [(x[0], x[1][0], x[1][1]) for x in ref] == [(float(mine.cost[i]), int(mine.r[i]), int(mine.c[i]))
                                                     for i in range(mine.n)]


def test_closest_point_regions():
    a = np.array([[0.0, 0.0, 0.0]])
    b = np.array([[1.0, 0.0, 0.0]])
    c = np.array([[0.0, 1.0, 0.0]])
    cases = [((0.25, 0.25, 0.7), 0, (0.25, 0.25, 0.0)),      # above the interior
             ((0.5, -0.3, 0.2), 1, (0.5, 0.0, 0.0)),         # edge a-b
             ((0.8, 0.8, -0.1), 2, (0.5, 0.5, 0.0)),         # edge b-c
             ((-0.4, 0.5, 0.0), 3, (0.0, 0.5, 0.0)),         # edge c-a
             ((-0.2, -0.1, 0.3), 4, (0.0, 0.0, 0.0)),        # vertex a
             ((1.5, -0.2, 0.0), 5, (1.0, 0.0, 0.0)),         # vertex b
             ((-0.1, 1.7, 0.1), 6, (0.0, 1.0, 0.0))]         # vertex c
    for p, part, q in cases:
        got_q, got_part = MS.closest_points_on_triangles(np.asarray(p), a, b, c)
        assert got_part[0] == part and np.allclose(got_q[0], q)
    # against a dense sampling of the triangle
    rng = np.random.RandomState(0)
    tri = rng.randn(3, 3)
    u, v = np.meshgrid(np.linspace(0, 1, 201), np.linspace(0, 1, 201))
    keep = u + v <= 1
    pts = tri[0] + u[keep][:, None] * (tri[1] - tri[0]) + v[keep][:, None] * (tri[2] - tri[0])
    for _ in range(50):
        p = rng.randn(3) * 1.5
        q, _ = MS.closest_points_on_triangles(p, tri[0:1], tri[1:2], tri[2:3])
        best = np.linalg.norm(pts - p, axis=1).min()
        assert np.linalg.norm(q[0] - p) <= best + 1e-12 and np.linalg.norm(q[0] - p) >= best - 0.02


def test_nearest_on_mesh_is_exact():
    mesh = icosphere(2)
    rng = np.random.RandomState(1)
    pts = rng.randn(40, 3) * 1.2
    faces, parts, closest = MS.nearest_on_mesh(mesh, pts)
    a, b, c = (mesh.v[mesh.f[:, k]] for k in range(3))
    for i, p in enumerate(pts):
        q, _ = MS.closest_points_on_triangles(p, a, b, c)             # brute force over every face
        d = np.linalg.norm(q - p, axis=1)
        assert abs(np.linalg.norm(closest[i] - p) - d.min()) < 1e-12


def test_obj_loader(tmp_path):
    fn = tmp_path / "m.obj"
    fn.write_text("# c\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvn 0 0 1\nf 1/1/1 2/2/1 3/3/1 4/4/1\nf 1 3 4\n")
    m = MS.TriMesh(filename=str(fn))
    assert m.v.shape == (4, 3) and m.f.tolist() == [[0, 1, 2], [0, 2, 3], [0, 2, 3]]
