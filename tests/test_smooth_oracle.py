"""The mesh-smoothing oracle (tests/smooth_oracle.py) against independent formulations, no GPU: the adjacency against Python
sets on random meshes with degenerate, repeated and out-of-cluster faces and unreferenced vertices; the Taubin iterates
against trimesh's formulation (a scipy.sparse.csr_matrix of 1 / degree weights), bit for bit; the identity at iterations=0,
vertices without neighbours, rows longer than the slot-by-slot path and the sign of a zero sum."""
import numpy as np
import pytest
import scipy.sparse as sp

import smooth_oracle as so


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def set_adjacency(faces, V):
    nbrs = [set() for _ in range(V)]
    for face in np.asarray(faces, dtype=np.int64).reshape(-1, 3):
        for a, b in ((face[0], face[1]), (face[1], face[2]), (face[2], face[0])):
            if a != b:
                nbrs[a].add(int(b))
                nbrs[b].add(int(a))
    off = np.concatenate([[0], np.cumsum([len(n) for n in nbrs])]).astype(np.int64)
    nb = np.array([j for n in nbrs for j in sorted(n)], dtype=np.int32)
    return off, nb


def random_mesh(rng, V, F, clusters):
    """Faces inside vertex clusters, some vertices unreferenced, degenerate faces (two or three equal corners) and repeated
    faces; coordinates of mixed magnitude and sign with zeros of both signs."""
    cl = rng.integers(0, clusters, V)
    faces = [rng.choice(np.flatnonzero(cl == c), 3) for c in rng.integers(0, clusters, F) if (cl == c).any()]
    f = np.array(faces, dtype=np.int64).reshape(-1, 3)
    f = f[~(f == V - 1).any(axis=1)]                              # the last vertex stays unreferenced
    if len(f) > 4:
        f = np.concatenate([f, f[:3], f[:2, [1, 2, 0]], f[:2, [0, 0, 1]], f[:1, [2, 2, 2]]])
    v = (rng.standard_normal((V, 3)) * 10.0 ** rng.integers(-2, 3, (V, 1))).astype(np.float32)
    v[rng.random((V, 3)) < 0.05] = 0.0
    v[rng.random((V, 3)) < 0.05] = -0.0
    return v, f


def scipy_taubin(vertices, off, nb, iterations, lamb, nu):
    """trimesh.smoothing.filter_taubin: laplacian_calculation(equal_weight=True) is a csr_matrix of 1 / degree; here rows with
    no neighbour are held fixed as the definition asks (trimesh would move them towards the origin)."""
    V = len(vertices)
    deg = np.diff(off)
    L = sp.csr_matrix((np.repeat(1.0 / np.maximum(deg, 1), deg), nb, off), shape=(V, V))
    x = np.asarray(vertices, np.float64).copy()
    moving = deg > 0
    for it in range(iterations):
        dot = L.dot(x) - x
        if it % 2 == 0:
            x[moving] += lamb * dot[moving]
        else:
            x[moving] -= nu * dot[moving]
    return x.astype(np.float32)


MESHES = [(0, 40, 60, 3), (1, 500, 900, 7), (2, 3000, 2000, 200), (3, 6, 40, 1)]


@pytest.mark.parametrize("seed,V,F,k", MESHES)
def test_adjacency_equals_python_sets(seed, V, F, k):
    v, f = random_mesh(np.random.default_rng(seed), V, F, k)
    off, nb = so.adjacency(f, V)
    want_off, want_nb = set_adjacency(f, V)
    assert bits_equal(off, want_off) and bits_equal(nb, want_nb)
    assert off[-1] == len(nb) and np.diff(off)[V - 1] == 0


@pytest.mark.parametrize("seed,V,F,k", MESHES)
@pytest.mark.parametrize("iterations,lamb,nu", [(1, 0.5, 0.5), (2, 0.5, 0.5), (10, 0.5, 0.5), (7, 0.33, 0.34), (4, 0.6, -0.1)])
def test_taubin_equals_the_scipy_formulation(seed, V, F, k, iterations, lamb, nu):
    v, f = random_mesh(np.random.default_rng(seed), V, F, k)
    off, nb = so.adjacency(f, V)
    got = so.taubin(v, off, nb, iterations, lamb, nu)
    assert bits_equal(got, scipy_taubin(v, off, nb, iterations, lamb, nu))
    assert bits_equal(got[np.diff(off) == 0], v[np.diff(off) == 0])    # vertices without neighbours stay put


def test_identity_empty_and_lone_vertices():
    v, f = random_mesh(np.random.default_rng(5), 300, 400, 4)
    assert bits_equal(so.smooth(v, f, 0)[0], v)
    out, off, nb = so.smooth(np.ones((5, 3), np.float32), np.zeros((0, 3), np.int64))
    assert bits_equal(out, np.ones((5, 3), np.float32)) and off.tolist() == [0] * 6 and len(nb) == 0
    out, off, nb = so.smooth(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int64))
    assert out.shape == (0, 3) and off.tolist() == [0] and len(nb) == 0


def test_long_rows_follow_the_same_order():
    """A fan: the hub's row is longer than the slot-by-slot path and is summed left to right on its own."""
    n = 500
    rng = np.random.default_rng(7)
    f = np.stack([np.zeros(n, np.int64), np.arange(1, n + 1), np.arange(2, n + 2)], axis=1)
    v = rng.standard_normal((n + 2, 3)).astype(np.float32)
    off, nb = so.adjacency(f, n + 2)
    assert np.diff(off)[0] == n + 1 > so.SHORT
    assert bits_equal(so.taubin(v, off, nb, 3), scipy_taubin(v, off, nb, 3, 0.5, 0.5))


def test_sums_start_at_positive_zero():
    """A vertex whose neighbours' products are all -0.0 sums to +0.0, as scipy's csr_matvec (its sum starts at +0.0);
    a sum started at the first product would be -0.0."""
    f = np.array([[0, 1, 2]])
    x = np.array([[1.0, 5.0, -0.0], [-0.0, 2.0, -0.0], [-0.0, 3.0, -0.0]])
    off, nb = so.adjacency(f, 3)
    s = so.neighbour_sums(x, off, nb)
    L = sp.csr_matrix((np.full(6, 0.5), nb, off), shape=(3, 3))
    assert bits_equal(s, L.dot(x))
    assert np.signbit(x[1:, 0]).all() and not np.signbit(s[0, 0]) and not np.signbit(s[0, 2])
