"""The mesh-bodies oracle (tests/bodies_oracle.py) against brute force on small meshes: breadth-first labelling, exact
fractions.Fraction sums rounded once, and the corner cases (unreferenced vertices, no faces, no vertices, one face, repeated and
degenerate faces).  Also the body filter through engine.component_keep.  No GPU."""
from collections import deque
from fractions import Fraction

import numpy as np
import pytest

import bodies_oracle as bo


def bfs_labels(faces, V):
    adj = [[] for _ in range(V)]
    for a, b, c in np.asarray(faces, dtype=np.int64).reshape(-1, 3):
        for u, w in ((a, b), (a, c)):
            adj[u].append(w)
            adj[w].append(u)
    lab = np.full(V, -1, np.int64)
    n = 0
    for s in range(V):                       # bodies numbered by their smallest vertex
        if lab[s] >= 0:
            continue
        lab[s] = n
        q = deque([s])
        while q:
            u = q.popleft()
            for w in adj[u]:
                if lab[w] < 0:
                    lab[w] = n
                    q.append(w)
        n += 1
    return lab, n


def exact_sum(terms):
    """sum of round_half_even(t * 2^64) as a Fraction-exact integer, then rounded once to float64 times 2^-64."""
    s = sum(round(Fraction(float(t)) * 2 ** 64) for t in terms)      # round() of a Fraction is half-to-even
    return float(Fraction(s, 2 ** 64))


def random_mesh(rng, V, F, n_clusters):
    """Faces drawn inside vertex clusters (so there are several bodies), some vertices left unreferenced, some faces repeated
    or degenerate; coordinates with a spread of magnitudes and both signs, zeros of both signs included."""
    cluster = rng.integers(0, n_clusters, V)
    faces = []
    for _ in range(F):
        c = rng.integers(0, n_clusters)
        members = np.flatnonzero(cluster == c)
        if len(members) == 0:
            continue
        faces.append(rng.choice(members, 3))
    f = np.array(faces, dtype=np.int64).reshape(-1, 3)
    if len(f) > 2:
        f = np.concatenate([f, f[:2]])                        # repeated faces
    v = (rng.standard_normal((V, 3)) * 10.0 ** rng.integers(-3, 4, (V, 1))).astype(np.float32)
    v[rng.random((V, 3)) < 0.05] = 0.0
    v[rng.random((V, 3)) < 0.05] = -0.0
    return v, f


def check_against_brute_force(v, f):
    V = len(v)
    lab, n = bo.labels(f, V)
    bl, bn = bfs_labels(f, V)
    assert n == bn and np.array_equal(lab, bl)
    st = bo.stats(v, f, lab, n)
    fb = lab[f[:, 0]] if len(f) else np.zeros(0, np.int64)
    tv, ta = bo.terms(v, f)
    for b in range(n):
        verts_b = np.flatnonzero(lab == b)
        assert st["vertex_counts"][b] == len(verts_b)
        assert st["face_counts"][b] == int((fb == b).sum())
        assert st["first_vertex"][b] == verts_b.min()
        for c in range(3):
            col = [float(x) for x in v[verts_b, c]]
            assert st["bbox_mm"][b, 2 * c] == min(col) and st["bbox_mm"][b, 2 * c + 1] == max(col)
        assert not np.signbit(st["bbox_mm"][b][st["bbox_mm"][b] == 0]).any()        # zero bounds are +0.0
        assert st["signed_volumes"][b] == exact_sum(tv[fb == b])
        assert st["areas"][b] == exact_sum(ta[fb == b])
    assert np.array_equal(st["face_body"], fb)
    return lab, n, st


@pytest.mark.parametrize("seed", range(12))
def test_oracle_equals_brute_force_on_random_meshes(seed):
    rng = np.random.default_rng(seed)
    V = int(rng.integers(1, 60))
    v, f = random_mesh(rng, V, int(rng.integers(0, 80)), int(rng.integers(1, 8)))
    check_against_brute_force(v, f)


def test_oracle_corner_cases():
    rng = np.random.default_rng(99)
    v = rng.standard_normal((7, 3)).astype(np.float32)
    # no faces: every vertex is a body of its own, with no faces and zero sums
    lab, n, st = check_against_brute_force(v, np.zeros((0, 3), np.int64))
    assert n == 7 and lab.tolist() == list(range(7)) and st["face_counts"].tolist() == [0] * 7
    assert (st["signed_volumes"] == 0).all() and (st["areas"] == 0).all()
    # no vertices
    lab, n = bo.labels(np.zeros((0, 3), np.int64), 0)
    assert n == 0 and len(lab) == 0
    # one face, two unreferenced vertices around it
    lab, n, st = check_against_brute_force(v, np.array([[2, 4, 5]]))
    assert n == 5 and lab.tolist() == [0, 1, 2, 3, 2, 2, 4]
    # degenerate faces (repeated corners) link what they name and add zero area
    lab, n, st = check_against_brute_force(v, np.array([[1, 1, 1], [3, 3, 6], [3, 6, 6]]))
    assert n == 6 and lab[3] == lab[6] and st["areas"][lab[3]] == 0.0
    # repeated faces count once each
    lab, n, st = check_against_brute_force(v, np.array([[0, 1, 2], [0, 1, 2], [2, 1, 0]]))
    assert st["face_counts"][0] == 3 and st["areas"][0] == exact_sum(np.repeat(bo.terms(v, [[0, 1, 2]])[1], 3))


def test_fixed_point_rounds_ties_to_even_and_sums_exactly():
    # ties at the 2^-64 grid: 2.5 and 3.5 ulps of it round to 2 and 4; the float64 sum of these terms would lose them
    t = np.array([2.5 * 2.0 ** -64, 3.5 * 2.0 ** -64, 1e6, -1e6], np.float64)
    assert bo.fixed_sums(t, np.zeros(4, np.int64), 1) == [6]
    big = np.array([2.0 ** 61, 2.0 ** 61, -(2.0 ** 61), 2.0 ** -60], np.float64)
    assert bo.fixed_sums(big, np.zeros(4, np.int64), 1) == [(1 << 125) + 16]
    with pytest.raises(OverflowError):
        bo.fixed_sums(np.array([2.0 ** 62]), np.zeros(1, np.int64), 1)


def test_select_is_the_numpy_compaction():
    rng = np.random.default_rng(5)
    v, f = random_mesh(rng, 40, 50, 5)
    lab, n = bo.labels(f, len(v))
    nrm = rng.standard_normal((len(v), 3)).astype(np.float32)
    keep = [b for b in range(n) if b % 2 == 0]
    for dt in (np.int32, np.int64):
        sv, sf, sn = bo.select(v, f.astype(dt), lab, keep, nrm)
        assert sf.dtype == dt
        kv = np.flatnonzero(np.isin(lab, keep))
        assert np.array_equal(sv, v[kv]) and np.array_equal(sn, nrm[kv])
        kf = f[np.isin(lab[f[:, 0]], keep)]
        assert np.array_equal(kv[sf], kf)                     # the renumbered faces name the same vertices, in order


def test_body_filter_is_component_keep_with_zero_based_ids():
    from tomography_3d_reconstructor_b200.engine import component_keep
    face_counts = np.array([0, 12, 3, 12, 1, 0, 7], np.int64)          # bodies 0..6
    assert (component_keep(face_counts, 1) - 1).tolist() == [1, 2, 3, 4, 6]          # the default drops face-less bodies
    assert (component_keep(face_counts, 4) - 1).tolist() == [1, 3, 6]
    assert (component_keep(face_counts, 1, 1) - 1).tolist() == [1]                   # tie 12 / 12: the lower body id
    assert (component_keep(face_counts, 1, 3) - 1).tolist() == [1, 3, 6]
    assert (component_keep(np.zeros(0, np.int64), 1, 1) - 1).tolist() == []
