"""Oracle of the mesh smoothing (engine.vertex_neighbors / engine.smooth_mesh, csrc/t3d_smooth.cu), numpy only; imported by the
tests, never by the package.

trimesh.smoothing.filter_taubin with the equal-weight laplacian_calculation, written out so that every float64 operation is
fixed: each face (a, b, c) gives the edges {a,b}, {b,c}, {c,a}; edges whose ends are equal are dropped; the neighbours of i are
the sorted distinct j joined to i (CSR: offsets int64 (V+1), neighbours int32).  From x = vertices.astype(float64) and
w = 1.0 / degree, each iteration sums s = +0.0, s = s + w * x[j] over the neighbours in ascending order, dd = s - x[i], and sets
x[i] + lamb * dd (even iterations) or x[i] - nu * dd (odd), every vertex from the previous iterate; a vertex with no neighbour
keeps its position.  The result is x.astype(float32).
"""
import numpy as np

SHORT = 64        # rows up to this degree are summed slot by slot over all such rows at once, longer ones one by one


def adjacency(faces, V):
    """(offsets int64 (V + 1,), neighbours int32 (N,))."""
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    e = e[e[:, 0] != e[:, 1]]
    e = np.concatenate([e, e[:, ::-1]])
    key = np.unique(e[:, 0] * V + e[:, 1])
    a, b = key // max(V, 1), key % max(V, 1)
    off = np.zeros(V + 1, np.int64)
    off[1:] = np.cumsum(np.bincount(a, minlength=V))
    return off, b.astype(np.int32)


def neighbour_sums(x, off, nb):
    """float64 (V, 3): s = +0.0, then s = s + w * x[j] over each row in ascending order (w = 1.0 / degree)."""
    deg = np.diff(off)
    w = np.zeros(len(deg))
    w[deg > 0] = 1.0 / deg[deg > 0]
    s = np.zeros_like(x)
    short = deg <= SHORT
    for k in range(int(deg[short].max()) if short.any() else 0):
        m = np.flatnonzero(short & (deg > k))
        s[m] = s[m] + w[m, None] * x[nb[off[m] + k]]
    for i in np.flatnonzero(~short):
        p = w[i] * x[nb[off[i]:off[i + 1]]]
        s[i] = np.add.accumulate(np.concatenate([s[i:i + 1], p]), axis=0)[-1]     # accumulate adds left to right
    return s


def taubin(vertices, off, nb, iterations=10, lamb=0.5, nu=0.5):
    """float32 (V, 3): the smoothed vertices."""
    x = np.asarray(vertices, dtype=np.float32).reshape(-1, 3).astype(np.float64)
    moving = (np.diff(off) > 0)[:, None]
    for it in range(iterations):
        dd = neighbour_sums(x, off, nb) - x
        y = x + lamb * dd if it % 2 == 0 else x - nu * dd
        x = np.where(moving, y, x)
    return x.astype(np.float32)


def smooth(vertices, faces, iterations=10, lamb=0.5, nu=0.5):
    """(smoothed float32 vertices, offsets, neighbours)."""
    off, nb = adjacency(faces, len(vertices))
    return taubin(vertices, off, nb, iterations, lamb, nu), off, nb
