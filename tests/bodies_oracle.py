"""Oracle of the mesh bodies (engine.mesh_bodies, csrc/t3d_label.cu), numpy / scipy and Python integers only; imported by the
tests, never by the package.

A body is a connected component of the graph with the edges f0-f1 and f0-f2 of every face, numbered as
scipy.sparse.csgraph.connected_components numbers them.  Per body: vertex / face counts, first vertex, the box of its vertex
columns (a zero bound is +0.0), and the signed volume and area: each face's float64 term (k_mesh_measure's expression, left to
right, no FMA), rounded half-to-even to a multiple of 2^-64, summed exactly as a Python int, the sum rounded once (float(int)).
"""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

TWO64 = 2.0 ** 64


def labels(faces, V):
    """(int32 (V,) body of each vertex, number of bodies)."""
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    if V == 0:
        return np.zeros(0, np.int32), 0
    r = np.concatenate([f[:, 0], f[:, 0]])
    c = np.concatenate([f[:, 1], f[:, 2]])
    g = coo_matrix((np.ones(len(r), np.int8), (r, c)), shape=(V, V)).tocsr()
    n, lab = connected_components(g, directed=False)
    return lab.astype(np.int32), int(n)


def terms(verts, faces):
    """float64 (F,) signed-volume and area terms of every face, evaluated as the device evaluates them."""
    v = np.asarray(verts, dtype=np.float32).astype(np.float64)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    a, b, c = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    ax, ay, az = a[:, 0], a[:, 1], a[:, 2]
    bx, by, bz = b[:, 0], b[:, 1], b[:, 2]
    cx, cy, cz = c[:, 0], c[:, 1], c[:, 2]
    nx, ny, nz = by * cz - bz * cy, bz * cx - bx * cz, bx * cy - by * cx
    vol = (ax * nx + ay * ny + az * nz) / 6.0
    ux, uy, uz, wx, wy, wz = bx - ax, by - ay, bz - az, cx - ax, cy - ay, cz - az
    px, py, pz = uy * wz - uz * wy, uz * wx - ux * wz, ux * wy - uy * wx
    area = 0.5 * np.sqrt(px * px + py * py + pz * pz)
    return vol, area


def fixed_sums(t, body, B):
    """Python ints (B,): per body, the sum of round_half_even(t * 2^64).  |t * 2^64| is exact for |t| < 2^62 and np.rint rounds
    half to even; its magnitude splits exactly into four 32-bit parts, which are summed with their sign per body by reduceat
    (each sum stays below 2^63 for fewer than 2^31 faces)."""
    t = np.asarray(t, dtype=np.float64)
    if len(t) and not (np.abs(t).max() < 2.0 ** 62):
        raise OverflowError("a term of magnitude >= 2^62")
    r = np.rint(t * TWO64)
    a = np.abs(r)
    h = np.floor(a / TWO64)                    # exact: division by a power of two, then an integer part
    lo = (a - h * TWO64).astype(np.uint64)     # exact: the low bits of a, in [0, 2^64)
    h = h.astype(np.int64)
    sgn = np.where(r < 0, -1, 1).astype(np.int64)
    parts = [sgn * (lo & np.uint64(0xffffffff)).astype(np.int64), sgn * (lo >> np.uint64(32)).astype(np.int64),
             sgn * (h & 0xffffffff), sgn * (h >> 32)]
    out = [0] * B
    if len(t) == 0:
        return out
    order = np.argsort(body, kind="stable")
    sb = np.asarray(body)[order]
    starts = np.flatnonzero(np.concatenate([[True], sb[1:] != sb[:-1]]))
    sums = [np.add.reduceat(p[order], starts) for p in parts]
    for k, b in enumerate(sb[starts]):
        out[int(b)] = int(sums[0][k]) + (int(sums[1][k]) << 32) + (int(sums[2][k]) << 64) + (int(sums[3][k]) << 96)
    return out


def fixed_to_f64(s):
    """The Python int s times 2^-64, rounded once to float64 (float(int) rounds correctly; the scaling is exact)."""
    return float(s) * 2.0 ** -64


def stats(verts, faces, vertex_body, B):
    """dict of the per-body arrays mesh_bodies computes."""
    v = np.asarray(verts, dtype=np.float32).reshape(-1, 3)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    lab = np.asarray(vertex_body)
    face_body = lab[f[:, 0]] if len(f) else np.zeros(0, np.int32)
    first = np.unique(lab, return_index=True)[1].astype(np.int64)   # every body 0..B-1 has a vertex
    box = np.empty((B, 6), np.float32)
    for c in range(3):
        lo = np.full(B, np.inf, np.float32)
        hi = np.full(B, -np.inf, np.float32)
        np.minimum.at(lo, lab, v[:, c])
        np.maximum.at(hi, lab, v[:, c])
        box[:, 2 * c], box[:, 2 * c + 1] = lo + np.float32(0), hi + np.float32(0)    # + 0: a zero bound is +0.0
    tv, ta = terms(v, f)
    return {"vertex_counts": np.bincount(lab, minlength=B).astype(np.int64),
            "face_counts": np.bincount(face_body, minlength=B).astype(np.int64),
            "first_vertex": first, "bbox_mm": box,
            "signed_volumes": np.array([fixed_to_f64(s) for s in fixed_sums(tv, face_body, B)], np.float64),
            "areas": np.array([fixed_to_f64(s) for s in fixed_sums(ta, face_body, B)], np.float64),
            "face_body": face_body.astype(np.int32)}


def select(verts, faces, vertex_body, keep, normals=None):
    """The kept bodies' vertices and faces in input order, faces (input dtype) renumbered with a cumsum of the vertex mask."""
    lab = np.asarray(vertex_body)
    f = np.asarray(faces)
    kb = np.zeros(int(lab.max()) + 1 if len(lab) else 0, bool)
    kb[np.asarray(keep, dtype=np.int64)] = True
    vm = kb[lab] if len(lab) else np.zeros(0, bool)
    newid = np.cumsum(vm) - 1
    fm = vm[f[:, 0]] if len(f) else np.zeros(0, bool)
    out = (np.asarray(verts)[vm], newid[f[fm]].astype(f.dtype).reshape(-1, 3))
    if normals is not None:
        out += (np.asarray(normals)[vm],)
    return out
