"""CPU oracle of the field-gradient vertex normals (DESIGN.md §2, "Vertex normals"), built from numpy alone.

It does not go through oracle/mc_ref.c: the vertices are re-derived from the cut edges of the marched field (strict
`> level` signs, skimage's interpolation weight), un-padded, z-mapped and scaled like extract_manifold_surface, and ordered
with np.unique.  The normal of a vertex is the np.gradient of the field at the two end nodes of its edge, blended with the
vertex's weight, taken into the (z mm, y mm, x mm) frame and normalised; where np.unique merges several raw vertices the
one whose edge has the smallest key (z, y, x, axis) of its lower end gives the normal.
"""
import numpy as np

EPS = np.spacing(1.0)
AXIS_CODE = {2: 2, 1: 1, 0: 0}      # key code of an x / y / z edge (vkey() in csrc/t3d_mc.cu)


def _z_map(slice_depths, add_padding):
    sd = np.asarray(slice_depths, dtype=np.float64)
    if len(sd) == 0:
        return None, None
    adj = np.concatenate([[sd[0]], sd, [sd[-1]]]) if add_padding else sd
    return np.cumsum(np.concatenate([[0], adj])), adj


def cut_edge_vertices(f, level, slice_depths, mm_per_pixel_y, mm_per_pixel_x, add_padding=True, unpad=True):
    """Raw vertices of the field f in the kernels' raw order ([x | y | z]-edge blocks, raster order of the lower end), with
    per vertex: the lower end (z, y, x), the axis, t and the un-padded float32 z before the z map."""
    f = np.ascontiguousarray(f, dtype=np.float32)
    f64 = f.astype(np.float64)
    pos = (f64 - level) > 0
    out = []
    for axis in (2, 1, 0):
        n = f.shape[axis]
        sl_a = [slice(None)] * 3
        sl_b = [slice(None)] * 3
        sl_a[axis], sl_b[axis] = slice(0, n - 1), slice(1, n)
        cut = pos[tuple(sl_a)] != pos[tuple(sl_b)]
        z, y, x = (c.astype(np.int64) for c in np.nonzero(cut))
        a = [z, y, x]
        b = [z.copy(), y.copy(), x.copy()]
        b[axis] = b[axis] + 1
        va = f64[z, y, x] - level
        vb = f64[b[0], b[1], b[2]] - level
        wa = 1.0 / (EPS + np.abs(va))
        wb = 1.0 / (EPS + np.abs(vb))
        t = wb / (wa + wb)
        p = [z.astype(np.float64), y.astype(np.float64), x.astype(np.float64)]
        p[axis] = p[axis] + t
        out.append((np.stack(a, 1), np.full(len(z), axis), t, [c.astype(np.float32) for c in p]))
    lo = np.concatenate([o[0] for o in out])
    axes = np.concatenate([o[1] for o in out])
    t = np.concatenate([o[2] for o in out])
    verts = np.stack([np.concatenate([o[3][k] for o in out]) for k in range(3)], 1)
    if unpad:
        verts -= np.float32(1)
    fz = verts[:, 0].copy()
    cum, adj = _z_map(slice_depths, add_padding)
    if cum is not None:
        zc = verts[:, 0]
        lo_z = np.floor(zc)
        neg, big = zc < 0, zc >= len(cum) - 1
        mid = ~(neg | big)
        loi = lo_z[mid].astype(np.int64)
        frac = (zc[mid] - lo_z[mid]).astype(np.float32)
        z_out = np.empty_like(zc)
        z_out[neg] = 0
        z_out[big] = cum[-1]
        z_out[mid] = (cum[loi] + frac.astype(np.float64) * adj[np.minimum(loi, len(adj) - 1)]).astype(np.float32)
        verts[:, 0] = z_out
    verts[:, 1] *= mm_per_pixel_y
    verts[:, 2] *= mm_per_pixel_x
    return verts, lo, axes, t, fz


def raw_normals(f, level, lo, axes, t, fz, slice_depths, mm_per_pixel_y, mm_per_pixel_x, add_padding=True):
    """The normal of every raw vertex (float32 (n, 3) [z, y, x])."""
    f64 = np.asarray(f, dtype=np.float32).astype(np.float64)
    g = np.gradient(f64)
    b = lo.copy()
    b[np.arange(len(lo)), axes] += 1
    ga = np.stack([g[k][lo[:, 0], lo[:, 1], lo[:, 2]] for k in range(3)], 1)
    gb = np.stack([g[k][b[:, 0], b[:, 1], b[:, 2]] for k in range(3)], 1)
    G = (1.0 - t)[:, None] * ga + t[:, None] * gb
    cum, adj = _z_map(slice_depths, add_padding)
    if cum is None:
        dz = np.ones(len(t))
    else:
        n_cum = len(cum)
        dz = np.empty(len(t))
        neg, big = fz < 0, fz >= n_cum - 1
        mid = ~(neg | big)
        dz[neg] = adj[0]
        dz[big] = adj[n_cum - 2]
        dz[mid] = adj[np.minimum(np.floor(fz[mid]).astype(np.int64), n_cum - 2)]
    gz, gy, gx = G[:, 0] / dz, G[:, 1] / float(mm_per_pixel_y), G[:, 2] / float(mm_per_pixel_x)
    nrm = np.sqrt(gz * gz + gy * gy + gx * gx)
    out = np.zeros((len(t), 3), dtype=np.float32)
    ok = nrm != 0
    out[ok, 0] = (-gz[ok] / nrm[ok]).astype(np.float32)
    out[ok, 1] = (-gy[ok] / nrm[ok]).astype(np.float32)
    out[ok, 2] = (-gx[ok] / nrm[ok]).astype(np.float32)
    return out


def edge_keys(lo, axes):
    """(z, y, x, axis) of the lower end as one integer, ordered like vkey() in csrc/t3d_mc.cu."""
    code = np.array([AXIS_CODE[0], AXIS_CODE[1], AXIS_CODE[2]], dtype=np.int64)[axes]
    return code | (lo[:, 2] << 2) | (lo[:, 1] << 22) | (lo[:, 0] << 42)


def canonical_normals(verts, normals, keys):
    """np.unique order of the vertices; a merged vertex takes the normal of the raw vertex of smallest key.  Returns
    (unique vertices, their normals, number of raw vertices that were merged away)."""
    uv, inv = np.unique(verts, axis=0, return_inverse=True)
    inv = np.asarray(inv).reshape(-1)
    order = np.argsort(keys, kind="stable")
    _, first = np.unique(inv[order], return_index=True)
    winners = order[first]
    out = np.empty((len(uv), 3), dtype=np.float32)
    out[inv[winners]] = normals[winners]
    return uv, out, len(verts) - len(uv)


def gradient_normals(volume_data, slice_depths, mm_per_pixel_y, mm_per_pixel_x, manifold=True, add_padding=True, field=None):
    """(vertices, normals) of extract_manifold_surface(volume_data, ...) -- canonical order when manifold, raw order
    otherwise -- from the occupancy's marched field (oracle.cpu_ref.scalar_field)."""
    from oracle import cpu_ref
    f = cpu_ref.scalar_field(volume_data, manifold, add_padding) if field is None else field
    verts, lo, axes, t, fz = cut_edge_vertices(f, 0.5, slice_depths, mm_per_pixel_y, mm_per_pixel_x, add_padding, unpad=manifold)
    n = raw_normals(f, 0.5, lo, axes, t, fz, slice_depths, mm_per_pixel_y, mm_per_pixel_x, add_padding)
    if not manifold:
        return verts, n
    uv, un, _ = canonical_normals(verts, n, edge_keys(lo, axes))
    return uv, un


def gradient_normals_dense(field, level, slice_depths, mm_per_pixel_y, mm_per_pixel_x):
    """(vertices, normals, merged count) of SurfaceExtractor.extract_surface_from_sdf(field, ..., level): the dense field
    marched as it is (no padding, no un-pad shift, z map without end padding), canonical order."""
    verts, lo, axes, t, fz = cut_edge_vertices(field, level, slice_depths, mm_per_pixel_y, mm_per_pixel_x, False, unpad=False)
    n = raw_normals(field, level, lo, axes, t, fz, slice_depths, mm_per_pixel_y, mm_per_pixel_x, False)
    return canonical_normals(verts, n, edge_keys(lo, axes))
