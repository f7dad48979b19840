// t3d_normals.cu -- field-gradient vertex normals of a marching-cubes mesh (DESIGN.md §2, "Vertex normals").
//
// One thread per raw vertex (the same keys, [x | y | z]-edge blocks, as k_mc_vertices_all).  For the vertex on grid edge
// a -> b of the marched field f (level L):
//   g[n]  = np.gradient(f.astype(float64)) at node n: (f[n+1] - f[n-1]) / 2 inside, one-sided f[1]-f[0] / f[-1]-f[-2] at
//           the first / last node of an axis;
//   G     = (1 - t) * g[a] + t * g[b], t = the vertex kernel's interpolation weight;
//   n     = -(Gz/dz, Gy/mm_y, Gx/mm_x) / |.|, float64, rounded to float32; dz = slope of the variable-depth z map there.
// Result rows are scattered into canonical slots through the raw -> canonical map of the canonicalisation (`newid`).
// Where np.unique merged raw vertices, the slot takes the normal of the raw vertex with the smallest edge key (z, y, x,
// axis): a tie pass over the sorted order picks that vertex first (skipped unless the unique pass saw an equal pair).
//
// Gaussian occupancy field: an edge needs f at 12 nodes (the four on its line, +-1 across both other axes at either end).
// They are evaluated from one fetch of the padded occupancy around the edge -- up to 8 planes x 8 rows x 8 x-bits, only
// the (plane, row) pairs some node reads -- with the 0/1 z pass done as 64-bit SWAR lookups (8 x columns at once), the
// same arithmetic as field_value().
#include "t3d.h"
#include "t3d_field.cuh"

#define NRM_EPS 2.220446049250313e-16   // np.spacing(1.0): skimage's vertex weights (as in t3d_mc.cu)

struct NormalArgs {
    OccView occ;               // Gaussian (or plain) padded occupancy; grid extents occ.Zp x occ.Hp x occ.Wp
    const float* field;        // or: dense float32 field of extents occ.Z x occ.H x occ.W (occ without bits, pad 0)
    double level;
    const unsigned long long* vkeys;
    const unsigned long long* sizes;   // device {n_active, n_x, n_y, n_z, ...}
    uint32_t cap_verts;        // nothing runs when n_x + n_y + n_z exceeds it
    int x_off;                 // key x minus this = x in the padded grid
    int z_offset;
    float shift;               // 1 if the vertices are un-padded
    const double* adj;         // adjusted slice depths (n_cum - 1 entries); n_cum = 0: no z map
    int n_cum;
    double mm_y, mm_x;
    const uint32_t* newid;     // raw -> canonical slot; null: raw order
    const uint32_t* perm;      // canonical sort order (position -> raw id); null: no vertex was merged
    const unsigned long long* dup;   // optional: the unique pass's "equal pair seen" flag (tie pass only if set)
    uint32_t* winner;          // per canonical slot: raw id whose normal it takes (tie pass scratch)
    float* normals;            // (V', 3) z, y, x
};

__device__ __forceinline__ uint32_t raw_count(const NormalArgs& p)
{
    const unsigned long long v = p.sizes[1] + p.sizes[2] + p.sizes[3];
    return v > p.cap_verts ? 0u : (uint32_t)v;
}

__device__ __forceinline__ bool ties_active(const NormalArgs& p) { return p.perm && (!p.dup || *p.dup); }

// bits of padded row (zp, yp) at padded x = xs .. xs+7 (x reflected at the padded border); zp, yp inside [0, Np)
__device__ __forceinline__ uint32_t get8(const OccView& v, int zp, int yp, int xs)
{
    const int z = zp - v.pad, y = yp - v.pad;
    if (z < 0 || z >= v.Z || y < 0 || y >= v.H) return 0u;
    const uint32_t* row = v.bits + (z * v.ps + (long long)y * v.rs);
    if (xs >= 0 && xs + 7 < v.Wp) {
        const int ox = xs - v.pad;
        const int w = ox >> 5, sh = ox & 31;
        const uint32_t lo = (w >= 0 && w < v.nw) ? row[w] : 0u;
        const uint32_t hi = (w + 1 >= 0 && w + 1 < v.nw) ? row[w + 1] : 0u;
        return __funnelshift_r(lo, hi, sh) & 255u;
    }
    uint32_t r = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int ox = reflect_idx(xs + k, v.Wp) - v.pad;
        if (ox >= 0 && ox < v.W) r |= ((row[ox >> 5] >> (ox & 31)) & 1u) << k;
    }
    return r;
}

// The 12 nodes of an edge along AXIS, offsets (dz, dy, dx) from its lower end a:
//   0..3: the line, offsets -1, 0, 1, 2 along AXIS (a = node 1, b = node 2);
//   4..11: node 4 + 4*j + 2*k + s = end k (0: a, 1: b) moved by -1 (s = 0) / +1 (s = 1) along the j-th other axis.
template <int AXIS>
struct EdgeNodes {
    __host__ __device__ static constexpr int other(int j) { return AXIS == 0 ? 1 + j : AXIS == 1 ? 2 * j : j; }
    __host__ __device__ static constexpr int off(int i, int ax)
    {
        return i < 4 ? (ax == AXIS ? i - 1 : 0)
                     : ((ax == AXIS ? ((i - 4) >> 1 & 1) : 0) + (ax == other((i - 4) >> 2) ? ((i & 1) ? 1 : -1) : 0));
    }
    // box plane bz / row by (origin -3 / -3 from a) is read by some node's 5 x 5 neighbourhood
    __host__ __device__ static constexpr bool used(int bz, int by)
    {
        bool u = false;
        for (int i = 0; i < 12; ++i) {
            const int dz = bz - 3 - off(i, 0), dy = by - 3 - off(i, 1);
            u = u || (dz >= -2 && dz <= 2 && dy >= -2 && dy <= 2);
        }
        return u;
    }
};

__device__ __forceinline__ unsigned long long spread8(const ZLut& L, uint32_t b)
{
    return (unsigned long long)L.spread[b & 63u] | ((unsigned long long)((b >> 6) & 1u) << 30) |
           ((unsigned long long)((b >> 7) & 1u) << 35);
}

// f at the 12 nodes of the edge (z, y, x) -> +1 along AXIS of the Gaussian of the padded occupancy (bit-exact with field_value)
template <int AXIS>
__device__ __forceinline__ void gaussian_nodes(const OccView& v, const ZLut& L, int z, int y, int x, float (&f)[12])
{
    using N = EdgeNodes<AXIS>;
    uint32_t box[8][8];
    const int oz0 = z - 3 - v.pad, oy0 = y - 3 - v.pad, ox0 = x - 3 - v.pad;
    if (oz0 >= 0 && oz0 + 8 <= v.Z && oy0 >= 0 && oy0 + 8 <= v.H && ox0 >= 0 && ox0 + 8 <= v.W) {
        const int sh = ox0 & 31;
        const bool two = sh > 24;   // the 8-bit window straddles two words
        const uint32_t* p = v.bits + (oz0 * v.ps + (long long)oy0 * v.rs) + (ox0 >> 5);
#pragma unroll
        for (int bz = 0; bz < 8; ++bz)
#pragma unroll
            for (int by = 0; by < 8; ++by) {
                if (!N::used(bz, by)) { box[bz][by] = 0u; continue; }
                const uint32_t* q = p + bz * v.ps + by * v.rs;
                box[bz][by] = __funnelshift_r(q[0], two ? q[1] : 0u, sh) & 255u;
            }
    } else {
#pragma unroll
        for (int bz = 0; bz < 8; ++bz) {
            const int zr = reflect_idx(z - 3 + bz, v.Zp);
#pragma unroll
            for (int by = 0; by < 8; ++by)
                box[bz][by] = N::used(bz, by) ? get8(v, zr, reflect_idx(y - 3 + by, v.Hp), x - 3) : 0u;
        }
    }
#pragma unroll
    for (int i = 0; i < 12; ++i) {
        const int dz = N::off(i, 0), dy = N::off(i, 1), dx = N::off(i, 2);
        // z pass of the five rows dy-2 .. dy+2 (all 8 x columns), y pass per x column, x pass
        unsigned long long idx[5];
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            const int by = dy + 1 + r;
            idx[r] = (spread8(L, box[dz + 1][by]) << 2) + spread8(L, box[dz + 2][by]) + (spread8(L, box[dz + 3][by]) << 4) +
                     spread8(L, box[dz + 4][by]) + (spread8(L, box[dz + 5][by]) << 2);
        }
        double Y[5];
#pragma unroll
        for (int c = 0; c < 5; ++c) {
            const int sh = 5 * (dx + 1 + c);
            Y[c] = corr5(L.z[(idx[0] >> sh) & 31u], L.z[(idx[1] >> sh) & 31u], L.z[(idx[2] >> sh) & 31u], L.z[(idx[3] >> sh) & 31u],
                         L.z[(idx[4] >> sh) & 31u], v.w0, v.w1, v.w2);
        }
        f[i] = __double2float_rn(corr5(Y[0], Y[1], Y[2], Y[3], Y[4], v.w0, v.w1, v.w2));
    }
}

// np.gradient along one axis at a node with coordinate c of n (f_m: node - 1, f_0: node, f_p: node + 1)
__device__ __forceinline__ double grad1(int c, int n, float f_m, float f_0, float f_p)
{
    if (c == 0) return __dsub_rn((double)f_p, (double)f_0);
    if (c == n - 1) return __dsub_rn((double)f_0, (double)f_m);
    return __ddiv_rn(__dsub_rn((double)f_p, (double)f_m), 2.0);
}

template <int AXIS>
__device__ __forceinline__ void normal_body(const NormalArgs& p, const ZLut& zlut, uint32_t id)
{
    using N = EdgeNodes<AXIS>;
    const uint32_t slot = p.newid ? p.newid[id] : id;
    if (p.perm && ties_active(p) && p.winner[slot] != id) return;
    const unsigned long long key = p.vkeys[id];
    const int x = (int)((key >> 2) & 0xfffffu) - p.x_off, y = (int)((key >> 22) & 0xfffffu), z = (int)(key >> 42);
    const int n3[3] = {p.occ.Zp, p.occ.Hp, p.occ.Wp};
    const int c3[3] = {z, y, x};
    float f[12];
    if (p.field) {
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            // nodes outside the grid are never used (one-sided differences there): clamp the address only
            const int zz = min(max(z + N::off(i, 0), 0), n3[0] - 1), yy = min(max(y + N::off(i, 1), 0), n3[1] - 1),
                      xx = min(max(x + N::off(i, 2), 0), n3[2] - 1);
            f[i] = p.field[((int64_t)zz * n3[1] + yy) * n3[2] + xx];
        }
    } else if (p.occ.gaussian) {
        gaussian_nodes<AXIS>(p.occ, zlut, z, y, x, f);
    } else {
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            const int zz = min(max(z + N::off(i, 0), 0), n3[0] - 1), yy = min(max(y + N::off(i, 1), 0), n3[1] - 1),
                      xx = min(max(x + N::off(i, 2), 0), n3[2] - 1);
            f[i] = pbit(p.occ, zz, yy, xx) ? 1.0f : 0.0f;
        }
    }
    // node gradients at a (k = 0) and b (k = 1), index space
    double g[2][3];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        g[k][AXIS] = grad1(c3[AXIS] + k, n3[AXIS], f[k], f[k + 1], f[k + 2]);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int ax = N::other(j);
            g[k][ax] = grad1(c3[ax], n3[ax], f[4 + 4 * j + 2 * k], f[1 + k], f[4 + 4 * j + 2 * k + 1]);
        }
    }
    // the vertex kernel's interpolation weight (vertex_body in t3d_mc.cu)
    const double va = (double)f[1] - p.level, vb = (double)f[2] - p.level;
    const double wa = __ddiv_rn(1.0, __dadd_rn(NRM_EPS, fabs(va)));
    const double wb = __ddiv_rn(1.0, __dadd_rn(NRM_EPS, fabs(vb)));
    const double t = __ddiv_rn(wb, __dadd_rn(wa, wb));
    const double s = __dsub_rn(1.0, t);
    double G[3];
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) G[ax] = __dadd_rn(__dmul_rn(s, g[0][ax]), __dmul_rn(t, g[1][ax]));
    // slope of the z map at the vertex: from the un-padded float32 z the vertex kernel forms
    double dz = 1.0;
    if (p.n_cum > 0) {
        double pz = (double)(z + p.z_offset);
        if (AXIS == 0) pz = __dadd_rn(pz, t);
        const float fz = __fsub_rn(__double2float_rn(pz), p.shift);
        if (fz < 0.0f) dz = p.adj[0];
        else if (fz >= (float)(p.n_cum - 1)) dz = p.adj[p.n_cum - 2];
        else dz = p.adj[min((int)floorf(fz), p.n_cum - 2)];
    }
    const double gz = __ddiv_rn(G[0], dz), gy = __ddiv_rn(G[1], p.mm_y), gx = __ddiv_rn(G[2], p.mm_x);
    const double nrm = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(gz, gz), __dmul_rn(gy, gy)), __dmul_rn(gx, gx)));
    float* o = p.normals + 3 * (int64_t)slot;
    if (nrm == 0.0) { o[0] = 0.0f; o[1] = 0.0f; o[2] = 0.0f; return; }
    o[0] = __double2float_rn(__ddiv_rn(-gz, nrm));
    o[1] = __double2float_rn(__ddiv_rn(-gy, nrm));
    o[2] = __double2float_rn(__ddiv_rn(-gx, nrm));
}

// one thread per raw vertex, all three axis blocks in one launch (as k_mc_vertices_all)
__global__ void __launch_bounds__(128) k_mc_normals(NormalArgs p)
{
    __shared__ ZLut zlut;
    fill_zlut(p.occ, zlut);
    __syncthreads();
    const uint32_t nx = (uint32_t)p.sizes[1], ny = (uint32_t)p.sizes[2];
    const uint32_t n = raw_count(p);
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    if (t < nx) normal_body<2>(p, zlut, t);
    else if (t < nx + ny) normal_body<1>(p, zlut, t);
    else normal_body<0>(p, zlut, t);
}

// tie rule: thread per sorted position; the first position of every canonical slot picks the raw vertex of smallest key
// among the (adjacent) positions that share the slot.  Returns at once unless the unique pass saw an equal pair.
__global__ void __launch_bounds__(256) k_mc_normal_ties(NormalArgs p)
{
    if (!ties_active(p)) return;
    const uint32_t n = raw_count(p);
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t raw = p.perm[i], slot = p.newid[raw];
    if (i > 0 && p.newid[p.perm[i - 1]] == slot) return;
    uint32_t best = raw;
    unsigned long long bk = p.vkeys[raw];
    for (uint32_t q = i + 1; q < n; ++q) {
        const uint32_t r = p.perm[q];
        if (p.newid[r] != slot) break;
        const unsigned long long k = p.vkeys[r];
        if (k < bk) { bk = k; best = r; }
    }
    p.winner[slot] = best;
}

static int launch_normals(NormalArgs& p, cudaStream_t st, const char* who)
{
    const uint32_t grid_verts = p.cap_verts;
    if (grid_verts == 0) return 0;
    int launches = 1;
    if (p.perm) {
        if (!p.newid || !p.winner) { t3d_set_error("%s: a sort order needs the map and the tie scratch", who); return 2; }
        k_mc_normal_ties<<<(grid_verts + 255) / 256, 256, 0, st>>>(p);
        ++launches;
    }
    k_mc_normals<<<(grid_verts + 127) / 128, 128, 0, st>>>(p);
    T3D_CHECK_LAUNCH(who);
    t3d_count_launches(launches);
    return 0;
}

static int make_args(NormalArgs& p, const void* occ_bits, int Z, int H, int W, int pad, int gaussian, const double* weights3_host,
                     const void* field_f32, double level, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts,
                     int unpad_shift, int z_offset, const void* adj_f64, int n_cum, double mm_y, double mm_x, const void* newid_u32,
                     const void* perm_u32, const void* dup_u64, void* winner_u32, void* normals_f32, const char* who)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("%s: empty volume", who); return 2; }
    if (field_f32) {
        p.occ = t3d_make_view(nullptr, Z, H, W, 0, 0, nullptr);
    } else {
        if (!gaussian && pad) { t3d_set_error("%s: pad requires gaussian", who); return 2; }
        p.occ = t3d_make_view(occ_bits, Z, H, W, pad, gaussian, weights3_host);
    }
    if (p.occ.Zp < 2 || p.occ.Hp < 2 || p.occ.Wp < 2) { t3d_set_error("%s: the marched grid must be at least 2x2x2", who); return 2; }
    p.field = (const float*)field_f32;
    p.level = field_f32 ? level : 0.5;
    p.vkeys = (const unsigned long long*)vkeys_u64;
    p.sizes = (const unsigned long long*)sizes_u64;
    p.cap_verts = cap_verts;
    p.x_off = 0;
    p.z_offset = z_offset;
    p.shift = unpad_shift ? 1.0f : 0.0f;
    p.adj = (const double*)adj_f64;
    p.n_cum = adj_f64 ? n_cum : 0;
    p.mm_y = mm_y; p.mm_x = mm_x;
    p.newid = (const uint32_t*)newid_u32;
    p.perm = (const uint32_t*)perm_u32;
    p.dup = (const unsigned long long*)dup_u64;
    p.winner = (uint32_t*)winner_u32;
    p.normals = (float*)normals_f32;
    return 0;
}

extern "C" int t3d_mc_normals_dev(const void* occ_bits, int Z, int H, int W, int pad, int gaussian, const double* weights3_host,
                                  const void* field_f32, double level, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts,
                                  int unpad_shift, int z_offset, const void* adj_f64, int n_cum, double mm_per_pixel_y,
                                  double mm_per_pixel_x, const void* newid_u32, const void* perm_u32, const void* dup_u64,
                                  void* winner_u32, void* normals_f32, void* stream)
{
    NormalArgs p;
    if (int rc = make_args(p, occ_bits, Z, H, W, pad, gaussian, weights3_host, field_f32, level, vkeys_u64, sizes_u64, cap_verts,
                           unpad_shift, z_offset, adj_f64, n_cum, mm_per_pixel_y, mm_per_pixel_x, newid_u32, perm_u32, dup_u64,
                           winner_u32, normals_f32, "t3d_mc_normals_dev"))
        return rc;
    return launch_normals(p, (cudaStream_t)stream, "t3d_mc_normals_dev");
}

// the fused step's variant: the field is a strided view whose padded x is the key's x minus x_off (t3d_pipeline.cu)
int t3d_mc_normals_view_dev(const OccView& view, int x_off, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts, int unpad_shift,
                            int z_offset, const void* adj_f64, int n_cum, double mm_per_pixel_y, double mm_per_pixel_x,
                            const void* newid_u32, const void* perm_u32, const void* dup_u64, void* winner_u32, void* normals_f32,
                            void* stream)
{
    NormalArgs p;
    if (int rc = make_args(p, view.bits, view.Z, view.H, view.W, view.pad, view.gaussian, nullptr, nullptr, 0.5, vkeys_u64, sizes_u64,
                           cap_verts, unpad_shift, z_offset, adj_f64, n_cum, mm_per_pixel_y, mm_per_pixel_x, newid_u32, perm_u32, dup_u64,
                           winner_u32, normals_f32, "t3d_reconstruct_normals"))
        return rc;
    p.occ = view;
    p.x_off = x_off;
    return launch_normals(p, (cudaStream_t)stream, "t3d_reconstruct_normals");
}
