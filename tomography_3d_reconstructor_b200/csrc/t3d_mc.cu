// t3d_mc.cu -- two-pass marching cubes on the packed sign volume (sm_100a).
//
// Replaces skimage.measure.marching_cubes(volume, level=0.5) as called at surface_extractor.py:55, plus the vertex
// post-transform of surface_extractor.py:57-65 / 82-113.  See SURVEY.md 8a-7, 8a-8.
//
// Work is proportional to the SURFACE, not the volume, after one cheap dense pass:
//   1. t3d_mc_flags    dense, one thread per 32-voxel word of the sign volume: does this word own a cut edge or the
//                      origin of an active cube?  -> one ballot word per warp (1 bit per word).
//   2. exclusive scan  of the ballot popcounts  -> rank of every active word (order-preserving compaction).
//   3. t3d_mc_words_dev    active words only: packed counts of owned x/y/z cut edges and triangles -> compact arrays.
//   4. exclusive scan      of those counts -> vertex / triangle bases per active word.
//   5. t3d_mc_emit_dev     one thread per active word: edge keys of the owned vertices, faces of its cubes
//                          (ids of vertices owned by neighbouring words through ballot-rank lookups).
//   6. t3d_mc_vertices_dev one thread per vertex: exact float64 field at the two end points, skimage's interpolation,
//                          un-pad, variable-depth z map, mm scaling.
// Steps 3, 5 and 6 read the data-dependent sizes from a device block {n_active, n_x, n_y, n_z, n_t} (scan totals).
// Vertex ids: [x-edge vertices | y-edge | z-edge], each in raster order of the owning voxel (edge owned by its lower
// corner).  Faces come out in the reference's order: cubes z-major, y, x fastest, table order inside a cube,
// winding reversed (gradient_direction='descent').
#include "mc_tables.h"
#include "mc33_tables.h"
#include "t3d.h"
#include "t3d_field.cuh"

// ------------------------------------------------------------------------------------------------
// tables
// ------------------------------------------------------------------------------------------------
__device__ __align__(16) const int8_t g_tri_table[256][T3D_MC_ROW] = {T3D_TRI_TABLE_ROWS};
static const int8_t h_tri_table[256][T3D_MC_ROW] = {T3D_TRI_TABLE_ROWS};

struct McLuts {
    uint8_t ntri[256];   // triangles of the classic row; bit 7 (MC_AMB): the index has an ambiguous face or is Lewiner's case 4
                         // -> resolved per cube (mc33_resolve).  One byte, one (divergent) constant load per cube.
};
#define MC_AMB 0x80u
__constant__ McLuts c_luts;

// Tilings of the ambiguous configurations (generated, tools/gen_mc33_tables.py): row = base[index] + (J | tube << k), J = bit i
// set iff the positive corners are joined across the i-th ambiguous face, tube = the interior test asks for a tunnel.
// These tables are only touched by cubes with an ambiguous index (none on smooth closed surfaces, a few % on noise).
__device__ const int8_t g33_rows[T3D_MC33_NROWS][T3D_MC33_ROW] = {T3D_MC33_TRI_ROWS};
__device__ const uint8_t g33_ntri[T3D_MC33_NROWS] = {T3D_MC33_NTRI_VALUES};
__device__ const uint16_t g33_base[256] = {T3D_MC33_BASE_VALUES};
__device__ const uint8_t g33_k[256] = {T3D_MC33_K_VALUES};
__device__ const uint8_t g33_faces[256][6] = {T3D_MC33_FACES_VALUES};
__device__ const unsigned long long g33_need[256] = {T3D_MC33_NEED_VALUES};
__device__ const uint8_t g33_pol[256] = {T3D_MC33_POL_VALUES};
__device__ const int8_t g33_sign[256] = {T3D_MC33_SIGN_VALUES};
__device__ const uint8_t g33_cyc[6][4] = {T3D_MC33_FACE_CYCLE_VALUES};
static const uint16_t h33_base[256] = {T3D_MC33_BASE_VALUES};

// The marched field as the ambiguity tests see it (value - level at the 8 corners of a cube).
//   mode 0: only the sign volume is known: value - level = +-0.5 (every face test is a tie -> positives joined)
//   mode 1: Gaussian(0.5) of the padded occupancy `occ` (or the occupancy itself), evaluated exactly like the vertex kernel
//   mode 2: dense float32 field of the sign volume's own shape (SDF path)
struct McField {
    OccView occ;
    const float* field;
    double level;
    int x_off;      // sign-volume x minus this = x in occ's padded grid (padded-storage layout of the fused pipeline)
    int mode;
};

#define MC33_EPS 2.220446049250313e-16   // np.spacing(1.0): skimage's `FLT_EPSILON` (tie threshold of the face test, vertex weights)

// Lewiner's test_face in the form "are the POSITIVE corners joined across face f" (oracle/mc_ref.c: face_joined)
__device__ __forceinline__ int mc33_face_joined(const double* v, int f)
{
    const double A = v[g33_cyc[f][0]], B = v[g33_cyc[f][1]], C = v[g33_cyc[f][2]], D = v[g33_cyc[f][3]];
    const double ac = __dmul_rn(A, C), bd = __dmul_rn(B, D);
    const double det = (A > 0.0) ? __dsub_rn(ac, bd) : __dsub_rn(bd, ac);
    return det > -MC33_EPS;
}

// Lewiner's test_interior, z-sweep variant (oracle/mc_ref.c: interior_test): 1 = the s-signed corners are NOT joined inside
__device__ __forceinline__ int mc33_interior_test(const double* v, int s)
{
    const double d40 = __dsub_rn(v[4], v[0]), d62 = __dsub_rn(v[6], v[2]), d73 = __dsub_rn(v[7], v[3]), d51 = __dsub_rn(v[5], v[1]);
    const double a = __dsub_rn(__dmul_rn(d40, d62), __dmul_rn(d73, d51));
    const double b = __dsub_rn(__dsub_rn(__dadd_rn(__dmul_rn(v[2], d40), __dmul_rn(v[0], d62)), __dmul_rn(v[1], d73)), __dmul_rn(v[3], d51));
    const double t = __ddiv_rn(-b, __dmul_rn(2.0, a));
    if (t < 0.0 || t > 1.0) return s > 0;
    const double At = __dadd_rn(v[0], __dmul_rn(d40, t)), Bt = __dadd_rn(v[3], __dmul_rn(d73, t));
    const double Ct = __dadd_rn(v[2], __dmul_rn(d62, t)), Dt = __dadd_rn(v[1], __dmul_rn(d51, t));
    const int test = (At >= 0.0 ? 1 : 0) | (Bt >= 0.0 ? 2 : 0) | (Ct >= 0.0 ? 4 : 0) | (Dt >= 0.0 ? 8 : 0);
    const double dec = __dsub_rn(__dmul_rn(At, Ct), __dmul_rn(Bt, Dt));
    switch (test) {
    case 5: if (dec < MC33_EPS) return s > 0; break;
    case 10: if (dec >= MC33_EPS) return s > 0; break;
    case 7: case 11: case 13: case 14: case 15: return s < 0;
    default: return s > 0;
    }
    return s < 0;
}

// row of g33_rows for the cube with origin (z, y, x) of the sign volume and ambiguous index cs
__device__ __noinline__ int mc33_resolve(const McField& f, int z, int y, int x, int cs)
{
    double v[8];
#pragma unroll 1
    for (int c = 0; c < 8; ++c) {
        const int dz = c >> 2, dy = (c >> 1) & 1, dx = (c ^ (c >> 1)) & 1;
        float val;
        if (f.mode == 1) val = field_value(f.occ, z + dz, y + dy, x - f.x_off + dx);
        else if (f.mode == 2) val = f.field[((int64_t)(z + dz) * f.occ.H + (y + dy)) * f.occ.W + (x + dx)];
        else val = ((cs >> c) & 1) ? 1.0f : 0.0f;
        v[c] = __dsub_rn((double)val, f.level);
    }
    const int k = g33_k[cs];
    int J = 0, tube = 0;
    for (int i = 0; i < k; ++i) J |= mc33_face_joined(v, g33_faces[cs][i]) << i;
    if ((g33_need[cs] >> J) & 1ull) {
        const int I = mc33_interior_test(v, g33_sign[cs]);
        tube = g33_pol[cs] ? I : !I;
    }
    return (int)g33_base[cs] + (J | (tube << k));
}

static McField mc_field_from_abi(const t3d_mc_field* a)
{
    McField f;
    f.field = nullptr; f.level = 0.5; f.x_off = 0; f.mode = 0;
    f.occ = t3d_make_view(nullptr, 1, 1, 1, 0, 0, nullptr);
    if (!a) return f;
    f.level = a->level;
    if (a->field_f32) {
        f.occ = t3d_make_view(nullptr, a->Z, a->H, a->W, 0, 0, nullptr);
        f.field = (const float*)a->field_f32;
        f.mode = 2;
    } else if (a->occ_bits) {
        f.occ = t3d_make_view(a->occ_bits, a->Z, a->H, a->W, a->pad, a->gaussian, a->weights3_host);
        f.mode = 1;
    }
    return f;
}

static int ensure_luts()
{
    if (!t3d_first_use_on_device(T3D_ONCE_MC_LUTS)) return 0;   // __constant__ memory is per device
    McLuts l;
    for (int i = 0; i < 256; ++i) {
        int n = 0;
        while (n < T3D_MC_ROW && h_tri_table[i][n] >= 0) n += 3;
        l.ntri[i] = (uint8_t)(n / 3) | (uint8_t)(h33_base[i] != T3D_MC33_NONE ? MC_AMB : 0u);
    }
    T3D_CUDA(cudaMemcpyToSymbol(c_luts, &l, sizeof(l)));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// per-word bit arithmetic
// ------------------------------------------------------------------------------------------------
struct Grid {
    const uint32_t* sign;
    int Zs, Hs, Ws, nws;
    int z_begin, z_end; // planes [z_begin, z_end) are owned (vertices + cube layers); plane z_end, if it exists, is a
                        // ghost plane: its x/y-edge vertices are emitted too (the cubes of layer z_end-1 use them) but
                        // it owns no z-edges and no cubes.  Single device: [0, Zs).  z-slab sharding: see sharded.py.
    int ncr;            // 32-word chunks per row = ceil(nws/32); one ballot word per (row, chunk)
    uint32_t n_rows;    // Zs*Hs
    int64_t n_words;    // n_rows*nws (flat word index i = row*nws + w)
};

struct WordMasks {
    uint32_t s00, s01, s10, s11;  // rows (z,y) (z,y+1) (z+1,y) (z+1,y+1), word w
    uint32_t a00, a01, a10, a11;  // the same rows shifted: value at x+1
    uint32_t X00, X01, X10, X11;  // cut x-edges owned by each row's word
    uint32_t Y0, Y1;              // cut y-edges owned by rows (z,y), (z+1,y)
    uint32_t Z0, Z1;              // cut z-edges owned by rows (z,y), (z,y+1)
    uint32_t act;                 // origins of active cubes
};

__device__ __forceinline__ uint32_t shr1(uint32_t s, uint32_t nbit) { return (s >> 1) | (nbit << 31); }

// s*: words of the four rows, n*: bit 0 of the next word of each row
__device__ __forceinline__ WordMasks make_masks(uint32_t s00, uint32_t s01, uint32_t s10, uint32_t s11, uint32_t n00,
                                                uint32_t n01, uint32_t n10, uint32_t n11, bool hy, bool hz, int w, int Ws,
                                                bool own = true)
{
    WordMasks m;
    hz = hz && own;  // a ghost plane owns neither z-edges nor cubes
    const uint32_t vm = valid_mask(w, Ws), em = valid_mask(w, Ws - 1);  // em: x+1 still inside the grid
    m.s00 = s00; m.s01 = s01; m.s10 = s10; m.s11 = s11;
    m.a00 = shr1(s00, n00); m.a01 = shr1(s01, n01); m.a10 = shr1(s10, n10); m.a11 = shr1(s11, n11);
    m.X00 = (s00 ^ m.a00) & em;
    m.X01 = hy ? (s01 ^ m.a01) & em : 0u;
    m.X10 = hz ? (s10 ^ m.a10) & em : 0u;
    m.X11 = (hy && hz) ? (s11 ^ m.a11) & em : 0u;
    m.Y0 = hy ? (s00 ^ s01) & vm : 0u;
    m.Y1 = (hy && hz) ? (s10 ^ s11) & vm : 0u;
    m.Z0 = hz ? (s00 ^ s10) & vm : 0u;
    m.Z1 = (hy && hz) ? (s01 ^ s11) & vm : 0u;
    m.act = 0u;
    if (hy && hz) {
        const uint32_t o = s00 | s01 | s10 | s11, a = s00 & s01 & s10 & s11;
        const uint32_t oa = m.a00 | m.a01 | m.a10 | m.a11, aa = m.a00 & m.a01 & m.a10 & m.a11;
        m.act = ((o | oa) & ~(a & aa)) & em;
    }
    return m;
}

__device__ __forceinline__ int cube_case(const WordMasks& m, int b)
{
    return (int)(((m.s00 >> b) & 1u) | (((m.a00 >> b) & 1u) << 1) | (((m.a01 >> b) & 1u) << 2) | (((m.s01 >> b) & 1u) << 3) |
                 (((m.s10 >> b) & 1u) << 4) | (((m.a10 >> b) & 1u) << 5) | (((m.a11 >> b) & 1u) << 6) | (((m.s11 >> b) & 1u) << 7));
}

// masks of word w of voxel row `row`, loading everything from memory (sparse kernels)
__device__ __forceinline__ WordMasks load_masks(const Grid& g, uint32_t row, int w, int& z, int& y)
{
    z = (int)(row / (uint32_t)g.Hs);
    y = (int)(row - (uint32_t)z * (uint32_t)g.Hs);
    const bool hy = (y + 1 < g.Hs), hz = (z + 1 < g.Zs), hx = (w + 1 < g.nws);
    const uint32_t* p = g.sign + (int64_t)row * g.nws + w;
    const int64_t dy = g.nws, dz = (int64_t)g.Hs * g.nws;
    const uint32_t s00 = p[0], s01 = hy ? p[dy] : 0u, s10 = hz ? p[dz] : 0u, s11 = (hy && hz) ? p[dz + dy] : 0u;
    uint32_t n00 = 0, n01 = 0, n10 = 0, n11 = 0;
    if (hx) {
        n00 = p[1] & 1u;
        if (hy) n01 = p[dy + 1] & 1u;
        if (hz) n10 = p[dz + 1] & 1u;
        if (hy && hz) n11 = p[dz + dy + 1] & 1u;
    }
    return make_masks(s00, s01, s10, s11, n00, n01, n10, n11, hy, hz, w, g.Ws, z < g.z_end);
}

// ------------------------------------------------------------------------------------------------
// 1. dense flags.  Same shape as the morphology kernels: a thread owns one uint4 column (128 voxels) of one plane
// and marches down GY rows, keeping the rows (z,y) and (z+1,y) in registers, so every sign word is loaded twice
// (as plane z and as plane z+1).  Active words are rare (a few % of all words): each thread ORs its four flag bits
// into the pre-zeroed bitmap (one bit per word, one 32-bit word per (row, 32-word chunk)) only when non-zero.
// ------------------------------------------------------------------------------------------------
#define GY 16

__global__ void __launch_bounds__(256, 4) k_mc_flags(Grid g, uint32_t* __restrict__ ballots, int lanes_x, int pz_per_block, int gy)
{
    const int lx = threadIdx.x % lanes_x, pz = threadIdx.x / lanes_x;
    const int nws4 = g.nws >> 2;
    const int w4 = blockIdx.x * lanes_x + lx, z = g.z_begin + blockIdx.z * pz_per_block + pz, y0 = blockIdx.y * gy;
    if (pz >= pz_per_block || w4 >= nws4 || z >= g.Zs || z > g.z_end) return;
    const bool hz = (z + 1 < g.Zs) && (z < g.z_end);  // ghost plane: x/y edges only
    const bool hx = (4 * w4 + 4 < g.nws);
    const uint4 vm = valid_mask4(w4, g.Ws), em = valid_mask4(w4, g.Ws - 1);
    const uint4 zero = make_uint4(0, 0, 0, 0);
    // running pointers: row (z, y) and row (z+1, y) of this uint4 column, the bitmap word of (z, y)
    const uint32_t* p0 = g.sign + ((long long)z * g.Hs + y0) * g.nws + 4 * w4;
    const uint32_t* p1 = p0 + (long long)g.Hs * g.nws;
    uint32_t* pb = ballots + ((long long)z * g.Hs + y0) * g.ncr + (w4 >> 3);
    const uint32_t bshift = (4 * w4) & 31;
    uint4 c0 = *reinterpret_cast<const uint4*>(p0), c1 = hz ? *reinterpret_cast<const uint4*>(p1) : zero;  // rows (z,y), (z+1,y)
    uint32_t n0 = hx ? p0[4] : 0u, n1 = (hx && hz) ? p1[4] : 0u;
    const int y1 = min(g.Hs, y0 + gy);
    // rows (z,y+1), (z+1,y+1) are loaded one iteration ahead of their use (two rows of loads in flight per thread: the loop
    // was bound by the latency of its single outstanding row at volumes beyond L2)
    auto load_row = [&](int y, uint4& d0, uint4& d1, uint32_t& m0, uint32_t& m1) {
        const bool hy = (y < g.Hs);
        d0 = hy ? *reinterpret_cast<const uint4*>(p0) : zero;
        d1 = (hy && hz) ? *reinterpret_cast<const uint4*>(p1) : zero;
        m0 = (hy && hx) ? p0[4] : 0u;
        m1 = (hy && hz && hx) ? p1[4] : 0u;
    };
    uint4 e0, e1; uint32_t q0, q1;           // the prefetched row
    p0 += g.nws; p1 += g.nws;
    load_row(y0 + 1, e0, e1, q0, q1);
    for (int y = y0; y < y1; ++y) {
        const bool hy = (y + 1 < g.Hs);
        const uint4 d0 = e0, d1 = e1;
        const uint32_t m0 = q0, m1 = q1;
        p0 += g.nws; p1 += g.nws;
        if (y + 1 < y1) load_row(y + 2, e0, e1, q0, q1);
        uint4 f;  // owned cut edges | active cube origins
        if (hy && hz) {
            // The common row.  A cube is active iff its 8 corners are not all equal: iff one of its two x slices (the four
            // values at x, the four at x+1) is non-uniform, or the slices differ at one corner.  u = non-uniformity of the
            // slice at x costs two operations per word and its value at x+1 is one funnel shift -- 2 shifts + 5 logic
            // operations per word where OR / AND over the eight shifted corners took 4 + 14.  The owned y / z edges are
            // yz = (c0^d0)|(c0^c1) (they matter beyond `em` only, in the last valid column); the owned x edge c0^a0 is
            // part of the cube test.
            const uint32_t un = (n0 ^ n1) | (n0 ^ m0) | (m0 ^ m1);            // slice non-uniformity of the next word (bit 0 used)
            uint4 yz, u;
            yz.x = (c0.x ^ d0.x) | (c0.x ^ c1.x); yz.y = (c0.y ^ d0.y) | (c0.y ^ c1.y);
            yz.z = (c0.z ^ d0.z) | (c0.z ^ c1.z); yz.w = (c0.w ^ d0.w) | (c0.w ^ c1.w);
            u.x = yz.x | (d0.x ^ d1.x); u.y = yz.y | (d0.y ^ d1.y); u.z = yz.z | (d0.z ^ d1.z); u.w = yz.w | (d0.w ^ d1.w);
            const uint4 us = shr1_4(u, un), a0 = shr1_4(c0, n0);
            f.x = ((u.x | us.x | (c0.x ^ a0.x)) & em.x) | (yz.x & vm.x);
            f.y = ((u.y | us.y | (c0.y ^ a0.y)) & em.y) | (yz.y & vm.y);
            f.z = ((u.z | us.z | (c0.z ^ a0.z)) & em.z) | (yz.z & vm.z);
            f.w = ((u.w | us.w | (c0.w ^ a0.w)) & em.w) | (yz.w & vm.w);
        } else {
            // last row of a plane / last or ghost plane: owned edges only (no cube starts here)
            const uint4 a0 = shr1_4(c0, n0);
            f.x = ((c0.x ^ a0.x) & em.x); f.y = ((c0.y ^ a0.y) & em.y); f.z = ((c0.z ^ a0.z) & em.z); f.w = ((c0.w ^ a0.w) & em.w);
            if (hy) { f.x |= (c0.x ^ d0.x) & vm.x; f.y |= (c0.y ^ d0.y) & vm.y; f.z |= (c0.z ^ d0.z) & vm.z; f.w |= (c0.w ^ d0.w) & vm.w; }
            if (hz) { f.x |= (c0.x ^ c1.x) & vm.x; f.y |= (c0.y ^ c1.y) & vm.y; f.z |= (c0.z ^ c1.z) & vm.z; f.w |= (c0.w ^ c1.w) & vm.w; }
        }
        const uint32_t nib = (f.x ? 1u : 0u) | (f.y ? 2u : 0u) | (f.z ? 4u : 0u) | (f.w ? 8u : 0u);
        if (nib) atomicOr(pb, nib << bshift);
        pb += g.ncr;
        c0 = d0; c1 = d1; n0 = m0; n1 = m1;
    }
}

// ------------------------------------------------------------------------------------------------
// 3a. compaction: flat index of every active word, in raster order (thread per bitmap word)
// 3b. counts of the active words (thread per active word)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_mc_compact(Grid g, const uint32_t* __restrict__ ballots,
                                                    const uint32_t* __restrict__ chunkbase, int64_t n_chunks,
                                                    uint32_t* __restrict__ aw_idx, uint32_t cap_active)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    uint32_t bal = ballots[c];
    if (!bal) return;
    uint32_t k = chunkbase[c];
    const uint32_t row = (uint32_t)(c / g.ncr);
    const uint32_t base = row * (uint32_t)g.nws + (uint32_t)((c - (int64_t)row * g.ncr) << 5);
    while (bal) {
        const int b = __ffs(bal) - 1;
        bal &= bal - 1;
        if (k < cap_active) aw_idx[k] = base + b;  // beyond the capacity: dropped, the caller sees n_active > capacity
        ++k;
    }
}

#define AW_AMB 0x80000000u     // bit 31 of an aw_idx entry: the word holds a cube with an ambiguous index (set by k_mc_words<0>)
#define AW_MASK 0x7fffffffu

// AMB = 0: every active word -- counts with the CLASSIC triangle counts, words holding an ambiguous cube are flagged in aw_idx.
// AMB = 1: the flagged words only -- the classic count of every ambiguous cube is replaced by the count of the row Lewiner's
//          tests select.  Two kernels so that the common one carries neither the call nor its registers / stack frame
//          (with the tests inlined behind a branch it ran at 28 us instead of 17 at 512 x 1024 x 1024).
template <int AMB>
__global__ void __launch_bounds__(128) k_mc_words(Grid g, McField fld, uint32_t* __restrict__ aw_idx, uint32_t cap_active,
                                                  const unsigned long long* __restrict__ n_active_dev, uint32_t* __restrict__ aw_cnt,
                                                  unsigned long long* __restrict__ n_ambiguous)
{
    const uint32_t n_active = cap_active;  // array stride
    const int64_t n = dev_n(cap_active, n_active_dev);
    if (!AMB) {
        const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
        if ((int64_t)k >= n) return;
        const uint32_t i = aw_idx[k];
        const uint32_t row = i / (uint32_t)g.nws;
        const int w = (int)(i - row * (uint32_t)g.nws);
        int z, y;
        const WordMasks m = load_masks(g, row, w, z, y);
        uint32_t nt = 0, amb = 0;
        for (uint32_t a = m.act; a;) {        // branch-free: classic triangle counts, ambiguous cubes only noted
            const int b = __ffs(a) - 1;
            a &= a - 1;
            const uint32_t c = c_luts.ntri[cube_case(m, b)];
            nt += c & 0x7fu;
            amb |= c;
        }
        aw_cnt[k] = __popc(m.X00);
        aw_cnt[(int64_t)n_active + k] = __popc(m.Y0);
        aw_cnt[2 * (int64_t)n_active + k] = __popc(m.Z0);
        aw_cnt[3 * (int64_t)n_active + k] = nt;
        if (amb & MC_AMB) aw_idx[k] = i | AW_AMB;
    } else {
        // a fixed, small grid striding over the word list: nearly every entry is skipped (a capacity-sized launch of
        // threads that return at once cost 10 us of CTA launches at 512 x 1024 x 1024)
        uint32_t na = 0;
        auto fix_word = [&](int64_t k, uint32_t iraw) {
            const uint32_t i = iraw & AW_MASK;
            const uint32_t row = i / (uint32_t)g.nws;
            const int w = (int)(i - row * (uint32_t)g.nws);
            int z, y;
            const WordMasks m = load_masks(g, row, w, z, y);
            int delta = 0;
            for (uint32_t a = m.act; a;) {
                const int b = __ffs(a) - 1;
                a &= a - 1;
                const int cs = cube_case(m, b);
                const uint32_t c = c_luts.ntri[cs];
                if (!(c & MC_AMB)) continue;
                delta += (int)g33_ntri[mc33_resolve(fld, z, y, (w << 5) + b, cs)] - (int)(c & 0x7fu);
                ++na;
            }
            aw_cnt[3 * (int64_t)n_active + k] += (uint32_t)delta;
        };
        // four list entries per load (the list is 16-byte aligned): the scan for flag bits is what this launch spends its time on
        const int64_t n4 = ((uintptr_t)aw_idx & 15) ? 0 : (n >> 2), stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        for (int64_t c = t0; c < n4; c += stride) {
            const uint4 v = reinterpret_cast<const uint4*>(aw_idx)[c];
            if (!((v.x | v.y | v.z | v.w) & AW_AMB)) continue;
            if (v.x & AW_AMB) fix_word(4 * c, v.x);
            if (v.y & AW_AMB) fix_word(4 * c + 1, v.y);
            if (v.z & AW_AMB) fix_word(4 * c + 2, v.z);
            if (v.w & AW_AMB) fix_word(4 * c + 3, v.w);
        }
        for (int64_t k = 4 * n4 + t0; k < n; k += stride) {      // (the last n % 4 entries)
            const uint32_t iraw = aw_idx[k];
            if (iraw & AW_AMB) fix_word(k, iraw);
        }
        if (na) atomicAdd(n_ambiguous, (unsigned long long)na);
    }
}

// grid of the launches that stride over the word list looking for flagged words
static unsigned amb_grid(uint32_t n) { const unsigned want = (n + 127) / 128, cap = (unsigned)T3D_NUM_SMS * 8; return want < cap ? (want ? want : 1) : cap; }

// ------------------------------------------------------------------------------------------------
// 5. emit: one thread per active word
// ------------------------------------------------------------------------------------------------
struct EmitArgs {
    Grid g;
    McField fld;
    const uint32_t* ballots;
    const uint32_t* chunkbase;
    const uint32_t* aw_idx;
    const uint32_t* aw_base;  // 4 arrays, `cap_active` elements apart: X, Y, Z, T (exclusive scans)
    uint32_t cap_active;      // capacity of the word arrays
    const unsigned long long* sizes;  // device block {n_active, n_x, n_y, n_z, n_t}
    uint32_t cap_verts, cap_faces;    // nothing is written beyond these
    unsigned long long* vkeys;  // per vertex: axis | x << 2 | y << 22 | z << 42
    int32_t* faces;
};

// rank of word w of row `row` among the active words (the word must be active)
__device__ __forceinline__ uint32_t active_rank(const EmitArgs& a, uint32_t row, int w)
{
    const int64_t c = (int64_t)row * a.g.ncr + (w >> 5);
    return a.chunkbase[c] + __popc(a.ballots[c] & ((1u << (w & 31)) - 1u));
}

__device__ __forceinline__ uint32_t lt_mask(int b) { return b >= 32 ? 0xffffffffu : ((1u << b) - 1u); }

__device__ __forceinline__ unsigned long long vkey(int axis, int z, int y, int x)
{
    return (unsigned long long)axis | ((unsigned long long)x << 2) | ((unsigned long long)y << 22) | ((unsigned long long)z << 42);
}

// PARTS: 1 = vertex keys only, 2 = faces only, 3 = both (the keys are all the vertex kernel needs, so the faces can be
// emitted concurrently with it on another stream)
// AMB = 0: faces of the words WITHOUT an ambiguous cube only (the common kernel: no call, no stack frame); AMB = 1: faces of the
// flagged words only; AMB = 2: all words in one kernel (staged path).  Vertex keys (PARTS & 1) are written for every word.
template <int PARTS, int AMB>
__global__ void __launch_bounds__(128) k_mc_emit(EmitArgs a)
{
    // per-thread tables indexed by cube edge (0..11), thread-major => bank-conflict free; the corner -> vertex id
    // computation below is a table look-up instead of a 12-way switch (which diverged to ~4 active lanes)
    __shared__ __align__(16) int8_t s_tri[256][T3D_MC_ROW];
    __shared__ uint32_t s_base[12][128];
    __shared__ uint32_t s_mask[12][128];
    __shared__ uint32_t s_next[4][128];   // ids of the y/z-edge vertices at bit 0 of the next word (edges 1, 5, 9, 10 at b = 31)
    if (AMB == 1) {                       // nearly every CTA of this launch finds no flagged word in its share of the list:
        int any = 0;                      // leave before the table copy (the second look at the list comes from L2)
        uint32_t nw_ = a.cap_active;
        if (a.sizes[0] < nw_) nw_ = (uint32_t)a.sizes[0];
        for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nw_; k += gridDim.x * blockDim.x) any |= (int)(a.aw_idx[k] >> 31);
        if (!__syncthreads_or(any)) return;
    }
    if (PARTS & 2) {
        const int4* src = reinterpret_cast<const int4*>(&g_tri_table[0][0]);
        int4* dst = reinterpret_cast<int4*>(&s_tri[0][0]);
        for (int i = threadIdx.x; i < 256; i += blockDim.x) {
            dst[i] = src[i];
            if (c_luts.ntri[i] & MC_AMB) s_tri[i][T3D_MC_ROW - 1] = -2;   // (classic rows end at or before entry 15)
        }
        __syncthreads();
    }
    const uint32_t tid = threadIdx.x;
    uint32_t n_words = a.cap_active;
    if (a.sizes[0] < n_words) n_words = (uint32_t)a.sizes[0];
    const uint32_t offY = (uint32_t)a.sizes[1], offZ = (uint32_t)(a.sizes[1] + a.sizes[2]);  // offX = 0
    if (a.sizes[1] + a.sizes[2] + a.sizes[3] > a.cap_verts || a.sizes[4] > a.cap_faces) return;  // overflow: flagged by the caller
    // one active word (the tables above are per thread: a thread may take several words in turn)
    auto emit_word = [&](const uint32_t k, const uint32_t iraw) {
    const uint32_t i = iraw & AW_MASK;
    const uint32_t row = i / (uint32_t)a.g.nws;
    const int w = (int)(i - row * (uint32_t)a.g.nws);
    int z, y;
    const WordMasks m = load_masks(a.g, row, w, z, y);
    const int64_t NA = a.cap_active;
    const uint32_t bX00 = a.aw_base[k], bY0 = offY + a.aw_base[NA + k], bZ0 = offZ + a.aw_base[2 * NA + k];
    uint32_t pT = a.aw_base[3 * NA + k];
    const int x0 = w << 5;

    // ---- keys of the vertices this word owns
    if (PARTS & 1) {
        uint32_t id = bX00;
        for (uint32_t q = m.X00; q;) { const int b = __ffs(q) - 1; q &= q - 1; a.vkeys[id++] = vkey(2, z, y, x0 + b); }
        id = bY0;
        for (uint32_t q = m.Y0; q;) { const int b = __ffs(q) - 1; q &= q - 1; a.vkeys[id++] = vkey(1, z, y, x0 + b); }
        id = bZ0;
        for (uint32_t q = m.Z0; q;) { const int b = __ffs(q) - 1; q &= q - 1; a.vkeys[id++] = vkey(0, z, y, x0 + b); }
    }
    if (!(PARTS & 2) || !m.act) return;
    if (AMB == 0 && (iraw & AW_AMB)) return;       // its faces come from the AMB = 1 launch

    // ---- bases of the neighbouring words whose vertices our cubes use (looked up only when they own any)
    const uint32_t Hs = (uint32_t)a.g.Hs;
    uint32_t bX01 = 0, bX10 = 0, bX11 = 0, bY1 = 0, bZ1 = 0;
    if (m.X01 | m.Z1) {
        const uint32_t r = active_rank(a, row + 1, w);
        bX01 = a.aw_base[r];
        bZ1 = offZ + a.aw_base[2 * NA + r];
    }
    if (m.X10 | m.Y1) {
        const uint32_t r = active_rank(a, row + Hs, w);
        bX10 = a.aw_base[r];
        bY1 = offY + a.aw_base[NA + r];
    }
    if (m.X11) bX11 = a.aw_base[active_rank(a, row + Hs + 1, w)];
    // y/z edges at x0+32 (bit 0 of the next word) are only used by the cube at bit 31
    uint32_t nY0 = 0, nY1 = 0, nZ0 = 0, nZ1 = 0;
    if ((m.act >> 31) & 1u) {
        const uint32_t v1 = (m.a00 >> 31) & 1u, v2 = (m.a01 >> 31) & 1u, v5 = (m.a10 >> 31) & 1u, v6 = (m.a11 >> 31) & 1u;
        if (v1 != v2) nY0 = offY + a.aw_base[NA + active_rank(a, row, w + 1)];            // edge 1
        if (v5 != v6) nY1 = offY + a.aw_base[NA + active_rank(a, row + Hs, w + 1)];       // edge 5
        if (v1 != v5) nZ0 = offZ + a.aw_base[2 * NA + active_rank(a, row, w + 1)];        // edge 9
        if (v2 != v6) nZ1 = offZ + a.aw_base[2 * NA + active_rank(a, row + 1, w + 1)];    // edge 10
    }
    // edge -> (base id of the owning word's block, cut mask of that block)
    s_base[0][tid] = bX00; s_mask[0][tid] = m.X00;
    s_base[1][tid] = bY0;  s_mask[1][tid] = m.Y0;
    s_base[2][tid] = bX01; s_mask[2][tid] = m.X01;
    s_base[3][tid] = bY0;  s_mask[3][tid] = m.Y0;
    s_base[4][tid] = bX10; s_mask[4][tid] = m.X10;
    s_base[5][tid] = bY1;  s_mask[5][tid] = m.Y1;
    s_base[6][tid] = bX11; s_mask[6][tid] = m.X11;
    s_base[7][tid] = bY1;  s_mask[7][tid] = m.Y1;
    s_base[8][tid] = bZ0;  s_mask[8][tid] = m.Z0;
    s_base[9][tid] = bZ0;  s_mask[9][tid] = m.Z0;
    s_base[10][tid] = bZ1; s_mask[10][tid] = m.Z1;
    s_base[11][tid] = bZ1; s_mask[11][tid] = m.Z1;
    s_next[0][tid] = nY0; s_next[1][tid] = nY1; s_next[2][tid] = nZ0; s_next[3][tid] = nZ1;
    // (each thread reads back only its own column: no barrier needed)

    // corner -> vertex id of the cube at bit b, through the per-thread tables above
    auto vertex_id = [&](int b, int e) -> uint32_t {
        const uint32_t at_next = (0x622u >> e) & 1u;           // edges 1, 5, 9, 10 sit at x + 1
        uint32_t id = s_base[e][tid] + __popc(s_mask[e][tid] & (at_next ? lt_mask(b + 1) : lt_mask(b)));
        if (b == 31 && at_next) id = s_next[((e >> 2) & 1) + 2 * ((e >> 3) & 1) + ((e >> 3) & 1) * ((e >> 1) & 1)][tid];
        return id;
    };
    auto emit_classic = [&](int b, int cs) {
        const int4 trow = *reinterpret_cast<const int4*>(s_tri[cs]);   // 16 edge ids, -1 terminated
        const uint32_t tw[4] = {(uint32_t)trow.x, (uint32_t)trow.y, (uint32_t)trow.z, (uint32_t)trow.w};
        auto edge_at = [&](int t) -> int { return (int)(int8_t)((tw[t >> 2] >> ((t & 3) * 8)) & 0xffu); };
        for (int t = 0; t < 15; t += 3) {
            const int e0 = edge_at(t);
            if (e0 < 0) break;
            uint32_t vid[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) vid[c] = vertex_id(b, (c == 0) ? e0 : edge_at(t + c));
            int32_t* f = a.faces + 3 * (int64_t)pT;
            f[0] = (int32_t)vid[2]; f[1] = (int32_t)vid[1]; f[2] = (int32_t)vid[0];
            ++pT;
        }
    };
    if constexpr (AMB == 0) {             // the common kernel: classic rows only
        for (uint32_t q = m.act; q;) {
            const int b = __ffs(q) - 1;
            q &= q - 1;
            emit_classic(b, cube_case(m, b));
        }
    } else {
    for (uint32_t q = m.act; q;) {        // words that may hold ambiguous cubes
        const int b = __ffs(q) - 1;
        q &= q - 1;
        const int cs = cube_case(m, b);
        if ((uint8_t)s_tri[cs][T3D_MC_ROW - 1] != 0xfeu) { emit_classic(b, cs); continue; }     // byte 15 = -2: ambiguous index
        // the row Lewiner's tests select (same decision as in k_mc_words<1>)
        const int r = mc33_resolve(a.fld, z, y, x0 + b, cs);
        const int8_t* row = g33_rows[r];
        const int n3 = 3 * (int)g33_ntri[r];
        for (int t = 0; t < n3; t += 3) {
            int32_t* f = a.faces + 3 * (int64_t)pT;
            f[0] = (int32_t)vertex_id(b, row[t + 2]); f[1] = (int32_t)vertex_id(b, row[t + 1]); f[2] = (int32_t)vertex_id(b, row[t]);
            ++pT;
        }
    }
    }
    };
    if (AMB == 1) {
        // a fixed, small grid striding over the word list for the flagged words (nearly every entry is skipped)
        for (uint32_t k = blockIdx.x * blockDim.x + tid; k < n_words; k += gridDim.x * blockDim.x) {
            const uint32_t iraw = a.aw_idx[k];
            if (iraw & AW_AMB) emit_word(k, iraw);
        }
    } else {
        const uint32_t k = blockIdx.x * blockDim.x + tid;
        if (k < n_words) emit_word(k, a.aw_idx[k]);
    }
}

// ------------------------------------------------------------------------------------------------
// 6. vertices: one thread per vertex
// ------------------------------------------------------------------------------------------------
struct VertexArgs {
    OccView occ;
    const float* field;       // optional dense float32 field (Z,H,W): marched directly at `level` (SDF path)
    double level;             // iso level (0.5 for the Gaussian occupancy field)
    const unsigned long long* vkeys;
    int x_off;                // the keys' x minus this = x in the (reference-)padded grid (padded-storage layout: 127)
    int z_offset;             // global padded plane of local padded plane 0 (z-slab sharding; 0 on a single device)
    float shift;              // 1 if manifold else 0 (surface_extractor.py:57-60)
    const double* cum;        // cumulative adjusted depths, n_cum entries (n_cum = 0: no z map)
    const double* adj;        // adjusted depths, n_cum-1 entries
    int n_cum;
    double mm_y, mm_x;
    int scale_f64;            // numpy float64 scalar operand: multiply in float64, then round
    float* verts;             // (V, 3) z, y, x
};

template <int AXIS>
__device__ __forceinline__ void vertex_body(const VertexArgs& p, const ZLut& zlut, uint32_t id)
{
    const unsigned long long key = p.vkeys[id];
    const int x = (int)((key >> 2) & 0xfffffu) - p.x_off, y = (int)((key >> 22) & 0xfffffu), z = (int)(key >> 42);
    float fa, fb;
    if (p.field) {
        const int64_t i = ((int64_t)z * p.occ.H + y) * p.occ.W + x;
        fa = p.field[i];
        fb = p.field[i + (AXIS == 0 ? (int64_t)p.occ.H * p.occ.W : AXIS == 1 ? p.occ.W : 1)];
    } else {
        edge_field_values<AXIS>(p.occ, zlut, z, y, x, fa, fb);
    }
    // skimage: strength = 1/(eps + |v - level|), eps = np.spacing(1.0), centre of mass of the two corners, all in double
    const double va = (double)fa - p.level, vb = (double)fb - p.level;
    const double wa = __ddiv_rn(1.0, __dadd_rn(MC33_EPS, fabs(va)));
    const double wb = __ddiv_rn(1.0, __dadd_rn(MC33_EPS, fabs(vb)));
    const double frac = __ddiv_rn(wb, __dadd_rn(wa, wb));
    double pz = (double)(z + p.z_offset), py = (double)y, px = (double)x;
    if (AXIS == 0) pz = __dadd_rn(pz, frac); else if (AXIS == 1) py = __dadd_rn(py, frac); else px = __dadd_rn(px, frac);
    float fz = __fsub_rn(__double2float_rn(pz), p.shift);
    float fy = __fsub_rn(__double2float_rn(py), p.shift);
    float fx = __fsub_rn(__double2float_rn(px), p.shift);
    if (p.n_cum > 0) {
        // surface_extractor.py:98-113, closed form verified bit-exact in SURVEY.md V8
        if (fz < 0.0f) fz = 0.0f;
        else if (fz >= (float)(p.n_cum - 1)) fz = __double2float_rn(p.cum[p.n_cum - 1]);
        else {
            const float fl = floorf(fz);
            const int lo = (int)fl;
            const float fr = __fsub_rn(fz, fl);
            const int ai = min(lo, p.n_cum - 2);
            fz = __double2float_rn(__dadd_rn(p.cum[lo], __dmul_rn((double)fr, p.adj[ai])));
        }
    }
    if (p.scale_f64) {
        fy = __double2float_rn(__dmul_rn((double)fy, p.mm_y));
        fx = __double2float_rn(__dmul_rn((double)fx, p.mm_x));
    } else {
        fy = __fmul_rn(fy, __double2float_rn(p.mm_y));
        fx = __fmul_rn(fx, __double2float_rn(p.mm_x));
    }
    float* o = p.verts + 3 * (int64_t)id;
    o[0] = fz; o[1] = fy; o[2] = fx;
}

// axis blocks selected by `which` (1: x-edge, 2: y-edge, 4: z-edge vertices) in one launch, block sizes read from device
// memory (sizes = {n_active, n_x, n_y, n_z, n_t}).  Thread t handles the t-th vertex of the selected blocks.
__global__ void __launch_bounds__(128) k_mc_vertices_all(VertexArgs p, const unsigned long long* __restrict__ sizes, uint32_t cap_verts,
                                                         int which)
{
    __shared__ ZLut zlut;
    fill_zlut(p.occ, zlut);
    __syncthreads();
    const unsigned long long nx = sizes[1], ny = sizes[2], nz = sizes[3];
    if (nx + ny + nz > cap_verts) return;
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (which & 1) {
        if (t < nx) { vertex_body<2>(p, zlut, t); return; }
        t -= (uint32_t)nx;
    }
    if (which & 2) {
        if (t < ny) { vertex_body<1>(p, zlut, (uint32_t)nx + t); return; }
        t -= (uint32_t)ny;
    }
    if ((which & 4) && t < nz) vertex_body<0>(p, zlut, (uint32_t)(nx + ny) + t);
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
static int make_grid(Grid& g, const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end, const char* who)
{
    if (Zs <= 0 || Hs <= 0 || Ws <= 0) { t3d_set_error("%s: empty volume", who); return 2; }
    if (z_end < 0 || z_end > Zs) z_end = Zs;
    if (z_begin < 0 || z_begin >= z_end) { t3d_set_error("%s: empty plane range", who); return 2; }
    g.z_begin = z_begin; g.z_end = z_end;
    g.sign = (const uint32_t*)sign_bits;
    g.Zs = Zs; g.Hs = Hs; g.Ws = Ws; g.nws = t3d_wpr(Ws);
    g.ncr = (g.nws + 31) >> 5;
    g.n_rows = (uint32_t)((int64_t)Zs * Hs);
    g.n_words = (int64_t)Zs * Hs * g.nws;
    if (g.n_words >= ((int64_t)1 << 31)) { t3d_set_error("%s: more than 2^31 words in one device slab", who); return 2; }
    return 0;
}

extern "C" int64_t t3d_mc_num_chunks(int Zs, int Hs, int Ws) { return (int64_t)Zs * Hs * ((t3d_wpr(Ws) + 31) >> 5); }

// ballots_u32: t3d_mc_num_chunks words, one per (voxel row, 32-word chunk): bit l = word 32*chunk+l of that row is active
extern "C" int t3d_mc_flags(const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end, void* ballots_u32,
                            void* stream)
{
    Grid g;
    if (int rc = make_grid(g, sign_bits, Zs, Hs, Ws, z_begin, z_end, "t3d_mc_flags")) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (t3d_zero_async(ballots_u32, sizeof(uint32_t) * (size_t)g.n_rows * g.ncr, st)) return 1;
    const int nws4 = g.nws / 4, lanes_x = nws4 < 256 ? nws4 : 256, pzb = 256 / lanes_x;
    const int nz = (g.z_end < Zs ? g.z_end + 1 : Zs) - g.z_begin;
    dim3 grid((nws4 + lanes_x - 1) / lanes_x, (Hs + GY - 1) / GY, (nz + pzb - 1) / pzb);
    k_mc_flags<<<grid, 256, 0, st>>>(g, (uint32_t*)ballots_u32, lanes_x, pzb, GY);
    T3D_CHECK_LAUNCH("t3d_mc_flags");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Every data-dependent size stays in device memory (sizes_u64 = {n_active, n_x, n_y, n_z, n_t}), arrays are capacity-sized
// and nothing is written beyond the capacities.  No host round trip => graph-capturable.
// ------------------------------------------------------------------------------------------------
static int mc_words_dev_impl(const McField& fld, const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end,
                             const void* ballots_u32, const void* chunkbase_u32, uint32_t cap_active, const void* sizes_u64,
                             void* aw_idx_u32, void* aw_cnt_u32, void* n_ambiguous_u64, void* stream)
{
    Grid g;
    if (int rc = make_grid(g, sign_bits, Zs, Hs, Ws, z_begin, z_end, "t3d_mc_words_dev")) return rc;
    if (ensure_luts()) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    if (t3d_zero_async(n_ambiguous_u64, 8, st)) return 1;
    if (cap_active == 0) return 0;
    const int64_t n_chunks = (int64_t)g.n_rows * g.ncr;
    k_mc_compact<<<(unsigned)((n_chunks + 255) / 256), 256, 0, st>>>(g, (const uint32_t*)ballots_u32, (const uint32_t*)chunkbase_u32,
                                                                      n_chunks, (uint32_t*)aw_idx_u32, cap_active);
    k_mc_words<0><<<(cap_active + 127) / 128, 128, 0, st>>>(g, fld, (uint32_t*)aw_idx_u32, cap_active, (const unsigned long long*)sizes_u64,
                                                            (uint32_t*)aw_cnt_u32, (unsigned long long*)n_ambiguous_u64);
    k_mc_words<1><<<amb_grid(cap_active), 128, 0, st>>>(g, fld, (uint32_t*)aw_idx_u32, cap_active, (const unsigned long long*)sizes_u64,
                                                            (uint32_t*)aw_cnt_u32, (unsigned long long*)n_ambiguous_u64);
    T3D_CHECK_LAUNCH("t3d_mc_words_dev");
    t3d_count_launches(3);
    return 0;
}

extern "C" int t3d_mc_words_dev(const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end, const void* ballots_u32,
                                const void* chunkbase_u32, uint32_t cap_active, const void* sizes_u64, void* aw_idx_u32,
                                void* aw_cnt_u32, void* n_ambiguous_u64, const t3d_mc_field* mc_field, void* stream)
{
    return mc_words_dev_impl(mc_field_from_abi(mc_field), sign_bits, Zs, Hs, Ws, z_begin, z_end, ballots_u32, chunkbase_u32, cap_active,
                             sizes_u64, aw_idx_u32, aw_cnt_u32, n_ambiguous_u64, stream);
}

static int mc_emit_dev_impl(const McField& fld, const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end,
                            const void* ballots_u32, const void* chunkbase_u32, const void* aw_idx_u32, const void* aw_base_u32,
                            uint32_t cap_active, const void* sizes_u64, uint32_t cap_verts, uint32_t cap_faces, void* vkeys_u64,
                            void* faces_i32, int parts, void* stream)
{
    EmitArgs a;
    if (int rc = make_grid(a.g, sign_bits, Zs, Hs, Ws, z_begin, z_end, "t3d_mc_emit_dev")) return rc;
    if (ensure_luts()) return 1;
    if (cap_active == 0) return 0;
    a.fld = fld;
    a.ballots = (const uint32_t*)ballots_u32;
    a.chunkbase = (const uint32_t*)chunkbase_u32;
    a.aw_idx = (const uint32_t*)aw_idx_u32;
    a.aw_base = (const uint32_t*)aw_base_u32;
    a.cap_active = cap_active;
    a.sizes = (const unsigned long long*)sizes_u64;
    a.cap_verts = cap_verts;
    a.cap_faces = cap_faces;
    a.vkeys = (unsigned long long*)vkeys_u64;
    a.faces = (int32_t*)faces_i32;
    const unsigned ge = (cap_active + 127) / 128;
    int launches = 1;
    if ((parts & 3) == 1) k_mc_emit<1, 0><<<ge, 128, 0, (cudaStream_t)stream>>>(a);
    else if ((parts & 3) == 2) {        // the common words, then the (rare) words holding ambiguous cubes
        k_mc_emit<2, 0><<<ge, 128, 0, (cudaStream_t)stream>>>(a);
        k_mc_emit<2, 1><<<amb_grid(cap_active), 128, 0, (cudaStream_t)stream>>>(a);
        launches = 2;
    } else k_mc_emit<3, 2><<<ge, 128, 0, (cudaStream_t)stream>>>(a);
    T3D_CHECK_LAUNCH("t3d_mc_emit_dev");
    t3d_count_launches(launches);
    return 0;
}

extern "C" int t3d_mc_emit_dev(const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end, const void* ballots_u32,
                               const void* chunkbase_u32, const void* aw_idx_u32, const void* aw_base_u32, uint32_t cap_active,
                               const void* sizes_u64, uint32_t cap_verts, uint32_t cap_faces, void* vkeys_u64, void* faces_i32,
                               int parts, const t3d_mc_field* mc_field, void* stream)
{
    return mc_emit_dev_impl(mc_field_from_abi(mc_field), sign_bits, Zs, Hs, Ws, z_begin, z_end, ballots_u32, chunkbase_u32, aw_idx_u32,
                            aw_base_u32, cap_active, sizes_u64, cap_verts, cap_faces, vkeys_u64, faces_i32, parts, stream);
}

// the same on a strided occupancy view (padded-storage layout of the fused pipeline, t3d_pipeline.cu)
int t3d_mc_words_view_dev(const OccView& view, int x_off, const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end,
                          const void* ballots_u32, const void* chunkbase_u32, uint32_t cap_active, const void* sizes_u64,
                          void* aw_idx_u32, void* aw_cnt_u32, void* n_ambiguous_u64, void* stream)
{
    McField f;
    f.occ = view; f.field = nullptr; f.level = 0.5; f.x_off = x_off; f.mode = 1;
    return mc_words_dev_impl(f, sign_bits, Zs, Hs, Ws, z_begin, z_end, ballots_u32, chunkbase_u32, cap_active, sizes_u64, aw_idx_u32,
                             aw_cnt_u32, n_ambiguous_u64, stream);
}

int t3d_mc_emit_view_dev(const OccView& view, int x_off, const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end,
                         const void* ballots_u32, const void* chunkbase_u32, const void* aw_idx_u32, const void* aw_base_u32,
                         uint32_t cap_active, const void* sizes_u64, uint32_t cap_verts, uint32_t cap_faces, void* vkeys_u64,
                         void* faces_i32, int parts, void* stream)
{
    McField f;
    f.occ = view; f.field = nullptr; f.level = 0.5; f.x_off = x_off; f.mode = 1;
    return mc_emit_dev_impl(f, sign_bits, Zs, Hs, Ws, z_begin, z_end, ballots_u32, chunkbase_u32, aw_idx_u32, aw_base_u32, cap_active,
                            sizes_u64, cap_verts, cap_faces, vkeys_u64, faces_i32, parts, stream);
}

// vertices of a mesh emitted on a sign volume whose x coordinates are shifted by x_off against `view`'s padded grid; with
// `field`, the dense float32 field of the view's extents is interpolated at `level` instead
static int mc_vertices_impl(const OccView& view, const float* field, double level, int x_off, const void* vkeys_u64, const void* sizes_u64,
                            uint32_t cap_verts, int unpad_shift, int z_offset, const void* cum_f64, const void* adj_f64, int n_cum,
                            double mm_per_pixel_y, double mm_per_pixel_x, int scale_in_f64, int which_blocks, void* verts_f32, void* stream)
{
    if ((which_blocks & 7) == 0) return 0;
    if (cap_verts == 0) return 0;
    VertexArgs p;
    p.occ = view;
    p.vkeys = (const unsigned long long*)vkeys_u64;
    p.field = field;
    p.level = level;
    p.x_off = x_off;
    p.shift = unpad_shift ? 1.0f : 0.0f;
    p.z_offset = z_offset;
    p.cum = (const double*)cum_f64;
    p.adj = (const double*)adj_f64;
    p.n_cum = n_cum;
    p.mm_y = mm_per_pixel_y;
    p.mm_x = mm_per_pixel_x;
    p.scale_f64 = scale_in_f64 ? 1 : 0;
    p.verts = (float*)verts_f32;
    k_mc_vertices_all<<<(cap_verts + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p, (const unsigned long long*)sizes_u64, cap_verts,
                                                                               which_blocks & 7);
    T3D_CHECK_LAUNCH("t3d_mc_vertices_dev");
    t3d_count_launches(1);
    return 0;
}

int t3d_mc_vertices_view_dev(const OccView& view, int x_off, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts,
                             int unpad_shift, int z_offset, const void* cum_f64, const void* adj_f64, int n_cum, double mm_per_pixel_y,
                             double mm_per_pixel_x, int scale_in_f64, int which_blocks, void* verts_f32, void* stream)
{
    return mc_vertices_impl(view, nullptr, 0.5, x_off, vkeys_u64, sizes_u64, cap_verts, unpad_shift, z_offset, cum_f64, adj_f64, n_cum,
                            mm_per_pixel_y, mm_per_pixel_x, scale_in_f64, which_blocks, verts_f32, stream);
}

// occ_*: the occupancy the sign volume was derived from (pad / gaussian as in t3d_field_sign; gaussian = 0: the sign volume IS
// the occupancy and pad must be 0), or field_f32: the dense field the sign volume was taken from (t3d_sign_from_f32).
extern "C" int t3d_mc_vertices_dev(const void* occ_bits, int Z, int H, int W, int pad, int gaussian, const double* weights3_host,
                                   const void* field_f32, double level, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts,
                                   int unpad_shift, int z_offset, const void* cum_f64, const void* adj_f64, int n_cum,
                                   double mm_per_pixel_y, double mm_per_pixel_x, int scale_in_f64, int which_blocks, void* verts_f32,
                                   void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_mc_vertices_dev: empty volume"); return 2; }
    if (!field_f32 && !gaussian && pad) { t3d_set_error("t3d_mc_vertices_dev: pad requires gaussian"); return 2; }
    const OccView view = field_f32 ? t3d_make_view(nullptr, Z, H, W, 0, 0, nullptr)
                                   : t3d_make_view(occ_bits, Z, H, W, pad, gaussian, weights3_host);
    return mc_vertices_impl(view, (const float*)field_f32, field_f32 ? level : 0.5, 0, vkeys_u64, sizes_u64, cap_verts, unpad_shift,
                            z_offset, cum_f64, adj_f64, n_cum, mm_per_pixel_y, mm_per_pixel_x, scale_in_f64, which_blocks, verts_f32,
                            stream);
}

// ------------------------------------------------------------------------------------------------
// marching a dense float32 field (additive SDF path, SURVEY.md 8a-16 / 8b): sign bits straight from it (the vertices come from
// t3d_mc_vertices_dev with field_f32)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_sign_from_f32(const float* __restrict__ field, int64_t n_rows, int W, int nw, double level,
                                                       uint32_t* __restrict__ bits)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * nw) return;
    const int64_t row = i / nw;
    const int w = (int)(i - row * nw);
    const float* p = field + row * W + (w << 5);
    const int n = min(32, W - (w << 5));
    uint32_t v = 0;
    for (int k = 0; k < n; ++k) v |= (uint32_t)(((double)p[k] - level) > 0.0) << k;
    bits[i] = v;
}

// bit = (field > level), packed like an occupancy volume (Z,H,wpr(W))
extern "C" int t3d_sign_from_f32(const void* field_f32, int Z, int H, int W, double level, void* sign_bits, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_sign_from_f32: empty volume"); return 2; }
    const int nw = t3d_wpr(W);
    const int64_t rows = (int64_t)Z * H, n = rows * nw;
    k_sign_from_f32<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const float*)field_f32, rows, W, nw, level,
                                                                                 (uint32_t*)sign_bits);
    T3D_CHECK_LAUNCH("t3d_sign_from_f32");
    t3d_count_launches(1);
    return 0;
}
