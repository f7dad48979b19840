// t3d_export.cu -- device-side mesh consumers (SURVEY.md 8f-3): the step right after the hot path.
//
//   * layer colours  (glb_exporter.py:52-91): per-vertex z-window tests -> RGBA
//   * OBJ text       (obj_exporter.py:17-41): "v %.6f %.6f %.6f\n" per vertex, "f a b c\n" (1-based) per face.
//     The reference formats in a Python loop (hours at 1e8 faces); here every line is formatted by one thread.
//     "%.6f" of a float32 is exact on the device: |x| * 1e6 is the product of a 24-bit and a 20-bit integer mantissa,
//     exactly representable in float64, so rint() (ties to even) gives printf's correctly rounded digits.
#include <math.h>

#include "t3d.h"
#include "t3d_common.cuh"

// ------------------------------------------------------------------------------------------------
// layer colours
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_layer_colors(const float* __restrict__ verts, int64_t V, double a0, double a1, int has_a,
                                                      double b0, double b1, int has_b, uchar4* __restrict__ rgba)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const double z = (double)verts[3 * i];   // numpy compares the float32 column with float64 scalars in float64
    uchar4 c = make_uchar4(200, 200, 200, 255);
    if (has_a && z >= a0 && z <= a1) c = make_uchar4(255, 0, 0, 255);
    if (has_b && z >= b0 && z <= b1) c = make_uchar4(0, 0, 255, 255);
    rgba[i] = c;
}

extern "C" int t3d_layer_colors(const void* verts_f32, int64_t V, int has_first, double first_start, double first_end, int has_last,
                                double last_start, double last_end, void* rgba_u8, void* stream)
{
    if (V <= 0) return 0;
    k_layer_colors<<<(unsigned)((V + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const float*)verts_f32, V, first_start, first_end,
                                                                                 has_first, last_start, last_end, has_last,
                                                                                 (uchar4*)rgba_u8);
    T3D_CHECK_LAUNCH("t3d_layer_colors");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// OBJ text
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int dec_digits(unsigned long long v)
{
    int n = 1;
    while (v >= 10ull) { v /= 10ull; ++n; }
    return n;
}

// "%.6f": [-]int.ffffff ; "nan" / "inf" / "-inf" as Python prints them
struct Fixed6 {
    unsigned long long ip;  // integer part
    uint32_t fp;            // six fractional digits
    int kind;               // 0 number, 1 nan, 2 inf
    bool neg;
};

__device__ __forceinline__ Fixed6 to_fixed6(float x)
{
    Fixed6 f;
    f.neg = signbit(x);
    f.kind = isnan(x) ? 1 : (isinf(x) ? 2 : 0);
    f.ip = 0; f.fp = 0;
    if (f.kind == 0) {
        const double m = rint(fabs((double)x) * 1000000.0);   // exact product, ties to even
        if (m < 1.8e19) {
            const unsigned long long q = (unsigned long long)m;
            f.ip = q / 1000000ull;
            f.fp = (uint32_t)(q % 1000000ull);
        } else {
            f.kind = 3;   // beyond 64-bit fixed point (|x| > 1.8e13): not a coordinate; written as "inf"
        }
    }
    if (f.kind == 1) f.neg = false;   // Python: "nan" without sign
    return f;
}

__device__ __forceinline__ int fixed6_len(const Fixed6& f)
{
    if (f.kind == 1) return 3;
    if (f.kind >= 2) return 3 + (f.neg ? 1 : 0);
    return (f.neg ? 1 : 0) + dec_digits(f.ip) + 7;
}

__device__ __forceinline__ char* put_uint(char* p, unsigned long long v)
{
    const int n = dec_digits(v);
    for (int k = n - 1; k >= 0; --k) { p[k] = (char)('0' + (int)(v % 10ull)); v /= 10ull; }
    return p + n;
}

__device__ __forceinline__ char* put_fixed6(char* p, const Fixed6& f)
{
    if (f.kind == 1) { p[0] = 'n'; p[1] = 'a'; p[2] = 'n'; return p + 3; }
    if (f.neg) *p++ = '-';
    if (f.kind >= 2) { p[0] = 'i'; p[1] = 'n'; p[2] = 'f'; return p + 3; }
    p = put_uint(p, f.ip);
    *p++ = '.';
    uint32_t v = f.fp;
    for (int k = 5; k >= 0; --k) { p[k] = (char)('0' + (int)(v % 10u)); v /= 10u; }
    return p + 6;
}

template <typename IdxT>
__global__ void __launch_bounds__(256) k_obj_lengths(const float* __restrict__ verts, int64_t V, const IdxT* __restrict__ faces, int64_t F,
                                                     uint32_t* __restrict__ len)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V) {
        const float* v = verts + 3 * i;
        len[i] = 2 + fixed6_len(to_fixed6(v[0])) + 1 + fixed6_len(to_fixed6(v[1])) + 1 + fixed6_len(to_fixed6(v[2])) + 1;   // "v a b c\n"
    } else if (i < V + F) {
        const IdxT* f = faces + 3 * (i - V);
        int n = 2 + 2 + 1;   // "f " + two spaces + newline
        for (int k = 0; k < 3; ++k) {
            const long long a = (long long)f[k] + 1;
            n += (a < 0 ? 1 : 0) + dec_digits((unsigned long long)(a < 0 ? -a : a));
        }
        len[i] = (uint32_t)n;
    }
}

// layout of the text: [vertex lines][one '\n'][face lines]; `offs` = exclusive scan of the line lengths
template <typename IdxT>
__global__ void __launch_bounds__(256) k_obj_emit(const float* __restrict__ verts, int64_t V, const IdxT* __restrict__ faces, int64_t F,
                                                  const unsigned long long* __restrict__ offs, char* __restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V) {
        char* p = out + offs[i];
        const float* v = verts + 3 * i;
        *p++ = 'v';
        for (int k = 0; k < 3; ++k) { *p++ = ' '; p = put_fixed6(p, to_fixed6(v[k])); }
        *p = '\n';
    } else if (i < V + F) {
        char* p = out + offs[i] + 1;   // after the blank line between the two blocks
        const IdxT* f = faces + 3 * (i - V);
        *p++ = 'f';
        for (int k = 0; k < 3; ++k) {
            *p++ = ' ';
            long long a = (long long)f[k] + 1;
            if (a < 0) { *p++ = '-'; a = -a; }
            p = put_uint(p, (unsigned long long)a);
        }
        *p = '\n';
    }
}

__global__ void k_obj_blank(const unsigned long long* __restrict__ offs, int64_t V, int64_t F, const unsigned long long* __restrict__ total,
                            char* __restrict__ out)
{
    // the blank line sits right after the last vertex line = at the start offset of face line 0 (or at the end)
    const unsigned long long at = F > 0 ? offs[V] : *total;
    out[at] = '\n';
}

extern "C" int64_t t3d_obj_workspace_bytes(int64_t V, int64_t F)
{
    const int64_t n = V + F;
    return ((4 * n + 255) & ~(int64_t)255) + ((8 * n + 255) & ~(int64_t)255) + t3d_scan_workspace_bytes(n, 1) + 256;
}

// Phase 1: line lengths and their exclusive scan (kept in `workspace`); total_len_u64 (device) = bytes of the vertex
// and face lines (the body is total + 1 bytes: one blank line between the blocks).
extern "C" int t3d_obj_measure(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64, void* total_len_u64,
                               void* workspace, void* stream)
{
    if (V < 0 || F < 0 || V + F > 0x7fffffff) { t3d_set_error("t3d_obj_measure: bad sizes"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = V + F;
    if (n == 0) { T3D_CUDA(cudaMemsetAsync(total_len_u64, 0, 8, st)); return 0; }
    char* ws = (char*)workspace;
    uint32_t* len = (uint32_t*)ws; ws += (4 * n + 255) & ~(int64_t)255;
    unsigned long long* offs = (unsigned long long*)ws; ws += (8 * n + 255) & ~(int64_t)255;
    const unsigned g = (unsigned)((n + 255) / 256);
    if (faces_are_i64) k_obj_lengths<long long><<<g, 256, 0, st>>>((const float*)verts_f32, V, (const long long*)faces, F, len);
    else k_obj_lengths<int32_t><<<g, 256, 0, st>>>((const float*)verts_f32, V, (const int32_t*)faces, F, len);
    T3D_CHECK_LAUNCH("t3d_obj_measure");
    t3d_count_launches(1);
    return t3d_exclusive_scan_u32_dev(len, offs, n, n, 1, 1, 0, nullptr, total_len_u64, ws, stream);
}

// Phase 2: the body of the OBJ file (everything after the two comment lines and the blank line that follow them):
// vertex lines, one blank line, face lines -- total + 1 bytes into out_bytes.
extern "C" int t3d_obj_emit(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64, const void* total_len_u64,
                            const void* workspace, void* out_bytes, void* stream)
{
    if (V < 0 || F < 0 || V + F > 0x7fffffff) { t3d_set_error("t3d_obj_emit: bad sizes"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = V + F;
    const char* ws = (const char*)workspace;
    ws += (4 * n + 255) & ~(int64_t)255;
    const unsigned long long* offs = (const unsigned long long*)ws;
    if (n > 0) {
        const unsigned g = (unsigned)((n + 255) / 256);
        if (faces_are_i64) k_obj_emit<long long><<<g, 256, 0, st>>>((const float*)verts_f32, V, (const long long*)faces, F, offs, (char*)out_bytes);
        else k_obj_emit<int32_t><<<g, 256, 0, st>>>((const float*)verts_f32, V, (const int32_t*)faces, F, offs, (char*)out_bytes);
    }
    k_obj_blank<<<1, 1, 0, st>>>(offs, V, F, (const unsigned long long*)total_len_u64, (char*)out_bytes);
    T3D_CHECK_LAUNCH("t3d_obj_emit");
    t3d_count_launches(2);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// GLB (binary glTF 2.0) payload: what trimesh's exporter writes for Trimesh(vertices, faces, vertex_colors) after
// fix_normals() (glb_exporter.py:36-43) -- one buffer = [uint32 indices | float32 positions | uint8 RGBA colours], plus the
// per-axis minima / maxima glTF requires on the POSITION accessor.  fix_normals() on a closed, consistently wound mesh
// amounts to reversing every face when the enclosed (signed) volume is negative: `flip`.
// ------------------------------------------------------------------------------------------------
template <typename IdxT>
__global__ void __launch_bounds__(256) k_glb_pack(const float* __restrict__ verts, int64_t V, const IdxT* __restrict__ faces, int64_t F,
                                                  const uchar4* __restrict__ rgba, int flip, uint32_t* __restrict__ idx_out,
                                                  float* __restrict__ pos_out, uchar4* __restrict__ col_out,
                                                  unsigned int* __restrict__ minmax /* 3 x min, 3 x max as ordered uints */)
{
    const int64_t n_idx = 3 * F, n_pos = 3 * V;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_idx + V; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < n_idx) {
            const int64_t f = i / 3;
            int c = (int)(i - 3 * f);
            if (flip && c) c = 3 - c;          // (a, b, c) -> (a, c, b)
            idx_out[i] = (uint32_t)faces[3 * f + c];
        } else {
            const int64_t v = i - n_idx;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float x = verts[3 * v + k];
                pos_out[3 * v + k] = x;
                lo[k] = fminf(lo[k], x);
                hi[k] = fmaxf(hi[k], x);
            }
            if (rgba) col_out[v] = rgba[v];
        }
    }
    (void)n_pos;
    // order-preserving float -> uint map, warp tree, one atomic per warp and axis
    auto enc = [](float x) -> unsigned int { const unsigned int u = __float_as_uint(x); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); };
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        unsigned int a = enc(lo[k]), b = enc(hi[k]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a = min(a, __shfl_xor_sync(0xffffffffu, a, o));
            b = max(b, __shfl_xor_sync(0xffffffffu, b, o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&minmax[k], a);
            atomicMax(&minmax[3 + k], b);
        }
    }
}

__global__ void k_glb_minmax_init(unsigned int* m)
{
    if (threadIdx.x < 3) m[threadIdx.x] = 0xffffffffu;
    else if (threadIdx.x < 6) m[threadIdx.x] = 0u;
}

__global__ void k_glb_minmax_decode(unsigned int* m)
{
    if (threadIdx.x < 6) {
        const unsigned int u = m[threadIdx.x];
        m[threadIdx.x] = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
    }
}

extern "C" int64_t t3d_glb_payload_bytes(int64_t V, int64_t F, int with_colors) { return 12 * F + 12 * V + (with_colors ? 4 * V : 0); }

// bin_out: t3d_glb_payload_bytes bytes; minmax_f32x6: {min x3, max x3} of the vertex columns (device, float32)
extern "C" int t3d_glb_pack(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64, const void* rgba_u8,
                            int flip_winding, void* bin_out, void* minmax_f32x6, void* stream)
{
    if (V <= 0 || F <= 0 || V > 0xffffffffll) { t3d_set_error("t3d_glb_pack: bad sizes"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    char* out = (char*)bin_out;
    uint32_t* idx_out = (uint32_t*)out;
    float* pos_out = (float*)(out + 12 * F);
    uchar4* col_out = (uchar4*)(out + 12 * F + 12 * V);
    unsigned int* mm = (unsigned int*)minmax_f32x6;
    k_glb_minmax_init<<<1, 32, 0, st>>>(mm);
    const int64_t items = 3 * F + V;
    int64_t blocks = (items + 255) / 256;
    if (blocks > (int64_t)T3D_NUM_SMS * 16) blocks = (int64_t)T3D_NUM_SMS * 16;
    if (faces_are_i64)
        k_glb_pack<long long><<<(unsigned)blocks, 256, 0, st>>>((const float*)verts_f32, V, (const long long*)faces, F, (const uchar4*)rgba_u8,
                                                                flip_winding, idx_out, pos_out, col_out, mm);
    else
        k_glb_pack<int><<<(unsigned)blocks, 256, 0, st>>>((const float*)verts_f32, V, (const int*)faces, F, (const uchar4*)rgba_u8,
                                                          flip_winding, idx_out, pos_out, col_out, mm);
    k_glb_minmax_decode<<<1, 32, 0, st>>>(mm);
    T3D_CHECK_LAUNCH("t3d_glb_pack");
    t3d_count_launches(3);
    return 0;
}
