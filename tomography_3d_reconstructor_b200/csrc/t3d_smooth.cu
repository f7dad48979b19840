// t3d_smooth.cu -- vertex adjacency and Taubin smoothing of a triangle mesh (oracle: tests/smooth_oracle.py, which writes
// trimesh.smoothing.filter_taubin with the equal-weight Laplacian out in numpy).
//
//   adjacency  count: one thread per face adds two raw entries per edge whose ends differ to the counters of its two end
//                vertices; scan -> raw row offsets (uint64)
//              fill: the same edges again, each entry placed in its row by a per-vertex cursor (the counter, counted down),
//                so a row holds its entries in no particular order
//              rows: one warp per row of at most 64 raw entries sorts them in registers (bitonic, two per lane) and writes
//                the first of each run of equal ids back to the front of the row; a longer row (only host meshes such as
//                fans have one) is listed and sorted in place by one block, whatever its length, then de-duplicated the
//                same way
//              scan of the unique counts -> offsets (int64) and N; emit: the unique prefix of each row -> neighbours
//   taubin     one launch per iteration, thread per vertex: s = +0.0, s = s + w * x[j] over the neighbours in ascending
//              order, dd = s - x[i], x[i] + lamb * dd (even) or x[i] - nu * dd (odd), all with __dmul_rn / __dadd_rn /
//              __dsub_rn so nothing contracts into an FMA; float64 iterates ping-pong in the workspace, the first step reads
//              the float32 input and the last writes the float32 output
#include <limits.h>
#include <math.h>
#include <stdint.h>

#include "t3d.h"
#include "t3d_common.cuh"

#define SM_THREADS 256
#define SM_WARP_ROW 64            // raw entries a warp sorts in registers, two per lane
#define SM_LONG_THREADS 512
#define SM_LONG_CHUNK 4096        // entries of a long row sorted in shared memory at a time (a power of two)
// the scan of the raw counts adds a tile's counts in 32 bits and a face adds at most 6 raw entries
#define SM_MAX_FACES ((int64_t)(UINT32_MAX / 6))

static inline int64_t sm_align(int64_t x) { return (x + 255) & ~(int64_t)255; }
static unsigned sm_blocks(int64_t threads) { return (unsigned)((threads + SM_THREADS - 1) / SM_THREADS); }

// ---- adjacency: raw entries -----------------------------------------------------------------------------------------
template <typename IdxT>
__device__ __forceinline__ bool sm_face(const IdxT* __restrict__ faces, int64_t f, int64_t V, int64_t v[3])
{
    v[0] = (int64_t)faces[3 * f];
    v[1] = (int64_t)faces[3 * f + 1];
    v[2] = (int64_t)faces[3 * f + 2];
    return v[0] >= 0 && v[0] < V && v[1] >= 0 && v[1] < V && v[2] >= 0 && v[2] < V;
}

template <typename IdxT>
__global__ void __launch_bounds__(SM_THREADS) k_adj_count(const IdxT* __restrict__ faces, int64_t F, int64_t V, uint32_t* __restrict__ cnt,
                                                          unsigned long long* __restrict__ n_bad)
{
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    int64_t v[3];
    if (!sm_face(faces, f, V, v)) {
        atomicAdd(n_bad, 1ull);
        return;
    }
#pragma unroll
    for (int e = 0; e < 3; ++e) {
        const int64_t a = v[e], b = v[e == 2 ? 0 : e + 1];
        if (a != b) {
            atomicAdd(cnt + a, 1u);
            atomicAdd(cnt + b, 1u);
        }
    }
}

template <typename IdxT>
__global__ void __launch_bounds__(SM_THREADS) k_adj_fill(const IdxT* __restrict__ faces, int64_t F, int64_t V,
                                                         const unsigned long long* __restrict__ raw_off, uint32_t* __restrict__ cursor,
                                                         int32_t* __restrict__ raw)
{
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    int64_t v[3];
    if (!sm_face(faces, f, V, v)) return;
#pragma unroll
    for (int e = 0; e < 3; ++e) {
        const int64_t a = v[e], b = v[e == 2 ? 0 : e + 1];
        if (a != b) {
            raw[raw_off[a] + atomicSub(cursor + a, 1u) - 1u] = (int32_t)b;
            raw[raw_off[b] + atomicSub(cursor + b, 1u) - 1u] = (int32_t)a;
        }
    }
}

// ---- adjacency: sort and de-duplicate each row ----------------------------------------------------------------------
// Rows of at most 64 entries: one warp, element k = 2 * lane + s in register e_s, padded with INT_MAX (above every vertex
// id, since V <= INT_MAX).  The cursors of k_adj_fill ended at 0, so ucnt holds 0 for every row until it is written here.
__global__ void __launch_bounds__(SM_THREADS) k_adj_rows(const unsigned long long* __restrict__ raw_off, int64_t V, int32_t* __restrict__ raw,
                                                         uint32_t* __restrict__ ucnt, int32_t* __restrict__ long_rows,
                                                         unsigned int* __restrict__ n_long)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= V) return;                                    // warp-uniform
    const int lane = threadIdx.x & 31;
    const unsigned long long b = raw_off[row];
    const int64_t n = (int64_t)(raw_off[row + 1] - b);
    if (n == 0) return;
    if (n > SM_WARP_ROW) {
        if (lane == 0) long_rows[atomicAdd(n_long, 1u)] = (int32_t)row;
        return;
    }
    int32_t* r = raw + b;
    int e0 = (2 * lane < n) ? r[2 * lane] : INT_MAX;
    int e1 = (2 * lane + 1 < n) ? r[2 * lane + 1] : INT_MAX;
#pragma unroll
    for (int size = 2; size <= SM_WARP_ROW; size <<= 1) {
        const bool up = ((2 * lane) & size) == 0;            // the same for both elements of a lane once size >= 2
#pragma unroll
        for (int stride = size >> 1; stride > 1; stride >>= 1) {
            const int o0 = __shfl_xor_sync(0xffffffffu, e0, stride >> 1), o1 = __shfl_xor_sync(0xffffffffu, e1, stride >> 1);
            const bool keep_min = (((2 * lane) & stride) == 0) == up;
            e0 = keep_min ? min(e0, o0) : max(e0, o0);
            e1 = keep_min ? min(e1, o1) : max(e1, o1);
        }
        const int lo = min(e0, e1), hi = max(e0, e1);        // stride 1: the two elements of the lane
        e0 = up ? lo : hi;
        e1 = up ? hi : lo;
    }
    const int p0 = __shfl_up_sync(0xffffffffu, e1, 1);
    const bool u0 = 2 * lane < n && (lane == 0 || e0 != p0);
    const bool u1 = 2 * lane + 1 < n && e1 != e0;
    const uint32_t b0 = __ballot_sync(0xffffffffu, u0), b1 = __ballot_sync(0xffffffffu, u1);
    const uint32_t lt = (1u << lane) - 1u;
    const int pos = __popc(b0 & lt) + __popc(b1 & lt);
    // every lane has read its entries (the shuffles above consumed them), so the row can be overwritten in place
    if (u0) r[pos] = e0;
    if (u1) r[pos + (u0 ? 1 : 0)] = e1;
    if (lane == 0) ucnt[row] = (uint32_t)(__popc(b0) + __popc(b1));
}

// One step of the bitonic network in its all-ascending form (every comparator puts the smaller value at the lower index):
// pair p of the flip of blocks of `size` (partner i ^ (size - 1)) when flip, else of the half-cleaner of `stride`
// (partner i + stride).
__device__ __forceinline__ void sm_pair(int64_t p, int64_t size, int64_t stride, bool flip, int64_t& i, int64_t& j)
{
    if (flip) {
        const int64_t half = size >> 1;
        i = (p / half) * size + p % half;
        j = i ^ (size - 1);
    } else {
        i = (p / stride) * 2 * stride + p % stride;
        j = i + stride;
    }
}

// a step over a[0, n) in global memory; comparators that reach past n are skipped (see sm_block_sort)
__device__ void sm_global_step(int32_t* a, int64_t n, int64_t P, int64_t size, int64_t stride, bool flip)
{
    for (int64_t p = threadIdx.x; p < P / 2; p += blockDim.x) {
        int64_t i, j;
        sm_pair(p, size, stride, flip, i, j);
        if (j < n) {
            const int32_t x = a[i], y = a[j];
            if (x > y) {
                a[i] = y;
                a[j] = x;
            }
        }
    }
    __syncthreads();
}

__device__ __forceinline__ void sm_shared_step(int32_t* sh, int64_t C, int64_t size, int64_t stride, bool flip)
{
    for (int64_t p = threadIdx.x; p < C / 2; p += blockDim.x) {
        int64_t i, j;
        sm_pair(p, size, stride, flip, i, j);
        const int32_t x = sh[i], y = sh[j];
        if (x > y) {
            sh[i] = y;
            sh[j] = x;
        }
    }
    __syncthreads();
}

// the steps whose partners lie in one chunk of C entries, chunk by chunk in shared memory (padded with INT_MAX): a whole
// sort of each chunk (full), or the half-cleaners of strides C/2 .. 1 that end every larger size
__device__ void sm_chunk_steps(int32_t* a, int64_t n, int64_t C, int32_t* sh, bool full)
{
    for (int64_t c0 = 0; c0 < n; c0 += C) {
        for (int64_t t = threadIdx.x; t < C; t += blockDim.x) sh[t] = (c0 + t < n) ? a[c0 + t] : INT_MAX;
        __syncthreads();
        if (full) {
            for (int64_t size = 2; size <= C; size <<= 1) {
                sm_shared_step(sh, C, size, 0, true);
                for (int64_t stride = size >> 2; stride >= 1; stride >>= 1) sm_shared_step(sh, C, size, stride, false);
            }
        } else {
            for (int64_t stride = C >> 1; stride >= 1; stride >>= 1) sm_shared_step(sh, C, 0, stride, false);
        }
        for (int64_t t = threadIdx.x; t < C; t += blockDim.x)
            if (c0 + t < n) a[c0 + t] = sh[t];
        __syncthreads();
    }
}

// Sort a[0, n) ascending in place, for any n, by one block.  With +inf in the positions n .. P - 1 (P the next power of
// two) the all-ascending network never moves a finite value there, so comparators that reach past n are skipped and
// nothing beyond n is read or written.  Sizes up to the chunk run in shared memory; for each larger size the flip and the
// strides of at least a chunk run over global memory, the rest again chunk by chunk in shared memory.
__device__ void sm_block_sort(int32_t* a, int64_t n, int32_t* sh)
{
    int64_t P = 1;
    while (P < n) P <<= 1;
    const int64_t C = P < SM_LONG_CHUNK ? P : SM_LONG_CHUNK;
    sm_chunk_steps(a, n, C, sh, true);
    for (int64_t size = 2 * C; size <= P; size <<= 1) {
        sm_global_step(a, n, P, size, 0, true);
        for (int64_t stride = size >> 2; stride >= C; stride >>= 1) sm_global_step(a, n, P, size, stride, false);
        sm_chunk_steps(a, n, C, sh, false);
    }
}

// Long rows: one block per listed row, in place: sort, then keep the first of each run of equal ids at the front.
__global__ void __launch_bounds__(SM_LONG_THREADS) k_adj_long(const unsigned long long* __restrict__ raw_off, int32_t* raw,
                                                              uint32_t* __restrict__ ucnt, const int32_t* __restrict__ long_rows,
                                                              const unsigned int* __restrict__ n_long)
{
    __shared__ int32_t sh[SM_LONG_CHUNK];
    __shared__ uint32_t s_warp[SM_LONG_THREADS / 32];
    const unsigned nl = *n_long;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (unsigned q = blockIdx.x; q < nl; q += gridDim.x) {
        const int32_t row = long_rows[q];
        const unsigned long long b = raw_off[row];
        const int64_t n = (int64_t)(raw_off[row + 1] - b);
        int32_t* a = raw + b;
        sm_block_sort(a, n, sh);
        // writes of a tile go below the positions it read, and a position the tile before wrote just below this tile's
        // first read holds the value it held (the map is the identity up to there), so one pass in place suffices
        uint32_t u = 0;
        for (int64_t t0 = 0; t0 < n; t0 += SM_LONG_THREADS) {
            const int64_t k = t0 + threadIdx.x;
            const int32_t v = k < n ? a[k] : 0;
            const bool f = k < n && (k == 0 || v != a[k - 1]);
            const uint32_t bal = __ballot_sync(0xffffffffu, f);
            if (lane == 0) s_warp[w] = __popc(bal);
            __syncthreads();
            uint32_t before = 0, tot = 0;
#pragma unroll
            for (int x = 0; x < SM_LONG_THREADS / 32; ++x) {
                if (x < w) before += s_warp[x];
                tot += s_warp[x];
            }
            __syncthreads();
            if (f) a[u + before + __popc(bal & ((1u << lane) - 1u))] = v;
            u += tot;
            __syncthreads();
        }
        if (threadIdx.x == 0) ucnt[row] = u;
    }
}

__global__ void __launch_bounds__(SM_THREADS) k_adj_emit(const unsigned long long* __restrict__ raw_off, const int32_t* __restrict__ raw,
                                                         int64_t V, const long long* __restrict__ off, int32_t* __restrict__ nb)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const long long o = off[i], m = off[i + 1] - o;
    const int32_t* src = raw + raw_off[i];
    for (long long k = 0; k < m; ++k) nb[o + k] = src[k];
}

// ---- Taubin step ----------------------------------------------------------------------------------------------------
template <typename InT, typename OutT>
__global__ void __launch_bounds__(SM_THREADS) k_taubin(const InT* __restrict__ x, int64_t V, const long long* __restrict__ off,
                                                       const int32_t* __restrict__ nb, double coef, int odd, OutT* __restrict__ y)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const long long b = off[i], e = off[i + 1];
    double r0 = (double)x[3 * i], r1 = (double)x[3 * i + 1], r2 = (double)x[3 * i + 2];
    if (e > b) {
        const double w = __ddiv_rn(1.0, (double)(e - b));
        double s0 = 0.0, s1 = 0.0, s2 = 0.0;
        for (long long k = b; k < e; ++k) {
            const int64_t j = nb[k];
            s0 = __dadd_rn(s0, __dmul_rn(w, (double)x[3 * j]));
            s1 = __dadd_rn(s1, __dmul_rn(w, (double)x[3 * j + 1]));
            s2 = __dadd_rn(s2, __dmul_rn(w, (double)x[3 * j + 2]));
        }
        const double d0 = __dsub_rn(s0, r0), d1 = __dsub_rn(s1, r1), d2 = __dsub_rn(s2, r2);
        if (odd) {
            r0 = __dsub_rn(r0, __dmul_rn(coef, d0));
            r1 = __dsub_rn(r1, __dmul_rn(coef, d1));
            r2 = __dsub_rn(r2, __dmul_rn(coef, d2));
        } else {
            r0 = __dadd_rn(r0, __dmul_rn(coef, d0));
            r1 = __dadd_rn(r1, __dmul_rn(coef, d1));
            r2 = __dadd_rn(r2, __dmul_rn(coef, d2));
        }
    }
    if (sizeof(OutT) == 4) {
        y[3 * i] = (OutT)__double2float_rn(r0);
        y[3 * i + 1] = (OutT)__double2float_rn(r1);
        y[3 * i + 2] = (OutT)__double2float_rn(r2);
    } else {
        y[3 * i] = (OutT)r0;
        y[3 * i + 1] = (OutT)r1;
        y[3 * i + 2] = (OutT)r2;
    }
}

// ---- C ABI ----------------------------------------------------------------------------------------------------------
struct AdjWs { unsigned int* n_long; unsigned long long* raw_total; uint32_t* cnt; int64_t zero_bytes; unsigned long long* raw_off;
               int32_t* long_rows; void* scan; int32_t* raw; };

// [n_long, raw total | counters (V + 1)] (zeroed together) [raw offsets (V + 1)] [long rows (V)] [scan] [raw entries (6F)]
static int64_t adj_ws(int64_t V, int64_t F, char* ws, AdjWs* o)
{
    int64_t off = 0;
    if (o) {
        o->n_long = (unsigned int*)ws;
        o->raw_total = (unsigned long long*)(ws + 8);
    }
    off += 256;
    if (o) o->cnt = (uint32_t*)(ws + off);
    off += sm_align(4 * (V + 1));
    if (o) o->zero_bytes = off;
    if (o) o->raw_off = (unsigned long long*)(ws + off);
    off += sm_align(8 * (V + 1));
    if (o) o->long_rows = (int32_t*)(ws + off);
    off += sm_align(4 * V);
    if (o) o->scan = ws + off;
    off += sm_align(t3d_scan_workspace_bytes(V + 1, 1));
    if (o) o->raw = (int32_t*)(ws + off);
    return off + sm_align(4 * 6 * F);
}

static int adj_sizes_ok(const char* who, int64_t V, int64_t F)
{
    if (V < 0 || V > INT_MAX) {
        t3d_set_error("%s: %lld vertices, more than the int32 neighbour ids allow (%d)", who, (long long)V, INT_MAX);
        return 2;
    }
    if (F < 0 || F > SM_MAX_FACES) {
        t3d_set_error("%s: %lld faces; the raw adjacency entries (up to 6 per face) are counted in 32 bits, so at most %lld faces",
                      who, (long long)F, (long long)SM_MAX_FACES);
        return 2;
    }
    return 0;
}

extern "C" int64_t t3d_mesh_adjacency_workspace_bytes(int64_t V, int64_t F)
{
    if (V < 0 || F < 0) return 0;
    return adj_ws(V, F, nullptr, nullptr);
}

extern "C" int t3d_mesh_adjacency_count(const void* faces, int64_t F, int faces_are_i64, int64_t V, void* offsets_i64, void* n_u64,
                                        void* workspace, void* stream)
{
    if (int rc = adj_sizes_ok("t3d_mesh_adjacency_count", V, F)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    AdjWs w;
    adj_ws(V, F, (char*)workspace, &w);
    if (t3d_zero_async(n_u64, 16, st) || t3d_zero_async(workspace, w.zero_bytes, st)) return 1;
    unsigned long long* n_bad = (unsigned long long*)n_u64 + 1;
    if (F > 0) {
        if (faces_are_i64)
            k_adj_count<long long><<<sm_blocks(F), SM_THREADS, 0, st>>>((const long long*)faces, F, V, w.cnt, n_bad);
        else
            k_adj_count<int32_t><<<sm_blocks(F), SM_THREADS, 0, st>>>((const int32_t*)faces, F, V, w.cnt, n_bad);
        T3D_CHECK_LAUNCH("t3d_mesh_adjacency_count count");
        t3d_count_launches(1);
    }
    if (int rc = t3d_exclusive_scan_u32_dev(w.cnt, w.raw_off, V + 1, V + 1, 1, 1, 0, nullptr, w.raw_total, w.scan, stream)) return rc;
    if (F > 0 && V > 0) {
        if (faces_are_i64)
            k_adj_fill<long long><<<sm_blocks(F), SM_THREADS, 0, st>>>((const long long*)faces, F, V, w.raw_off, w.cnt, w.raw);
        else
            k_adj_fill<int32_t><<<sm_blocks(F), SM_THREADS, 0, st>>>((const int32_t*)faces, F, V, w.raw_off, w.cnt, w.raw);
        T3D_CHECK_LAUNCH("t3d_mesh_adjacency_count fill");
        k_adj_rows<<<sm_blocks(32 * V), SM_THREADS, 0, st>>>(w.raw_off, V, w.raw, w.cnt, w.long_rows, w.n_long);
        T3D_CHECK_LAUNCH("t3d_mesh_adjacency_count rows");
        k_adj_long<<<2 * T3D_NUM_SMS, SM_LONG_THREADS, 0, st>>>(w.raw_off, w.raw, w.cnt, w.long_rows, w.n_long);
        T3D_CHECK_LAUNCH("t3d_mesh_adjacency_count long rows");
        t3d_count_launches(3);
    }
    return t3d_exclusive_scan_u32_dev(w.cnt, offsets_i64, V + 1, V + 1, 1, 1, 0, nullptr, n_u64, w.scan, stream);
}

extern "C" int t3d_mesh_adjacency_emit(int64_t V, int64_t F, const void* offsets_i64, void* neighbours_i32, void* workspace, void* stream)
{
    if (int rc = adj_sizes_ok("t3d_mesh_adjacency_emit", V, F)) return rc;
    if (V == 0 || F == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    AdjWs w;
    adj_ws(V, F, (char*)workspace, &w);
    k_adj_emit<<<sm_blocks(V), SM_THREADS, 0, st>>>(w.raw_off, w.raw, V, (const long long*)offsets_i64, (int32_t*)neighbours_i32);
    T3D_CHECK_LAUNCH("t3d_mesh_adjacency_emit");
    t3d_count_launches(1);
    return 0;
}

extern "C" int64_t t3d_mesh_taubin_workspace_bytes(int64_t V)
{
    return V > 0 ? 2 * sm_align(24 * V) : 0;
}

extern "C" int t3d_mesh_taubin(const void* verts_f32, int64_t V, const void* offsets_i64, const void* neighbours_i32, int iterations,
                               double lamb, double nu, void* verts_out_f32, void* workspace, void* stream)
{
    if (V < 0 || V > INT_MAX) {
        t3d_set_error("t3d_mesh_taubin: %lld vertices, more than the int32 neighbour ids allow (%d)", (long long)V, INT_MAX);
        return 2;
    }
    if (iterations < 0 || !isfinite(lamb) || !isfinite(nu)) {
        t3d_set_error("t3d_mesh_taubin: iterations %d, lamb %g, nu %g (iterations >= 0 and finite factors required)", iterations, lamb, nu);
        return 2;
    }
    if (V == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (iterations == 0) {
        if (verts_out_f32 != verts_f32) T3D_CUDA(cudaMemcpyAsync(verts_out_f32, verts_f32, 12 * V, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    const long long* off = (const long long*)offsets_i64;
    const int32_t* nb = (const int32_t*)neighbours_i32;
    const float* in = (const float*)verts_f32;
    float* out = (float*)verts_out_f32;
    double* buf[2] = {(double*)workspace, (double*)((char*)workspace + sm_align(24 * V))};
    const unsigned g = sm_blocks(V);
    for (int it = 0; it < iterations; ++it) {
        const double c = (it & 1) ? nu : lamb;
        const bool first = it == 0, last = it == iterations - 1;
        if (first && last)
            k_taubin<float, float><<<g, SM_THREADS, 0, st>>>(in, V, off, nb, c, it & 1, out);
        else if (first)
            k_taubin<float, double><<<g, SM_THREADS, 0, st>>>(in, V, off, nb, c, it & 1, buf[0]);
        else if (last)
            k_taubin<double, float><<<g, SM_THREADS, 0, st>>>(buf[(it - 1) & 1], V, off, nb, c, it & 1, out);
        else
            k_taubin<double, double><<<g, SM_THREADS, 0, st>>>(buf[(it - 1) & 1], V, off, nb, c, it & 1, buf[it & 1]);
        T3D_CHECK_LAUNCH("t3d_mesh_taubin");
    }
    t3d_count_launches(iterations);
    return 0;
}
