// t3d_label.cu -- connected components of a bit-packed occupancy volume (oracle: scipy.ndimage.label with the 6- or
// 26-connected structure), labelled over x-runs instead of voxels.
//
// A run is a maximal stretch of set bits along x in one row; in the packed layout its first bit is b & ~((b << 1) | carry)
// and its last bit b & ~((b >> 1) | carry'), so a row's runs are found word by word without looking at single voxels.
//   count   k_cc_count: runs per row (warp per row), then t3d_exclusive_scan_u32_dev -> row bases and the total R
//   label   k_cc_emit: (x_begin, x_end, row) per run in raster order, parent[i] = i
//           k_cc_merge: each run is united with the overlapping runs of the earlier neighbour rows (found by a binary search
//             over the sorted run ends of that row); union-find with roots linked towards the smaller run index by
//             atomicMin (Playne & Hawick), so the root of a component is its first run in raster order whatever the
//             order the merges happen in
//           k_cc_flatten: parent[i] = root, a bitmask of the roots; scan of its popcounts; k_cc_number: label = 1 + roots
//             before the run's root = scipy's numbering (components in raster order of their first voxel)
//   stats   counts and extents by integer atomics (exact in any order; a warp whose 32 runs share a label adds once)
//   volumes a component spans every plane between its zmin and zmax (z steps by at most one along a path), so its
//           per-plane counts fit a dense table of zmax - zmin + 1 entries, sum <= R; integer atomics fill it, then one
//           thread per component adds count * slice volume in float64 in ascending z (the reference's order)
//   expand / select: warp per row, the run of a set bit is the row's base + (run starts at or before it) - 1
#include <limits.h>
#include <stdint.h>
#include <string.h>

#include "t3d.h"
#include "t3d_common.cuh"

#define CC_THREADS 256

static inline int64_t cc_align(int64_t x) { return (x + 255) & ~(int64_t)255; }

// word w of a row (0 outside [0, nw)), the first bits (s) and last bits (e) of its runs
__device__ __forceinline__ void cc_word(const uint32_t* __restrict__ row, int w, int nw, uint32_t& b, uint32_t& s, uint32_t& e)
{
    b = (w < nw) ? row[w] : 0u;
    const uint32_t prev = (w > 0 && w <= nw) ? row[w - 1] : 0u;
    const uint32_t next = (w + 1 < nw) ? row[w + 1] : 0u;
    s = b & ~((b << 1) | (prev >> 31));
    e = b & ~((b >> 1) | (next << 31));
}

__global__ void __launch_bounds__(CC_THREADS) k_cc_count(const uint32_t* __restrict__ bits, int64_t rows, int wpr, int nw,
                                                         uint32_t* __restrict__ row_runs)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row > rows) return;
    uint32_t c = 0;
    if (row < rows) {
        const uint32_t* r = bits + row * wpr;
        for (int w = lane_id(); w < nw; w += 32) {
            uint32_t b, s, e;
            cc_word(r, w, nw, b, s, e);
            c += __popc(s);
        }
        c = warp_sum(c);
    }
    if (lane_id() == 0) row_runs[row] = c;   // row_runs[rows] = 0: the scan leaves R there
}

__global__ void __launch_bounds__(CC_THREADS) k_cc_emit(const uint32_t* __restrict__ bits, int64_t rows, int wpr, int nw,
                                                        const uint32_t* __restrict__ row_base, int64_t R, int32_t* __restrict__ rx0,
                                                        int32_t* __restrict__ rx1, int32_t* __restrict__ rrow,
                                                        int32_t* __restrict__ parent)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= rows) return;
    const uint32_t* r = bits + row * wpr;
    const uint32_t l = lane_id();
    int64_t bs = row_base[row], be = bs;
    for (int g = 0; g < nw; g += 32) {
        const int w = g + (int)l;
        uint32_t b, s, e;
        cc_word(r, w, nw, b, s, e);
        const uint32_t cs = __popc(s), ce = __popc(e);
        const uint32_t is = warp_incl_scan(cs), ie = warp_incl_scan(ce);
        int64_t ps = bs + is - cs, pe = be + ie - ce;
        while (s) {
            const int x = (w << 5) + __ffs(s) - 1;
            s &= s - 1;
            rx0[ps] = x;
            rrow[ps] = (int32_t)row;
            parent[ps] = (int32_t)ps;
            ++ps;
        }
        while (e) {
            const int x = (w << 5) + __ffs(e) - 1;
            e &= e - 1;
            rx1[pe++] = x;
        }
        bs += __shfl_sync(0xffffffffu, is, 31);
        be += __shfl_sync(0xffffffffu, ie, 31);
    }
}

// Root of x.  Parent pointers only ever decrease and always stay inside the component, so path halving with atomicMin
// keeps every link valid while merges run concurrently; loads bypass L1, which is not coherent between SMs.
__device__ __forceinline__ int cc_find(int32_t* P, int x)
{
    while (true) {
        const int p = __ldcg(P + x);
        if (p == x) return x;
        const int gp = __ldcg(P + p);
        if (gp == p) return p;
        atomicMin(P + x, gp);
        x = gp;
    }
}

__device__ __forceinline__ void cc_unite(int32_t* P, int a, int b)
{
    while (true) {
        a = cc_find(P, a);
        b = cc_find(P, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(P + b, a);   // link the larger root under the smaller one
        if (old == b) return;
        b = old;                               // b was linked elsewhere meanwhile: unite that tree with a
    }
}

template <bool C26>
__global__ void __launch_bounds__(CC_THREADS) k_cc_merge(const int32_t* __restrict__ rx0, const int32_t* __restrict__ rx1,
                                                         const int32_t* __restrict__ rrow, const uint32_t* __restrict__ row_base,
                                                         int64_t R, int H, int32_t* P)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    const int row = rrow[i];
    const int z = row / H, y = row - z * H;
    const int d = C26 ? 1 : 0;
    const int a = rx0[i] - d, b = rx1[i] + d;   // neighbour runs overlap [a, b]
    auto scan_row = [&](int nrow) {
        int lo = (int)row_base[nrow], hi = (int)row_base[nrow + 1];
        const int end = hi;
        while (lo < hi) {                        // first run of the row that ends at or after a
            const int mid = (lo + hi) >> 1;
            if (rx1[mid] < a) lo = mid + 1; else hi = mid;
        }
        for (int j = lo; j < end && rx0[j] <= b; ++j) cc_unite(P, (int)i, j);
    };
    if (y > 0) scan_row(row - 1);
    if (z > 0) {
        const int below = row - H;
        if (C26 && y > 0) scan_row(below - 1);
        scan_row(below);
        if (C26 && y + 1 < H) scan_row(below + 1);
    }
}

__global__ void __launch_bounds__(CC_THREADS) k_cc_flatten(int32_t* P, int64_t R, uint32_t* __restrict__ root_mask)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool root = false;
    if (i < R) {
        const int r = cc_find(P, (int)i);
        P[i] = r;
        root = (r == (int)i);
    }
    const uint32_t m = __ballot_sync(0xffffffffu, root);
    if (lane_id() == 0 && i < R) root_mask[i >> 5] = m;
}

// label = first_label + roots before the element's root (1: scipy.ndimage.label's numbering, 0: csgraph's)
__global__ void __launch_bounds__(CC_THREADS) k_cc_number(const int32_t* __restrict__ P, int64_t R, const uint32_t* __restrict__ root_mask,
                                                          const uint32_t* __restrict__ word_base, int32_t first_label,
                                                          int32_t* __restrict__ run_label)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    const int r = P[i];
    run_label[i] = first_label + (int32_t)word_base[r >> 5] + __popc(root_mask[r >> 5] & ((1u << (r & 31)) - 1u));
}

// extents are accumulated as {INT_MAX - zmin, zmax + 1, INT_MAX - ymin, ymax + 1, INT_MAX - xmin, xmax + 1} with atomicMax
// into zeroed memory, then rewritten in place as int32 {zmin, zmax, ymin, ymax, xmin, xmax}
__global__ void __launch_bounds__(CC_THREADS) k_cc_stats(const int32_t* __restrict__ rx0, const int32_t* __restrict__ rx1,
                                                         const int32_t* __restrict__ rrow, const int32_t* __restrict__ run_label,
                                                         int64_t R, int H, unsigned long long* __restrict__ counts,
                                                         uint32_t* __restrict__ box)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < R;
    int c = -1;
    uint32_t v[6] = {0u, 0u, 0u, 0u, 0u, 0u};
    unsigned long long n = 0;
    if (live) {
        c = run_label[i] - 1;
        const int row = rrow[i], z = row / H, y = row - z * H, x0 = rx0[i], x1 = rx1[i];
        v[0] = (uint32_t)(INT_MAX - z); v[1] = (uint32_t)(z + 1);
        v[2] = (uint32_t)(INT_MAX - y); v[3] = (uint32_t)(y + 1);
        v[4] = (uint32_t)(INT_MAX - x0); v[5] = (uint32_t)(x1 + 1);
        n = (unsigned long long)(x1 - x0 + 1);
    }
    const int c0 = __shfl_sync(0xffffffffu, c, 0);
    if (__all_sync(0xffffffffu, c == c0)) {     // one component under the whole warp (large objects): one set of atomics
        if (c0 < 0) return;
        n = warp_sum(n);
#pragma unroll
        for (int k = 0; k < 6; ++k) v[k] = (uint32_t)warp_max((int)v[k]);
        if (lane_id() != 0) return;
    }
    if (!live) return;
    atomicAdd(counts + c, n);
#pragma unroll
    for (int k = 0; k < 6; ++k) atomicMax(box + 6 * (int64_t)c + k, v[k]);
}

__global__ void __launch_bounds__(CC_THREADS) k_cc_stats_final(int64_t K, uint32_t* __restrict__ box)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= K) return;
    uint32_t* b = box + 6 * c;
#pragma unroll
    for (int k = 0; k < 6; k += 2) {
        const uint32_t lo = b[k], hi = b[k + 1];
        b[k] = (uint32_t)(INT_MAX - (int)lo);
        b[k + 1] = hi - 1u;
    }
}

__global__ void __launch_bounds__(CC_THREADS) k_cc_extent(const int32_t* __restrict__ box, int64_t K, uint32_t* __restrict__ ext)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < K) ext[c] = (uint32_t)(box[6 * c + 1] - box[6 * c] + 1);
}

__global__ void __launch_bounds__(CC_THREADS) k_cc_zcount(const int32_t* __restrict__ rx0, const int32_t* __restrict__ rx1,
                                                          const int32_t* __restrict__ rrow, const int32_t* __restrict__ run_label,
                                                          int64_t R, int H, const int32_t* __restrict__ box,
                                                          const uint32_t* __restrict__ zoff, uint32_t* __restrict__ zc)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t slot = -1;
    uint32_t n = 0;
    if (i < R) {
        const int c = run_label[i] - 1, z = rrow[i] / H;
        slot = (int64_t)zoff[c] + (z - box[6 * (int64_t)c]);
        n = (uint32_t)(rx1[i] - rx0[i] + 1);
    }
    const long long s0 = __shfl_sync(0xffffffffu, (long long)slot, 0);
    if (__all_sync(0xffffffffu, slot == s0)) {  // the warp's runs lie in one plane of one component
        n = warp_sum(n);
        if (lane_id() != 0 || s0 < 0) return;
    }
    if (slot >= 0) atomicAdd(zc + slot, n);
}

// volume_calculator.py:23-35 per component: total = 0.0; for z ascending: total += count[z] * slice_volume[z], with
// slice_volume[z] = mm_x * mm_y * slice_depths[z] computed by the caller; z < n_sv only; no FMA contraction
__global__ void __launch_bounds__(CC_THREADS) k_cc_volume(const int32_t* __restrict__ box, int64_t K, const uint32_t* __restrict__ zoff,
                                                          const uint32_t* __restrict__ zc, const double* __restrict__ sv, int n_sv,
                                                          double* __restrict__ vol)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= K) return;
    const int z0 = box[6 * c], z1 = min(box[6 * c + 1], n_sv - 1);
    const uint32_t* t = zc + zoff[c];
    double total = 0.0;
    for (int z = z0; z <= z1; ++z) {
        const uint32_t n = t[z - z0];
        if (n) total = __dadd_rn(total, __dmul_rn((double)n, sv[z]));
    }
    vol[c] = total;
}

// Expand: one warp per row, 32 words at a time; for word k of the group, lane l writes voxel x = 32 (g + k) + l (coalesced):
// the label of its run, base + (starts before the word) + (starts in the word at or below bit l) - 1, or 0 if the bit is clear.
__global__ void __launch_bounds__(CC_THREADS) k_cc_expand(const uint32_t* __restrict__ bits, int64_t rows, int W, int wpr, int nw,
                                                          const uint32_t* __restrict__ row_base, const int32_t* __restrict__ run_label,
                                                          int32_t* __restrict__ labels)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= rows) return;
    const uint32_t* r = bits + row * wpr;
    const uint32_t l = lane_id();
    const uint32_t upto = (2u << l) - 1u;       // bits 0..l
    int64_t base = (int64_t)row_base[row] - 1;
    for (int g = 0; g < nw; g += 32) {
        uint32_t b, s, e;
        cc_word(r, g + (int)l, nw, b, s, e);
        const uint32_t cs = __popc(s), is = warp_incl_scan(cs), pre = is - cs;
        const int kn = min(32, nw - g);
        for (int k = 0; k < kn; ++k) {
            const uint32_t bk = __shfl_sync(0xffffffffu, b, k), sk = __shfl_sync(0xffffffffu, s, k);
            const uint32_t pk = __shfl_sync(0xffffffffu, pre, k);
            const int x = ((g + k) << 5) + (int)l;
            int32_t lab = 0;
            if ((bk >> l) & 1u) lab = run_label[base + pk + __popc(sk & upto)];
            if (x < W) labels[row * W + x] = lab;
        }
        base += __shfl_sync(0xffffffffu, is, 31);
    }
}

// Select: one warp per row, lane l owns word g + l and walks the runs inside it (one step for a full or empty word); the out
// word keeps the bits of the runs whose label has keep_u8 != 0.  Every word of the row is written, padding included.
__global__ void __launch_bounds__(CC_THREADS) k_cc_select(const uint32_t* __restrict__ bits, int64_t rows, int wpr, int nw,
                                                          const uint32_t* __restrict__ row_base, const int32_t* __restrict__ run_label,
                                                          const uint8_t* __restrict__ keep, uint32_t* __restrict__ out_bits)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= rows) return;
    const uint32_t* r = bits + row * wpr;
    const int l = (int)lane_id();
    int64_t base = (int64_t)row_base[row] - 1;
    for (int g = 0; g < wpr; g += 32) {
        uint32_t b, s, e;
        cc_word(r, g + l, nw, b, s, e);
        const uint32_t cs = __popc(s), is = warp_incl_scan(cs);
        const int64_t first = base + (is - cs);
        uint32_t out = 0, cur = b;
        while (cur) {
            const int p = __ffs(cur) - 1;                                  // first bit of a run (or of its part in this word)
            const uint32_t gaps = ~(cur | ((1u << p) - 1u));
            const uint32_t hi = gaps ? (1u << (__ffs(gaps) - 1)) : 0u;      // first clear bit above p (0: none)
            const uint32_t m = hi - (1u << p);                               // bits [p, that bit)
            if (keep[run_label[first + __popc(s & ((2u << p) - 1u))]]) out |= m;
            cur &= ~m;
        }
        if (g + l < wpr) out_bits[row * wpr + g + l] = out;
        base += __shfl_sync(0xffffffffu, is, 31);
    }
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
static unsigned cc_blocks(int64_t threads) { return (unsigned)((threads + CC_THREADS - 1) / CC_THREADS); }

static int cc_rows_ok(const char* who, int Z, int H, int W)
{
    if (Z < 0 || H < 0 || W < 0 || (int64_t)Z * H >= INT_MAX) {
        t3d_set_error("%s: bad volume shape (%d, %d, %d): Z*H must be below 2^31 - 1", who, Z, H, W);
        return 2;
    }
    return 0;
}

extern "C" int64_t t3d_cc_count_workspace_bytes(int Z, int H)
{
    return t3d_scan_workspace_bytes((int64_t)Z * H + 1, 1);
}

extern "C" int t3d_cc_count(const void* bits, int Z, int H, int W, void* row_base_u32, void* n_runs_u64, void* workspace, void* stream)
{
    if (int rc = cc_rows_ok("t3d_cc_count", Z, H, W)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rows = (int64_t)Z * H;
    k_cc_count<<<cc_blocks((rows + 1) * 32), CC_THREADS, 0, st>>>((const uint32_t*)bits, rows, t3d_wpr(W), t3d_wvalid(W),
                                                                  (uint32_t*)row_base_u32);
    T3D_CHECK_LAUNCH("t3d_cc_count");
    t3d_count_launches(1);
    return t3d_exclusive_scan_u32_dev(row_base_u32, row_base_u32, rows + 1, rows + 1, 1, 0, 0, nullptr, n_runs_u64, workspace, stream);
}

extern "C" int64_t t3d_cc_label_workspace_bytes(int64_t n_runs)
{
    const int64_t nw = (n_runs + 31) / 32;
    return cc_align(4 * n_runs) + 2 * cc_align(4 * nw) + cc_align(t3d_scan_workspace_bytes(nw, 1));
}

extern "C" int t3d_cc_label(const void* bits, int Z, int H, int W, int connectivity, const void* row_base_u32, int64_t n_runs,
                            void* runs_i32, void* run_label_i32, void* n_components_u64, void* workspace, void* stream)
{
    if (int rc = cc_rows_ok("t3d_cc_label", Z, H, W)) return rc;
    if (connectivity != 6 && connectivity != 26) {
        t3d_set_error("t3d_cc_label: connectivity must be 6 or 26, got %d", connectivity);
        return 2;
    }
    if (n_runs < 0 || n_runs > INT_MAX) {
        t3d_set_error("t3d_cc_label: %lld runs, more than the int32 run index allows (%d)", (long long)n_runs, INT_MAX);
        return 2;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (n_runs == 0) return t3d_zero_async(n_components_u64, 8, st);
    const int64_t rows = (int64_t)Z * H, R = n_runs, nw = (R + 31) / 32;
    int32_t* rx0 = (int32_t*)runs_i32;
    int32_t* rx1 = rx0 + R;
    int32_t* rrow = rx1 + R;
    char* ws = (char*)workspace;
    int32_t* parent = (int32_t*)ws; ws += cc_align(4 * R);
    uint32_t* root_mask = (uint32_t*)ws; ws += cc_align(4 * nw);
    uint32_t* word_base = (uint32_t*)ws; ws += cc_align(4 * nw);
    void* scan_ws = ws;
    const uint32_t* rb = (const uint32_t*)row_base_u32;
    k_cc_emit<<<cc_blocks(rows * 32), CC_THREADS, 0, st>>>((const uint32_t*)bits, rows, t3d_wpr(W), t3d_wvalid(W), rb, R, rx0, rx1,
                                                           rrow, parent);
    T3D_CHECK_LAUNCH("t3d_cc_label emit");
    if (connectivity == 26)
        k_cc_merge<true><<<cc_blocks(R), CC_THREADS, 0, st>>>(rx0, rx1, rrow, rb, R, H, parent);
    else
        k_cc_merge<false><<<cc_blocks(R), CC_THREADS, 0, st>>>(rx0, rx1, rrow, rb, R, H, parent);
    T3D_CHECK_LAUNCH("t3d_cc_label merge");
    k_cc_flatten<<<cc_blocks(R), CC_THREADS, 0, st>>>(parent, R, root_mask);
    T3D_CHECK_LAUNCH("t3d_cc_label flatten");
    t3d_count_launches(3);
    if (int rc = t3d_exclusive_scan_u32_dev(root_mask, word_base, nw, nw, 1, 0, 1, nullptr, n_components_u64, scan_ws, stream))
        return rc;
    k_cc_number<<<cc_blocks(R), CC_THREADS, 0, st>>>(parent, R, root_mask, word_base, 1, (int32_t*)run_label_i32);
    T3D_CHECK_LAUNCH("t3d_cc_label number");
    t3d_count_launches(1);
    return 0;
}

static int cc_k_ok(const char* who, int64_t n_runs, int64_t K)
{
    if (n_runs < 0 || n_runs > INT_MAX || K < 0 || K > n_runs) {
        t3d_set_error("%s: %lld runs / %lld components: both must fit int32 and K <= R", who, (long long)n_runs, (long long)K);
        return 2;
    }
    return 0;
}

extern "C" int t3d_cc_stats(const void* runs_i32, const void* run_label_i32, int64_t n_runs, int H, int64_t n_components,
                            void* counts_i64, void* bbox_i32, void* stream)
{
    if (int rc = cc_k_ok("t3d_cc_stats", n_runs, n_components)) return rc;
    if (n_components == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t R = n_runs, K = n_components;
    const int32_t* rx0 = (const int32_t*)runs_i32;
    if (t3d_zero_async(counts_i64, 8 * K, st) || t3d_zero_async(bbox_i32, 24 * K, st)) return 1;
    k_cc_stats<<<cc_blocks(R), CC_THREADS, 0, st>>>(rx0, rx0 + R, rx0 + 2 * R, (const int32_t*)run_label_i32, R, H,
                                                    (unsigned long long*)counts_i64, (uint32_t*)bbox_i32);
    T3D_CHECK_LAUNCH("t3d_cc_stats");
    k_cc_stats_final<<<cc_blocks(K), CC_THREADS, 0, st>>>(K, (uint32_t*)bbox_i32);
    T3D_CHECK_LAUNCH("t3d_cc_stats final");
    t3d_count_launches(2);
    return 0;
}

extern "C" int64_t t3d_cc_volumes_workspace_bytes(int64_t n_runs, int64_t n_components)
{
    return 2 * cc_align(4 * n_components) + cc_align(4 * n_runs) + cc_align(t3d_scan_workspace_bytes(n_components, 1)) + 256;
}

extern "C" int t3d_cc_volumes(const void* runs_i32, const void* run_label_i32, int64_t n_runs, int H, int64_t n_components,
                              const void* bbox_i32, const void* slice_volumes_f64, int n_slices, void* volumes_f64, void* workspace,
                              void* stream)
{
    if (int rc = cc_k_ok("t3d_cc_volumes", n_runs, n_components)) return rc;
    if (n_components == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t R = n_runs, K = n_components;
    const int32_t* rx0 = (const int32_t*)runs_i32;
    const int32_t* box = (const int32_t*)bbox_i32;
    char* ws = (char*)workspace;
    uint32_t* ext = (uint32_t*)ws; ws += cc_align(4 * K);
    uint32_t* zoff = (uint32_t*)ws; ws += cc_align(4 * K);
    uint32_t* zc = (uint32_t*)ws; ws += cc_align(4 * R);
    void* scan_ws = ws; ws += cc_align(t3d_scan_workspace_bytes(K, 1));
    void* total = ws;
    k_cc_extent<<<cc_blocks(K), CC_THREADS, 0, st>>>(box, K, ext);
    T3D_CHECK_LAUNCH("t3d_cc_volumes extent");
    t3d_count_launches(1);
    if (int rc = t3d_exclusive_scan_u32_dev(ext, zoff, K, K, 1, 0, 0, nullptr, total, scan_ws, stream)) return rc;
    if (t3d_zero_async(zc, 4 * R, st)) return 1;
    k_cc_zcount<<<cc_blocks(R), CC_THREADS, 0, st>>>(rx0, rx0 + R, rx0 + 2 * R, (const int32_t*)run_label_i32, R, H, box, zoff, zc);
    T3D_CHECK_LAUNCH("t3d_cc_volumes zcount");
    k_cc_volume<<<cc_blocks(K), CC_THREADS, 0, st>>>(box, K, zoff, zc, (const double*)slice_volumes_f64, n_slices < 0 ? 0 : n_slices,
                                                     (double*)volumes_f64);
    T3D_CHECK_LAUNCH("t3d_cc_volumes volume");
    t3d_count_launches(2);
    return 0;
}

extern "C" int t3d_cc_expand(const void* bits, int Z, int H, int W, const void* row_base_u32, const void* run_label_i32,
                             void* labels_i32, void* stream)
{
    if (int rc = cc_rows_ok("t3d_cc_expand", Z, H, W)) return rc;
    const int64_t rows = (int64_t)Z * H;
    if (rows == 0 || W == 0) return 0;
    k_cc_expand<<<cc_blocks(rows * 32), CC_THREADS, 0, (cudaStream_t)stream>>>(
        (const uint32_t*)bits, rows, W, t3d_wpr(W), t3d_wvalid(W), (const uint32_t*)row_base_u32, (const int32_t*)run_label_i32,
        (int32_t*)labels_i32);
    T3D_CHECK_LAUNCH("t3d_cc_expand");
    t3d_count_launches(1);
    return 0;
}

extern "C" int t3d_cc_select(const void* bits, int Z, int H, int W, const void* row_base_u32, const void* run_label_i32,
                             const void* keep_u8, void* out_bits, void* stream)
{
    if (int rc = cc_rows_ok("t3d_cc_select", Z, H, W)) return rc;
    const int64_t rows = (int64_t)Z * H;
    if (rows == 0 || W == 0) return 0;
    k_cc_select<<<cc_blocks(rows * 32), CC_THREADS, 0, (cudaStream_t)stream>>>(
        (const uint32_t*)bits, rows, t3d_wpr(W), t3d_wvalid(W), (const uint32_t*)row_base_u32, (const int32_t*)run_label_i32,
        (const uint8_t*)keep_u8, (uint32_t*)out_bits);
    T3D_CHECK_LAUNCH("t3d_cc_select");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Mesh bodies: connected components of a triangle mesh's vertex graph (oracle: scipy.sparse.csgraph.connected_components
// of the edges f0-f1 and f0-f2 of every face), with the voxel labeller's union-find over vertices instead of runs.
//   label   k_mb_init: parent[v] = v; k_mb_merge: unite(f0, f1), unite(f0, f2) per face (faces with an index outside
//           [0, V) are counted and skipped); k_cc_flatten / scan / k_cc_number with first label 0: the root of a body is
//           its smallest vertex, so bodies are numbered by their smallest vertex, as csgraph numbers them
//   stats   k_mb_vstats per vertex (count, first vertex, box) and k_mb_fstats per face (count, signed volume and area as
//           128-bit fixed point in four 32-bit limbs, each summed in a 64-bit integer); a block or warp whose elements share
//           a body sends one set of atomics; k_mb_final normalises the limbs and rounds each sum once to float64
//   select  keep bitmasks of vertices and faces, scans of their popcounts, then the compaction with remapped face ids
// ------------------------------------------------------------------------------------------------
#define MB_WARPS (CC_THREADS / 32)

__global__ void __launch_bounds__(CC_THREADS) k_mb_init(int32_t* __restrict__ P, int64_t V)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V) P[i] = (int32_t)i;
}

template <typename IdxT>
__global__ void __launch_bounds__(CC_THREADS) k_mb_merge(const IdxT* __restrict__ faces, int64_t F, int64_t V, int32_t* P,
                                                         unsigned long long* __restrict__ n_bad)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    const int64_t a = (int64_t)faces[3 * i], b = (int64_t)faces[3 * i + 1], c = (int64_t)faces[3 * i + 2];
    if (a < 0 || a >= V || b < 0 || b >= V || c < 0 || c >= V) {
        atomicAdd(n_bad, 1ull);
        return;
    }
    cc_unite(P, (int)a, (int)b);
    cc_unite(P, (int)a, (int)c);
}

// per-body accumulators of one pass: NS summed and NX max-reduced 64-bit values, NM max-reduced 32-bit values
template <int NS, int NX, int NM>
struct MbVals {
    unsigned long long s[NS > 0 ? NS : 1];
    unsigned long long x[NX > 0 ? NX : 1];
    uint32_t m[NM > 0 ? NM : 1];
};

template <int NS, int NX, int NM>
__device__ __forceinline__ void mb_warp_reduce(MbVals<NS, NX, NM>& v)
{
#pragma unroll
    for (int k = 0; k < NS; ++k) v.s[k] = warp_sum(v.s[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < NX; ++k) v.x[k] = max(v.x[k], (unsigned long long)__shfl_xor_sync(0xffffffffu, v.x[k], o));
#pragma unroll
        for (int k = 0; k < NM; ++k) v.m[k] = max(v.m[k], __shfl_xor_sync(0xffffffffu, v.m[k], o));
    }
}

template <int NS, int NX, int NM>
__device__ __forceinline__ void mb_atomics(int b, const MbVals<NS, NX, NM>& v, unsigned long long* S, unsigned long long* X, uint32_t* M)
{
#pragma unroll
    for (int k = 0; k < NS; ++k) if (v.s[k]) atomicAdd(S + (int64_t)NS * b + k, v.s[k]);
#pragma unroll
    for (int k = 0; k < NX; ++k) atomicMax(X + (int64_t)NX * b + k, v.x[k]);
#pragma unroll
    for (int k = 0; k < NM; ++k) atomicMax(M + (int64_t)NM * b + k, v.m[k]);
}

// Adds the values of every thread of the block (body b, or -1 for none) into the per-body accumulators.  All threads of the
// block call it.  A block whose threads all hold one body sends one set of atomics, a warp that does sends one, any other
// thread its own: the integer sums and maxima are the same whichever way they are grouped.
template <int NS, int NX, int NM>
__device__ __forceinline__ void mb_commit(int b, MbVals<NS, NX, NM> v, unsigned long long* S, unsigned long long* X, uint32_t* M)
{
    __shared__ int sb[MB_WARPS];
    __shared__ MbVals<NS, NX, NM> sv[MB_WARPS];
    const int w = threadIdx.x >> 5;
    const int b0 = __shfl_sync(0xffffffffu, b, 0);
    const bool wuni = __all_sync(0xffffffffu, b == b0);
    if (lane_id() == 0) sb[w] = wuni ? b0 : -1;
    __syncthreads();
    bool buni = sb[0] >= 0;
#pragma unroll
    for (int k = 1; k < MB_WARPS; ++k) buni = buni && sb[k] == sb[0];
    if (wuni) {
        mb_warp_reduce(v);
        if (!buni && lane_id() == 0 && b0 >= 0) mb_atomics(b0, v, S, X, M);
    } else if (b >= 0) {
        mb_atomics(b, v, S, X, M);
    }
    if (!buni) return;                          // the same for the whole block
    if (lane_id() == 0) sv[w] = v;
    __syncthreads();
    if (threadIdx.x != 0) return;
    MbVals<NS, NX, NM> t = sv[0];
    for (int k = 1; k < MB_WARPS; ++k) {
#pragma unroll
        for (int j = 0; j < NS; ++j) t.s[j] += sv[k].s[j];
#pragma unroll
        for (int j = 0; j < NX; ++j) t.x[j] = max(t.x[j], sv[k].x[j]);
#pragma unroll
        for (int j = 0; j < NM; ++j) t.m[j] = max(t.m[j], sv[k].m[j]);
    }
    mb_atomics(b0, t, S, X, M);
}

// float -> uint32 key in the float order; -0.0 is taken as +0.0, so a zero bound comes out as +0.0
__device__ __forceinline__ uint32_t mb_key(float f)
{
    uint32_t u = __float_as_uint(f);
    if (u == 0x80000000u) u = 0u;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float mb_unkey(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// per vertex: count, first vertex (max of ~v), box {~key(min), key(max)} per column
__global__ void __launch_bounds__(CC_THREADS) k_mb_vstats(const float* __restrict__ verts, int64_t V, const int32_t* __restrict__ vb,
                                                          unsigned long long* __restrict__ vcount, unsigned long long* __restrict__ first_inv,
                                                          uint32_t* __restrict__ box_key)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    MbVals<1, 1, 6> v = {};
    int b = -1;
    if (i < V) {
        b = vb[i];
        v.s[0] = 1;
        v.x[0] = ~(unsigned long long)i;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint32_t k = mb_key(verts[3 * i + c]);
            v.m[2 * c] = ~k;
            v.m[2 * c + 1] = k;
        }
    }
    mb_commit(b, v, vcount, first_inv, box_key);
}

// k_mesh_measure's two terms (t3d_surface.cu), left to right without FMA contraction
__device__ __forceinline__ void mb_terms(const float* a, const float* b, const float* c, double& vol, double& area)
{
    const double ax = a[0], ay = a[1], az = a[2], bx = b[0], by = b[1], bz = b[2], cx = c[0], cy = c[1], cz = c[2];
    const double nx = __dsub_rn(__dmul_rn(by, cz), __dmul_rn(bz, cy));
    const double ny = __dsub_rn(__dmul_rn(bz, cx), __dmul_rn(bx, cz));
    const double nz = __dsub_rn(__dmul_rn(bx, cy), __dmul_rn(by, cx));
    vol = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(ax, nx), __dmul_rn(ay, ny)), __dmul_rn(az, nz)), 6.0);
    const double ux = __dsub_rn(bx, ax), uy = __dsub_rn(by, ay), uz = __dsub_rn(bz, az);
    const double vx = __dsub_rn(cx, ax), vy = __dsub_rn(cy, ay), vz = __dsub_rn(cz, az);
    const double px = __dsub_rn(__dmul_rn(uy, vz), __dmul_rn(uz, vy));
    const double py = __dsub_rn(__dmul_rn(uz, vx), __dmul_rn(ux, vz));
    const double pz = __dsub_rn(__dmul_rn(ux, vy), __dmul_rn(uy, vx));
    area = __dmul_rn(0.5, __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(px, px), __dmul_rn(py, py)), __dmul_rn(pz, pz))));
}

// t rounded half-to-even to a multiple of 2^-64, as a 128-bit two's complement integer in four 32-bit limbs (in 64-bit
// slots).  |t| < 2^62 makes t * 2^64 exact and below 2^126; anything else (never accepted, see t3d_mesh_bodies_stats) is 0.
__device__ __forceinline__ void mb_fixed(double t, unsigned long long* L)
{
    L[0] = L[1] = L[2] = L[3] = 0;
    if (!(fabs(t) < 0x1p62)) return;
    const double r = rint(__dmul_rn(t, 0x1p64));
    const unsigned long long u = (unsigned long long)__double_as_longlong(r);
    const int e = (int)((u >> 52) & 0x7ff);
    if (e == 0) return;                         // r == 0
    const unsigned long long m = (u & ((1ull << 52) - 1)) | (1ull << 52);
    const int sh = e - 1075;                    // |r| = m * 2^sh, -52 <= sh <= 73 (r is an integer below 2^126)
    unsigned long long lo, hi;
    if (sh <= 0) { lo = m >> -sh; hi = 0; }
    else if (sh < 64) { lo = m << sh; hi = m >> (64 - sh); }
    else { lo = 0; hi = m << (sh - 64); }
    if (r < 0) { lo = ~lo + 1; hi = ~hi + (lo == 0 ? 1 : 0); }
    L[0] = lo & 0xffffffffull; L[1] = lo >> 32; L[2] = hi & 0xffffffffull; L[3] = hi >> 32;
}

// per face: acc[9 b] = {count, 4 volume limbs, 4 area limbs}, tmax[b] = max over the body's faces of |term| (float64 bits)
template <typename IdxT>
__global__ void __launch_bounds__(CC_THREADS) k_mb_fstats(const float* __restrict__ verts, const IdxT* __restrict__ faces, int64_t F,
                                                          const int32_t* __restrict__ vb, unsigned long long* __restrict__ acc,
                                                          unsigned long long* __restrict__ tmax)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    MbVals<9, 1, 0> v = {};
    int b = -1;
    if (i < F) {
        const int64_t f0 = (int64_t)faces[3 * i];
        b = vb[f0];
        double tv, ta;
        mb_terms(verts + 3 * f0, verts + 3 * (int64_t)faces[3 * i + 1], verts + 3 * (int64_t)faces[3 * i + 2], tv, ta);
        v.s[0] = 1;
        mb_fixed(tv, v.s + 1);
        mb_fixed(ta, v.s + 5);
        const unsigned long long mv = (unsigned long long)__double_as_longlong(fabs(tv));
        const unsigned long long ma = (unsigned long long)__double_as_longlong(fabs(ta));   // NaN sorts above every number
        v.x[0] = max(mv, ma);
    }
    mb_commit(b, v, acc, tmax, (uint32_t*)nullptr);
}

// the 128-bit sum of four limb sums c[k] (value sum_k c[k] 2^(32k) mod 2^128, read as signed) times 2^-64, rounded once
__device__ __forceinline__ double mb_to_double(const unsigned long long* c)
{
    unsigned long long w[4], carry = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned long long t = c[k] + carry;
        w[k] = t & 0xffffffffull;
        carry = t >> 32;
    }
    unsigned long long lo = w[0] | (w[1] << 32), hi = w[2] | (w[3] << 32);
    const bool neg = (hi >> 63) != 0;
    if (neg) { lo = ~lo + 1; hi = ~hi + (lo == 0 ? 1 : 0); }
    double d;
    int scale;
    if (hi == 0) {
        d = __ull2double_rn(lo);
        scale = -64;
    } else {
        // keep the top 64 bits and fold the rest into a sticky bit: the 64 -> 53-bit rounding then equals the 128 -> 53-bit one
        const int p = 63 - __clzll((long long)hi);             // leading bit of hi
        const int s = p + 1;                                    // bits shifted out of lo, 1..64
        const unsigned long long top = s == 64 ? hi : (hi << (64 - s)) | (lo >> s);
        const unsigned long long sticky = s == 64 ? (lo != 0) : ((lo << (64 - s)) != 0);
        d = __ull2double_rn(top | sticky);
        scale = s - 64;
    }
    d = __dmul_rn(d, __longlong_as_double((long long)(1023 + scale) << 52));   // exact: a power of two in the normal range
    return neg ? -d : d;
}

__global__ void __launch_bounds__(CC_THREADS) k_mb_final(int64_t B, const unsigned long long* __restrict__ acc,
                                                         const unsigned long long* __restrict__ tmax,
                                                         const unsigned long long* __restrict__ first_inv,
                                                         const uint32_t* __restrict__ box_key, long long* __restrict__ fcount,
                                                         long long* __restrict__ first, float* __restrict__ bbox,
                                                         double* __restrict__ vol, double* __restrict__ area,
                                                         unsigned long long* __restrict__ tmax_all)
{
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const unsigned long long* a = acc + 9 * b;
    fcount[b] = (long long)a[0];
    first[b] = (long long)~first_inv[b];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const uint32_t key = box_key[6 * b + k];
        bbox[6 * b + k] = mb_unkey((k & 1) ? key : ~key);
    }
    vol[b] = mb_to_double(a + 1);
    area[b] = mb_to_double(a + 5);
    if (a[0]) atomicMax(tmax_all, tmax[b]);
}

// keep bitmasks: threads [0, 32 nwv) vertices, [32 nwv, 32 (nwv + nwf)) faces; bit set iff keep[body]
template <typename IdxT>
__global__ void __launch_bounds__(CC_THREADS) k_mb_keep(const IdxT* __restrict__ faces, int64_t F, int64_t V, const int32_t* __restrict__ vb,
                                                        const uint8_t* __restrict__ keep, int64_t nwv, int64_t nwf,
                                                        uint32_t* __restrict__ vmask, uint32_t* __restrict__ fmask)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool is_v = t < 32 * nwv;
    const int64_t i = is_v ? t : t - 32 * nwv;
    bool k = false;
    if (is_v) { if (i < V) k = keep[vb[i]] != 0; }
    else if (i < F) k = keep[vb[faces[3 * i]]] != 0;
    const uint32_t m = __ballot_sync(0xffffffffu, k);
    if (lane_id() == 0 && (i >> 5) < (is_v ? nwv : nwf)) (is_v ? vmask : fmask)[i >> 5] = m;
}

__device__ __forceinline__ int64_t mb_rank(const uint32_t* mask, const uint32_t* base, int64_t i)
{
    return (int64_t)base[i >> 5] + __popc(mask[i >> 5] & ((1u << (i & 31)) - 1u));
}

__global__ void __launch_bounds__(CC_THREADS) k_mb_compact_verts(const float* __restrict__ verts, const float* __restrict__ normals,
                                                                 int64_t V, const uint32_t* __restrict__ vmask, const uint32_t* __restrict__ vbase,
                                                                 float* __restrict__ verts_out, float* __restrict__ normals_out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V || !((vmask[i >> 5] >> (i & 31)) & 1u)) return;
    const int64_t o = mb_rank(vmask, vbase, i);
#pragma unroll
    for (int c = 0; c < 3; ++c) verts_out[3 * o + c] = verts[3 * i + c];
    if (normals) {
#pragma unroll
        for (int c = 0; c < 3; ++c) normals_out[3 * o + c] = normals[3 * i + c];
    }
}

template <typename IdxT>
__global__ void __launch_bounds__(CC_THREADS) k_mb_compact_faces(const IdxT* __restrict__ faces, int64_t F, const uint32_t* __restrict__ vmask,
                                                                 const uint32_t* __restrict__ vbase, const uint32_t* __restrict__ fmask,
                                                                 const uint32_t* __restrict__ fbase, IdxT* __restrict__ faces_out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F || !((fmask[i >> 5] >> (i & 31)) & 1u)) return;
    const int64_t o = mb_rank(fmask, fbase, i);
#pragma unroll
    for (int c = 0; c < 3; ++c) faces_out[3 * o + c] = (IdxT)mb_rank(vmask, vbase, (int64_t)faces[3 * i + c]);
}

template <typename IdxT>
__global__ void __launch_bounds__(CC_THREADS) k_mb_face_body(const IdxT* __restrict__ faces, int64_t F, const int32_t* __restrict__ vb,
                                                             int32_t* __restrict__ fb)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < F) fb[i] = vb[faces[3 * i]];
}

// ---- mesh bodies: C ABI --------------------------------------------------------------------------
static int mb_sizes_ok(const char* who, int64_t F, int64_t V, int64_t B)
{
    if (V < 0 || V > INT_MAX) {
        t3d_set_error("%s: %lld vertices, more than the int32 body labels allow (%d)", who, (long long)V, INT_MAX);
        return 2;
    }
    if (B < 0 || B > V) {
        t3d_set_error("%s: %lld bodies for %lld vertices", who, (long long)B, (long long)V);
        return 2;
    }
    if (F < 0 || F > INT_MAX) {
        t3d_set_error("%s: %lld faces; the per-body sums are exact up to %d faces", who, (long long)F, INT_MAX);
        return 2;
    }
    return 0;
}

struct MbLabelWs { int32_t* parent; uint32_t* root_mask; uint32_t* word_base; void* scan; };
struct MbStatsWs { unsigned long long* acc; unsigned long long* tmax; unsigned long long* first_inv; uint32_t* box_key;
                   unsigned long long* tmax_all; int64_t zero_bytes; };
struct MbSelectWs { uint32_t* vmask; uint32_t* vbase; uint32_t* fmask; uint32_t* fbase; unsigned long long* totals; void* scan; };

static int64_t mb_label_ws(int64_t V, char* ws, MbLabelWs* o)
{
    const int64_t nw = (V + 31) / 32;
    int64_t off = 0;
    if (o) o->parent = (int32_t*)(ws + off);
    off += cc_align(4 * V);
    if (o) o->root_mask = (uint32_t*)(ws + off);
    off += cc_align(4 * nw);
    if (o) o->word_base = (uint32_t*)(ws + off);
    off += cc_align(4 * nw);
    if (o) o->scan = ws + off;
    return off + cc_align(t3d_scan_workspace_bytes(nw, 1));
}

static int64_t mb_stats_ws(int64_t B, char* ws, MbStatsWs* o)
{
    // everything the passes accumulate into lies in one range zeroed by one memset
    int64_t off = 0;
    if (o) o->acc = (unsigned long long*)(ws + off);
    off += cc_align(72 * B);
    if (o) o->tmax = (unsigned long long*)(ws + off);
    off += cc_align(8 * B);
    if (o) o->first_inv = (unsigned long long*)(ws + off);
    off += cc_align(8 * B);
    if (o) o->box_key = (uint32_t*)(ws + off);
    off += cc_align(24 * B);
    if (o) o->tmax_all = (unsigned long long*)(ws + off);
    off += 256;
    if (o) o->zero_bytes = off;
    return off;
}

static int64_t mb_select_ws(int64_t V, int64_t F, char* ws, MbSelectWs* o)
{
    const int64_t nwv = (V + 31) / 32, nwf = (F + 31) / 32;
    int64_t off = 0;
    if (o) o->vmask = (uint32_t*)(ws + off);
    off += cc_align(4 * nwv);
    if (o) o->vbase = (uint32_t*)(ws + off);
    off += cc_align(4 * nwv);
    if (o) o->fmask = (uint32_t*)(ws + off);
    off += cc_align(4 * nwf);
    if (o) o->fbase = (uint32_t*)(ws + off);
    off += cc_align(4 * nwf);
    if (o) o->totals = (unsigned long long*)(ws + off);
    off += 256;
    if (o) o->scan = ws + off;
    const int64_t sv = t3d_scan_workspace_bytes(nwv, 1), sf = t3d_scan_workspace_bytes(nwf, 1);
    return off + cc_align(sv > sf ? sv : sf);
}

extern "C" int64_t t3d_mesh_bodies_workspace_bytes(int64_t V, int64_t F, int64_t B)
{
    int64_t n = mb_label_ws(V, nullptr, nullptr);
    const int64_t s = mb_stats_ws(B, nullptr, nullptr), c = mb_select_ws(V, F, nullptr, nullptr);
    if (s > n) n = s;
    if (c > n) n = c;
    return n;
}

extern "C" int t3d_mesh_bodies_label(const void* faces, int64_t F, int faces_are_i64, int64_t V, void* vertex_body_i32,
                                     void* n_bodies_u64, void* workspace, void* stream)
{
    if (V < 0 || V > INT_MAX) {
        t3d_set_error("t3d_mesh_bodies_label: %lld vertices, more than the int32 body labels allow (%d)", (long long)V, INT_MAX);
        return 2;
    }
    if (F < 0) {
        t3d_set_error("t3d_mesh_bodies_label: bad face count %lld", (long long)F);
        return 2;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (t3d_zero_async(n_bodies_u64, 16, st)) return 1;
    MbLabelWs w;
    mb_label_ws(V, (char*)workspace, &w);
    unsigned long long* n_bad = (unsigned long long*)n_bodies_u64 + 1;
    if (V > 0) {
        k_mb_init<<<cc_blocks(V), CC_THREADS, 0, st>>>(w.parent, V);
        t3d_count_launches(1);
    }
    if (F > 0) {
        if (faces_are_i64)
            k_mb_merge<long long><<<cc_blocks(F), CC_THREADS, 0, st>>>((const long long*)faces, F, V, w.parent, n_bad);
        else
            k_mb_merge<int32_t><<<cc_blocks(F), CC_THREADS, 0, st>>>((const int32_t*)faces, F, V, w.parent, n_bad);
        t3d_count_launches(1);
    }
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_label merge");
    if (V == 0) return 0;
    const int64_t nw = (V + 31) / 32;
    k_cc_flatten<<<cc_blocks(V), CC_THREADS, 0, st>>>(w.parent, V, w.root_mask);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_label flatten");
    t3d_count_launches(1);
    if (int rc = t3d_exclusive_scan_u32_dev(w.root_mask, w.word_base, nw, nw, 1, 0, 1, nullptr, n_bodies_u64, w.scan, stream)) return rc;
    k_cc_number<<<cc_blocks(V), CC_THREADS, 0, st>>>(w.parent, V, w.root_mask, w.word_base, 0, (int32_t*)vertex_body_i32);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_label number");
    t3d_count_launches(1);
    return 0;
}

extern "C" int t3d_mesh_bodies_stats(const void* verts_f32, const void* faces, int64_t F, int faces_are_i64, int64_t V,
                                     const void* vertex_body_i32, int64_t B, void* vertex_counts_i64, void* face_counts_i64,
                                     void* first_vertex_i64, void* bbox_f32, void* volumes_f64, void* areas_f64, void* workspace,
                                     void* stream)
{
    if (int rc = mb_sizes_ok("t3d_mesh_bodies_stats", F, V, B)) return rc;
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    MbStatsWs w;
    mb_stats_ws(B, (char*)workspace, &w);
    if (t3d_zero_async(w.acc, w.zero_bytes, st) || t3d_zero_async(vertex_counts_i64, 8 * B, st)) return 1;
    const int32_t* vb = (const int32_t*)vertex_body_i32;
    k_mb_vstats<<<cc_blocks(V), CC_THREADS, 0, st>>>((const float*)verts_f32, V, vb, (unsigned long long*)vertex_counts_i64, w.first_inv,
                                                     w.box_key);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_stats vertices");
    if (F > 0) {
        if (faces_are_i64)
            k_mb_fstats<long long><<<cc_blocks(F), CC_THREADS, 0, st>>>((const float*)verts_f32, (const long long*)faces, F, vb, w.acc, w.tmax);
        else
            k_mb_fstats<int32_t><<<cc_blocks(F), CC_THREADS, 0, st>>>((const float*)verts_f32, (const int32_t*)faces, F, vb, w.acc, w.tmax);
        T3D_CHECK_LAUNCH("t3d_mesh_bodies_stats faces");
    }
    k_mb_final<<<cc_blocks(B), CC_THREADS, 0, st>>>(B, w.acc, w.tmax, w.first_inv, w.box_key, (long long*)face_counts_i64,
                                                    (long long*)first_vertex_i64, (float*)bbox_f32, (double*)volumes_f64,
                                                    (double*)areas_f64, w.tmax_all);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_stats final");
    t3d_count_launches(F > 0 ? 3 : 2);
    // the sums are exact only while no limb carries out of 128 bits: read the largest |term| back and refuse beyond it
    unsigned long long tm = 0;
    T3D_CUDA(cudaMemcpyAsync(&tm, w.tmax_all, 8, cudaMemcpyDeviceToHost, st));
    T3D_CUDA(cudaStreamSynchronize(st));
    double m;
    memcpy(&m, &tm, 8);
    if (!(m < 0x1p62) || (double)F * m >= 0x1p63) {
        t3d_set_error("t3d_mesh_bodies_stats: a face term of magnitude %g mm^3 over %lld faces: the 128-bit fixed-point sums are "
                      "exact only for |term| < 2^62 and F * max|term| < 2^63", m, (long long)F);
        return 2;
    }
    return 0;
}

extern "C" int t3d_mesh_bodies_face_body(const void* faces, int64_t F, int faces_are_i64, const void* vertex_body_i32, void* face_body_i32,
                                         void* stream)
{
    if (F < 0 || F > INT_MAX) {
        t3d_set_error("t3d_mesh_bodies_face_body: bad face count %lld", (long long)F);
        return 2;
    }
    if (F == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (faces_are_i64)
        k_mb_face_body<long long><<<cc_blocks(F), CC_THREADS, 0, st>>>((const long long*)faces, F, (const int32_t*)vertex_body_i32, (int32_t*)face_body_i32);
    else
        k_mb_face_body<int32_t><<<cc_blocks(F), CC_THREADS, 0, st>>>((const int32_t*)faces, F, (const int32_t*)vertex_body_i32, (int32_t*)face_body_i32);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_face_body");
    t3d_count_launches(1);
    return 0;
}

extern "C" int t3d_mesh_bodies_select(const void* verts_f32, const void* normals_f32, const void* faces, int64_t F, int faces_are_i64,
                                      int64_t V, const void* vertex_body_i32, int64_t B, const void* keep_u8, void* verts_out_f32,
                                      void* normals_out_f32, void* faces_out, void* workspace, void* stream)
{
    if (int rc = mb_sizes_ok("t3d_mesh_bodies_select", F, V, B)) return rc;
    if (V == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    MbSelectWs w;
    mb_select_ws(V, F, (char*)workspace, &w);
    const int64_t nwv = (V + 31) / 32, nwf = (F + 31) / 32;
    const int32_t* vb = (const int32_t*)vertex_body_i32;
    const uint8_t* keep = (const uint8_t*)keep_u8;
    if (faces_are_i64)
        k_mb_keep<long long><<<cc_blocks(32 * (nwv + nwf)), CC_THREADS, 0, st>>>((const long long*)faces, F, V, vb, keep, nwv, nwf, w.vmask, w.fmask);
    else
        k_mb_keep<int32_t><<<cc_blocks(32 * (nwv + nwf)), CC_THREADS, 0, st>>>((const int32_t*)faces, F, V, vb, keep, nwv, nwf, w.vmask, w.fmask);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_select keep");
    t3d_count_launches(1);
    if (int rc = t3d_exclusive_scan_u32_dev(w.vmask, w.vbase, nwv, nwv, 1, 0, 1, nullptr, w.totals, w.scan, stream)) return rc;
    k_mb_compact_verts<<<cc_blocks(V), CC_THREADS, 0, st>>>((const float*)verts_f32, (const float*)normals_f32, V, w.vmask, w.vbase,
                                                            (float*)verts_out_f32, (float*)normals_out_f32);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_select vertices");
    t3d_count_launches(1);
    if (F == 0) return 0;
    if (int rc = t3d_exclusive_scan_u32_dev(w.fmask, w.fbase, nwf, nwf, 1, 0, 1, nullptr, w.totals + 1, w.scan, stream)) return rc;
    if (faces_are_i64)
        k_mb_compact_faces<long long><<<cc_blocks(F), CC_THREADS, 0, st>>>((const long long*)faces, F, w.vmask, w.vbase, w.fmask, w.fbase,
                                                                          (long long*)faces_out);
    else
        k_mb_compact_faces<int32_t><<<cc_blocks(F), CC_THREADS, 0, st>>>((const int32_t*)faces, F, w.vmask, w.vbase, w.fmask, w.fbase,
                                                                        (int32_t*)faces_out);
    T3D_CHECK_LAUNCH("t3d_mesh_bodies_select faces");
    t3d_count_launches(1);
    return 0;
}
