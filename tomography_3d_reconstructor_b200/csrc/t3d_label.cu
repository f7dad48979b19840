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

__global__ void __launch_bounds__(CC_THREADS) k_cc_number(const int32_t* __restrict__ P, int64_t R, const uint32_t* __restrict__ root_mask,
                                                          const uint32_t* __restrict__ word_base, int32_t* __restrict__ run_label)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    const int r = P[i];
    run_label[i] = 1 + (int32_t)word_base[r >> 5] + __popc(root_mask[r >> 5] & ((1u << (r & 31)) - 1u));
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
    k_cc_number<<<cc_blocks(R), CC_THREADS, 0, st>>>(parent, R, root_mask, word_base, (int32_t*)run_label_i32);
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
