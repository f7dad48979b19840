// t3d_surface.cu -- SurfaceExtractor kernels (sm_100a).
//
// Reference semantics (file:line into the reference repository, and SURVEY.md section 8a):
//   field      : np.pad(1) -> float64 -> scipy gaussian_filter(sigma=0.5), surface_extractor.py:43-53
//   mc         : skimage.measure.marching_cubes(volume, level=0.5), surface_extractor.py:55
//   transform  : un-pad, _apply_variable_slice_depths, mm scaling, surface_extractor.py:57-65,82-113
//   canonical  : _ensure_manifold_mesh (np.unique rows + degenerate-face drop), :115-126
//   measures   : calculate_mesh_volume / calculate_surface_area, :128-148
//
// Design.  The marched field is a 5x5x5 Gaussian blur of a 0/1 occupancy.  Its centre tap is 0.48665 and
// each face tap 0.06586 (weights sum to 1), hence
//     voxel set   and >=1 (reflected) face neighbour set   => field >= 0.5525 > 0.5
//     voxel unset and >=1 (reflected) face neighbour unset => field <= 0.4475 < 0.5
// so the SIGN of (field - 0.5) equals the occupancy bit except at voxels whose six face neighbours all
// disagree with them; only those are evaluated exactly.  All topology (cube cases, vertex ownership,
// counts, ranks) is therefore pure bit arithmetic on a packed sign volume; float64 arithmetic in scipy's
// exact summation order is spent only on the two end points of each cut edge (vertex interpolation).
#include <stdlib.h>

#include <cub/device/device_radix_sort.cuh>

#include "t3d_field.cuh"

// ------------------------------------------------------------------------------------------------
// sign volume: S(q) = float32(field(q)) > 0.5, packed in padded coordinates (Zp, Hp, nwp).
// S equals the padded occupancy P except at voxels all of whose six (reflected) face neighbours disagree with
// them (see the header comment); those few are evaluated exactly (slow path, not inlined).
// Same shape as the morphology kernel: a thread owns one uint4 column of one padded plane and marches down FY
// rows; the padded words are funnel-shifted out of the un-padded occupancy on the fly.
// ------------------------------------------------------------------------------------------------
#define FY 8

__device__ __noinline__ uint32_t exact_sign_bits(const OccView* v, int zp, int yp, int wp, uint32_t need, uint32_t s)
{
    while (need) {
        const int b = __ffs(need) - 1;
        need &= need - 1;
        if (field_value(*v, zp, yp, (wp << 5) + b) > 0.5f) s |= 1u << b; else s &= ~(1u << b);
    }
    return s;
}

// four padded words wp = 4*wp4 .. 4*wp4+3 of padded row (zp, yp), plus the padded words to their left and right
__device__ __forceinline__ uint4 prow4(const OccView& v, int zp, int yp, int wp4, uint32_t& left, uint32_t& right)
{
    const int z = zp - v.pad, y = yp - v.pad;
    if (z < 0 || z >= v.Z || y < 0 || y >= v.H) { left = right = 0u; return make_uint4(0, 0, 0, 0); }
    const uint32_t* row = v.bits + (z * v.ps + (long long)y * v.rs);
    const int w0 = 4 * wp4;
    const uint4 o = (w0 < v.nw) ? *reinterpret_cast<const uint4*>(row + w0) : make_uint4(0, 0, 0, 0);
    const uint32_t om1 = (w0 >= 1 && w0 - 1 < v.nw) ? row[w0 - 1] : 0u;
    const uint32_t o4 = (w0 + 4 < v.nw) ? row[w0 + 4] : 0u;
    if (!v.pad) { left = om1; right = o4; return o; }
    const uint32_t om2 = (w0 >= 2 && w0 - 2 < v.nw) ? row[w0 - 2] : 0u;
    left = __funnelshift_l(om2, om1, 1);
    right = __funnelshift_l(o.w, o4, 1);
    return make_uint4(__funnelshift_l(om1, o.x, 1), __funnelshift_l(o.x, o.y, 1), __funnelshift_l(o.y, o.z, 1),
                      __funnelshift_l(o.z, o.w, 1));
}

// LEAN: words that need the exact evaluation are only RECORDED (flat word index << 32 | bit mask) and patched by
// k_field_sign_fix afterwards; the kernel then carries no call and half the registers.  If more than exc_cap words are
// recorded the caller must rerun the robust (LEAN = false) variant.
template <bool LEAN>
__global__ void __launch_bounds__(256, LEAN ? 4 : 2) k_field_sign(OccView v, uint32_t* __restrict__ sign, int nwp, int lanes_x,
                                                    int pz_per_block, int fy, unsigned long long* __restrict__ n_exact,
                                                    unsigned long long* __restrict__ exc, unsigned long long exc_cap,
                                                    unsigned long long* __restrict__ exc_count)
{
    __shared__ OccView sv;  // the rare exact path takes the view by pointer (keeps it out of registers / local memory)
    if (!LEAN) {
        if (threadIdx.x == 0) sv = v;
        __syncthreads();
    }
    const int lx = threadIdx.x % lanes_x, pz = threadIdx.x / lanes_x;
    const int nwp4 = nwp >> 2;
    const int wp4 = blockIdx.x * lanes_x + lx, zp = blockIdx.z * pz_per_block + pz, y0 = blockIdx.y * fy;
    if (pz >= pz_per_block || wp4 >= nwp4 || zp >= v.Zp) return;
    const uint4 vm = valid_mask4(wp4, v.Wp);
    const int zm_i = reflect_idx(zp - 1, v.Zp), zq_i = reflect_idx(zp + 1, v.Zp);
    const int last = v.Wp - 1, last_w = last >> 5;
    const uint32_t last_bit = 1u << (last & 31);
    uint32_t l0, r0, lc, rc, ln, rn;
    uint4 prev = prow4(v, zp, reflect_idx(y0 - 1, v.Hp), wp4, l0, r0);
    uint4 cur = prow4(v, zp, y0, wp4, lc, rc);
    const int y1 = min(v.Hp, y0 + fy);
    for (int yp = y0; yp < y1; ++yp) {
        const uint4 next = prow4(v, zp, reflect_idx(yp + 1, v.Hp), wp4, ln, rn);
        uint32_t d0, d1;
        const uint4 zm = prow4(v, zm_i, yp, wp4, d0, d1), zq = prow4(v, zq_i, yp, wp4, d0, d1);
        uint4 xm = shl1_4(cur, lc), xq = shr1_4(cur, rc);
        if (wp4 == 0) xm.x = (xm.x & ~1u) | (cur.x & 1u);  // reflect: x = -1 -> x = 0
        if ((last_w >> 2) == wp4) {                        // reflect: x = Wp -> x = Wp-1
            const int j = last_w & 3;
            if (j == 0) xq.x = (xq.x & ~last_bit) | (cur.x & last_bit);
            else if (j == 1) xq.y = (xq.y & ~last_bit) | (cur.y & last_bit);
            else if (j == 2) xq.z = (xq.z & ~last_bit) | (cur.z & last_bit);
            else xq.w = (xq.w & ~last_bit) | (cur.w & last_bit);
        }
        const uint4 any1 = or4(or4(or4(zm, zq), or4(prev, next)), or4(xm, xq));
        const uint4 all1 = and4(and4(and4(zm, zq), and4(prev, next)), and4(xm, xq));
        uint4 s = and4(cur, any1);
        uint4 need;
        need.x = ((cur.x & ~any1.x) | (~cur.x & all1.x)) & vm.x;
        need.y = ((cur.y & ~any1.y) | (~cur.y & all1.y)) & vm.y;
        need.z = ((cur.z & ~any1.z) | (~cur.z & all1.z)) & vm.z;
        need.w = ((cur.w & ~any1.w) | (~cur.w & all1.w)) & vm.w;
        if (need.x | need.y | need.z | need.w) {
            atomicAdd(n_exact, (unsigned long long)popc4(need));
            if (LEAN) {
                const unsigned long long flat = ((unsigned long long)zp * v.Hp + yp) * nwp + 4 * wp4;
                const uint32_t nd[4] = {need.x, need.y, need.z, need.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (nd[j]) {
                        const unsigned long long k = atomicAdd(exc_count, 1ull);
                        if (k < exc_cap) exc[k] = ((flat + j) << 32) | nd[j];
                    }
                }
            } else {
                if (need.x) s.x = exact_sign_bits(&sv, zp, yp, 4 * wp4, need.x, s.x);
                if (need.y) s.y = exact_sign_bits(&sv, zp, yp, 4 * wp4 + 1, need.y, s.y);
                if (need.z) s.z = exact_sign_bits(&sv, zp, yp, 4 * wp4 + 2, need.z, s.z);
                if (need.w) s.w = exact_sign_bits(&sv, zp, yp, 4 * wp4 + 3, need.w, s.w);
            }
        }
        *reinterpret_cast<uint4*>(sign + ((int64_t)zp * v.Hp + yp) * nwp + 4 * wp4) = and4(s, vm);
        prev = cur;
        cur = next; lc = ln; rc = rn;
    }
}

// patch the recorded words: exact float64 evaluation of the flagged voxels (one thread per word)
__global__ void __launch_bounds__(128) k_field_sign_fix(OccView v, uint32_t* __restrict__ sign, int nwp,
                                                        const unsigned long long* __restrict__ exc, unsigned long long exc_cap,
                                                        const unsigned long long* __restrict__ exc_count)
{
    const unsigned long long n = min(*exc_count, exc_cap);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long e = exc[i];
        const unsigned long long flat = e >> 32;
        uint32_t need = (uint32_t)e;
        const int wp = (int)(flat % nwp);
        const unsigned long long row = flat / nwp;
        const int yp = (int)(row % v.Hp), zp = (int)(row / v.Hp);
        uint32_t s = sign[flat];
        while (need) {
            const int b = __ffs(need) - 1;
            need &= need - 1;
            if (field_value(v, zp, yp, (wp << 5) + b) > 0.5f) s |= 1u << b; else s &= ~(1u << b);
        }
        sign[flat] = s;
    }
}

// ------------------------------------------------------------------------------------------------
// exclusive scan of n_arrays independent uint32 arrays (in place allowed for uint32 output), totals -> totals[k].
// Single pass with decoupled look-back (Merrill & Garland): a tile of SC_TILE items per CTA, tiles ordered by an
// atomic ticket, each tile publishes (status | value) in one 64-bit word; a tile's exclusive prefix is found by a
// warp walking back over its predecessors until it meets an inclusive prefix.  One launch, data read once.
// ------------------------------------------------------------------------------------------------
#define SC_THREADS 256
#define SC_ITEMS 8
#define SC_TILE (SC_THREADS * SC_ITEMS)
#define SC_FLAG_A (1ull << 62)   // aggregate of this tile available
#define SC_FLAG_P (2ull << 62)   // inclusive prefix available
#define SC_VALUE_MASK ((1ull << 62) - 1)

template <typename OutT>
__global__ void __launch_bounds__(SC_THREADS) k_scan_lookback(const uint32_t* __restrict__ in, OutT* __restrict__ out, int64_t n_cap,
                                                              int64_t stride, unsigned long long* __restrict__ desc, int n_tiles,
                                                              unsigned int* __restrict__ tickets, int popc_in,
                                                              const unsigned long long* __restrict__ n_dev,
                                                              unsigned long long* __restrict__ totals)
{
    const int64_t n = dev_n(n_cap, n_dev);
    const uint32_t* a = in + (int64_t)blockIdx.y * stride;
    OutT* o = out + (int64_t)blockIdx.y * stride;
    volatile unsigned long long* d = desc + (int64_t)blockIdx.y * n_tiles;   // (stride of the launch, before clamping below)
    __shared__ int s_tile;
    __shared__ uint32_t sh[SC_THREADS / 32];
    __shared__ unsigned long long s_prefix;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(tickets + blockIdx.y, 1u);
    __syncthreads();
    const int tile = s_tile;
    // only the tiles that hold data take part (capacity-sized launches with a small device-side n)
    const int64_t need = (n + SC_TILE - 1) / SC_TILE;
    n_tiles = (int)(need < 1 ? 1 : (need < n_tiles ? need : n_tiles));
    if (tile >= n_tiles) return;
    const int64_t base = (int64_t)tile * SC_TILE + (int64_t)threadIdx.x * SC_ITEMS;  // blocked arrangement
    uint32_t v[SC_ITEMS];
    uint32_t sum = 0;
#pragma unroll
    for (int k = 0; k < SC_ITEMS; ++k) {
        v[k] = (base + k < n) ? (popc_in ? (uint32_t)__popc(a[base + k]) : a[base + k]) : 0u;
        sum += v[k];
    }
    const uint32_t incl = warp_incl_scan(sum);
    if (lane_id() == 31) sh[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t woff = 0, agg = 0;
#pragma unroll
    for (int k = 0; k < SC_THREADS / 32; ++k) {
        if (k < (int)(threadIdx.x >> 5)) woff += sh[k];
        agg += sh[k];
    }
    // publish the aggregate, look back for the exclusive prefix of this tile (warp 0)
    if (threadIdx.x < 32) {
        unsigned long long prefix = 0;
        if (tile == 0) {
            if (threadIdx.x == 0) { d[0] = SC_FLAG_P | (unsigned long long)agg; }
        } else {
            if (threadIdx.x == 0) { d[tile] = SC_FLAG_A | (unsigned long long)agg; }
            int idx = tile - 1 - (int)threadIdx.x;
            while (true) {
                unsigned long long w = (idx >= 0) ? d[idx] : SC_FLAG_P;  // before tile 0: an (empty) inclusive prefix
                while (__any_sync(0xffffffffu, (w >> 62) == 0)) {        // spin until the 32 predecessors have published
                    if ((w >> 62) == 0) w = (idx >= 0) ? d[idx] : SC_FLAG_P;
                }
                const uint32_t is_p = __ballot_sync(0xffffffffu, (w >> 62) == 2);
                const int first_p = is_p ? (__ffs(is_p) - 1) : 32;       // nearest predecessor holding an inclusive prefix
                unsigned long long val = ((int)threadIdx.x <= first_p) ? (w & SC_VALUE_MASK) : 0ull;
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) val += __shfl_xor_sync(0xffffffffu, val, off);
                prefix += val;
                if (is_p) break;
                idx -= 32;
            }
            if (threadIdx.x == 0) { d[tile] = SC_FLAG_P | ((prefix + agg) & SC_VALUE_MASK); }
        }
        if (threadIdx.x == 0) {
            s_prefix = prefix;
            if (tile == n_tiles - 1) totals[blockIdx.y] = prefix + agg;
        }
    }
    __syncthreads();
    unsigned long long run = s_prefix + woff + (incl - sum);
#pragma unroll
    for (int k = 0; k < SC_ITEMS; ++k) {
        if (base + k < n) o[base + k] = (OutT)run;
        run += v[k];
    }
}

extern "C" int64_t t3d_scan_workspace_bytes(int64_t n, int n_arrays)
{
    // sized for the smallest tile any scan-like kernel of this file uses (k_unique_fused: SC_THREADS * 4 items)
    const int64_t nb = (n + SC_THREADS * 4 - 1) / (SC_THREADS * 4);
    return (nb * n_arrays + 16) * 8 + 256;
}

// in: n_arrays arrays of n_cap uint32, `stride` elements apart; out: same layout, uint32 (out_is_u64 = 0) or uint64 (1); may
// alias `in` only for uint32 output.  popcount_input = 1 scans popcount(in[i]) instead of in[i].  n_dev_u64 (optional, device):
// the true length when n_cap is only a capacity.  totals: n_arrays uint64 (device).
extern "C" int t3d_exclusive_scan_u32_dev(const void* in, void* out, int64_t n_cap, int64_t stride, int n_arrays, int out_is_u64,
                                          int popcount_input, const void* n_dev_u64, void* totals_u64, void* workspace, void* stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (n_cap <= 0 || n_arrays <= 0) {
        if (n_arrays > 0) T3D_CUDA(cudaMemsetAsync(totals_u64, 0, 8 * n_arrays, st));
        return 0;
    }
    if (n_arrays > 16) { t3d_set_error("t3d_exclusive_scan_u32_dev: at most 16 arrays per call"); return 2; }
    const int64_t nb = (n_cap + SC_TILE - 1) / SC_TILE;
    if (nb > 0x7fffffff) { t3d_set_error("t3d_exclusive_scan_u32_dev: too many elements"); return 2; }
    // workspace: [tile descriptors: nb * n_arrays u64][tickets: 16 u32], zeroed for every scan
    const size_t desc_bytes = (size_t)nb * n_arrays * 8;
    if (t3d_zero_async(workspace, desc_bytes + 64, st)) return 1;
    unsigned long long* desc = (unsigned long long*)workspace;
    unsigned int* tickets = (unsigned int*)((char*)workspace + desc_bytes);
    const unsigned long long* nd = (const unsigned long long*)n_dev_u64;
    dim3 grid((unsigned)nb, n_arrays);
    if (out_is_u64)
        k_scan_lookback<unsigned long long><<<grid, SC_THREADS, 0, st>>>((const uint32_t*)in, (unsigned long long*)out, n_cap, stride, desc,
                                                                         (int)nb, tickets, popcount_input, nd,
                                                                         (unsigned long long*)totals_u64);
    else
        k_scan_lookback<uint32_t><<<grid, SC_THREADS, 0, st>>>((const uint32_t*)in, (uint32_t*)out, n_cap, stride, desc, (int)nb, tickets,
                                                               popcount_input, nd, (unsigned long long*)totals_u64);
    T3D_CHECK_LAUNCH("t3d_exclusive_scan_u32_dev");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// C ABI: field sign / count / emit
// ------------------------------------------------------------------------------------------------
// sign volume dims: (Z+2p, H+2p, words_per_row(W+2p)).  n_exact_u64 (device, zeroed here) receives the
// number of voxels that needed the exact float64 evaluation.
extern "C" int t3d_field_sign(const void* occ_bits, int Z, int H, int W, int pad, const double* weights3, void* sign_bits,
                              void* n_exact_u64, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_field_sign: empty volume"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const OccView v = t3d_make_view(occ_bits, Z, H, W, pad, 1, weights3);
    const int nwp = t3d_wpr(v.Wp);
    T3D_CUDA(cudaMemsetAsync(n_exact_u64, 0, 8, st));
    const int nwp4 = nwp / 4, lanes_x = nwp4 < 256 ? nwp4 : 256, pzb = 256 / lanes_x;
    dim3 grid((nwp4 + lanes_x - 1) / lanes_x, (v.Hp + FY - 1) / FY, (v.Zp + pzb - 1) / pzb);
    k_field_sign<false><<<grid, 256, 0, st>>>(v, (uint32_t*)sign_bits, nwp, lanes_x, pzb, FY, (unsigned long long*)n_exact_u64, nullptr, 0,
                                              nullptr);
    T3D_CHECK_LAUNCH("t3d_field_sign");
    t3d_count_launches(1);
    return 0;
}

// Same result through the lean kernel: the (rare) words needing the exact evaluation are recorded in exc_list_u64
// (exc_cap entries) and patched by a second small kernel.  exc_count_u64 (device) receives the number of recorded
// words: if it exceeds exc_cap the sign volume is incomplete and the caller must run t3d_field_sign instead.
extern "C" int t3d_field_sign_lean(const void* occ_bits, int Z, int H, int W, int pad, const double* weights3, void* sign_bits,
                                   void* n_exact_u64, void* exc_list_u64, uint32_t exc_cap, void* exc_count_u64, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_field_sign_lean: empty volume"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const OccView v = t3d_make_view(occ_bits, Z, H, W, pad, 1, weights3);
    const int nwp = t3d_wpr(v.Wp);
    if (t3d_zero_async(n_exact_u64, 8, st) || t3d_zero_async(exc_count_u64, 8, st)) return 1;
    const int nwp4 = nwp / 4, lanes_x = nwp4 < 256 ? nwp4 : 256, pzb = 256 / lanes_x;
    dim3 grid((nwp4 + lanes_x - 1) / lanes_x, (v.Hp + FY - 1) / FY, (v.Zp + pzb - 1) / pzb);
    k_field_sign<true><<<grid, 256, 0, st>>>(v, (uint32_t*)sign_bits, nwp, lanes_x, pzb, FY, (unsigned long long*)n_exact_u64,
                                             (unsigned long long*)exc_list_u64, exc_cap, (unsigned long long*)exc_count_u64);
    k_field_sign_fix<<<T3D_NUM_SMS, 128, 0, st>>>(v, (uint32_t*)sign_bits, nwp, (const unsigned long long*)exc_list_u64, exc_cap,
                                                  (const unsigned long long*)exc_count_u64);
    T3D_CHECK_LAUNCH("t3d_field_sign_lean");
    t3d_count_launches(2);
    return 0;
}

// rowcnt: 4 * Zs*Hs uint32 (x-edge, y-edge, z-edge vertex counts and triangle counts per voxel row)
// float32 field of the whole padded grid (test / debugging aid: lets the parity tests compare the field
// itself with scipy bit for bit)
__global__ void __launch_bounds__(256) k_field_dense(OccView v, float* __restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)v.Zp * v.Hp * v.Wp;
    if (i >= total) return;
    const int x = (int)(i % v.Wp);
    const int64_t r = i / v.Wp;
    out[i] = field_value(v, (int)(r / v.Hp), (int)(r % v.Hp), x);
}

extern "C" int t3d_field_dense(const void* occ_bits, int Z, int H, int W, int pad, int gaussian, const double* weights3,
                               void* out_f32, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_field_dense: empty volume"); return 2; }
    const OccView v = t3d_make_view(occ_bits, Z, H, W, pad, gaussian, weights3);
    const int64_t total = (int64_t)v.Zp * v.Hp * v.Wp;
    k_field_dense<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(v, (float*)out_f32);
    T3D_CHECK_LAUNCH("t3d_field_dense");
    t3d_count_launches(1);
    return 0;
}

// cube-case volume (Zs-1, Hs-1, Ws-1) uint8 from a sign volume (parity tests: bit-exact cube cases)
__global__ void __launch_bounds__(256) k_cube_cases(const uint32_t* __restrict__ sign, int Zs, int Hs, int Ws, int nws,
                                                    uint8_t* __restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)(Zs - 1) * (Hs - 1) * (Ws - 1);
    if (i >= total) return;
    const int x = (int)(i % (Ws - 1));
    const int64_t r = i / (Ws - 1);
    const int y = (int)(r % (Hs - 1)), z = (int)(r / (Hs - 1));
    auto sb = [&](int zz, int yy, int xx) -> int {
        return (int)((sign[((int64_t)zz * Hs + yy) * nws + (xx >> 5)] >> (xx & 31)) & 1u);
    };
    out[i] = (uint8_t)(sb(z, y, x) | (sb(z, y, x + 1) << 1) | (sb(z, y + 1, x + 1) << 2) | (sb(z, y + 1, x) << 3) |
                       (sb(z + 1, y, x) << 4) | (sb(z + 1, y, x + 1) << 5) | (sb(z + 1, y + 1, x + 1) << 6) |
                       (sb(z + 1, y + 1, x) << 7));
}

extern "C" int t3d_cube_cases(const void* sign_bits, int Zs, int Hs, int Ws, void* out_u8, void* stream)
{
    if (Zs < 2 || Hs < 2 || Ws < 2) { t3d_set_error("t3d_cube_cases: volume smaller than 2x2x2"); return 2; }
    const int64_t total = (int64_t)(Zs - 1) * (Hs - 1) * (Ws - 1);
    k_cube_cases<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const uint32_t*)sign_bits, Zs, Hs, Ws,
                                                                                  t3d_wpr(Ws), (uint8_t*)out_u8);
    T3D_CHECK_LAUNCH("t3d_cube_cases");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// canonical mesh (_ensure_manifold_mesh): lexicographic sort of float32 rows (z, y, x), merge exact
// duplicates, remap faces, drop faces with a repeated index (order otherwise preserved).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t float_key(float f)
{
    uint32_t u = __float_as_uint(f);
    if (u == 0x80000000u) u = 0u;  // -0.0 == +0.0
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(256) k_make_keys(const float* __restrict__ verts, int64_t V, int col, const uint32_t* __restrict__ perm,
                                                   uint32_t* __restrict__ keys, uint32_t* __restrict__ iota)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const uint32_t src = perm ? perm[i] : (uint32_t)i;
    keys[i] = float_key(verts[3 * (int64_t)src + col]);
    if (iota) iota[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(256) k_unique_heads(const float* __restrict__ verts, const uint32_t* __restrict__ perm, int64_t V,
                                                      uint32_t* __restrict__ head)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    uint32_t h = 1;
    if (i > 0) {
        const float* a = verts + 3 * (int64_t)perm[i];
        const float* b = verts + 3 * (int64_t)perm[i - 1];
        h = (float_key(a[0]) != float_key(b[0]) || float_key(a[1]) != float_key(b[1]) || float_key(a[2]) != float_key(b[2])) ? 1u : 0u;
    }
    head[i] = h;
}

__global__ void __launch_bounds__(256) k_scatter_unique(const float* __restrict__ verts, const uint32_t* __restrict__ perm,
                                                        const uint32_t* __restrict__ head, const uint32_t* __restrict__ pos,
                                                        int64_t V_cap, float* __restrict__ out_verts, uint32_t* __restrict__ newid,
                                                        const unsigned long long* __restrict__ V_dev = nullptr)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dev_n(V_cap, V_dev)) return;
    // pos = exclusive scan of head => unique index of element i is pos[i] + head[i] - 1
    const uint32_t u = pos[i] + head[i] - 1u;
    const uint32_t src = perm[i];
    newid[src] = u;
    if (head[i]) {
        const float* a = verts + 3 * (int64_t)src;
        float* o = out_verts + 3 * (int64_t)u;
        o[0] = a[0]; o[1] = a[1]; o[2] = a[2];
    }
}

__global__ void __launch_bounds__(256) k_face_valid(const int32_t* __restrict__ faces, int64_t F_cap, const uint32_t* __restrict__ newid,
                                                    uint32_t* __restrict__ valid, const unsigned long long* __restrict__ F_dev = nullptr)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dev_n(F_cap, F_dev)) return;
    const uint32_t a = newid[faces[3 * i]], b = newid[faces[3 * i + 1]], c = newid[faces[3 * i + 2]];
    valid[i] = (a != b && b != c && a != c) ? 1u : 0u;
}

__global__ void __launch_bounds__(256) k_face_compact(const int32_t* __restrict__ faces, int64_t F_cap, const uint32_t* __restrict__ newid,
                                                      const uint32_t* __restrict__ valid, const uint32_t* __restrict__ pos,
                                                      long long* __restrict__ out64, int32_t* __restrict__ out32,
                                                      const unsigned long long* __restrict__ F_dev = nullptr)
{
    const int64_t F = dev_n(F_cap, F_dev);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < F; i += (int64_t)gridDim.x * blockDim.x) {
        if (!valid[i]) continue;
        const uint32_t a = newid[faces[3 * i]], b = newid[faces[3 * i + 1]], c = newid[faces[3 * i + 2]];
        const int64_t o = 3 * (int64_t)pos[i];
        if (out64) { out64[o] = a; out64[o + 1] = b; out64[o + 2] = c; }
        if (out32) { out32[o] = (int32_t)a; out32[o + 1] = (int32_t)b; out32[o + 2] = (int32_t)c; }
    }
}

// faces through newid straight into the output (degenerate faces are rare): counts the invalid ones; the compaction
// below runs only when there are any.  meta[0] = number of invalid faces.
__global__ void __launch_bounds__(256) k_face_remap(const int32_t* __restrict__ faces, int64_t F_cap, const uint32_t* __restrict__ newid,
                                                    uint32_t* __restrict__ valid, long long* __restrict__ out64, int32_t* __restrict__ out32,
                                                    unsigned long long* __restrict__ n_invalid, const unsigned long long* __restrict__ F_dev)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t F = dev_n(F_cap, F_dev);
    bool bad = false;
    if (i < F) {
        const uint32_t a = newid[faces[3 * i]], b = newid[faces[3 * i + 1]], c = newid[faces[3 * i + 2]];
        bad = !(a != b && b != c && a != c);
        valid[i] = bad ? 0u : 1u;
        if (out64) { out64[3 * i] = a; out64[3 * i + 1] = b; out64[3 * i + 2] = c; }
        if (out32) { out32[3 * i] = (int32_t)a; out32[3 * i + 1] = (int32_t)b; out32[3 * i + 2] = (int32_t)c; }
    }
    const uint32_t nb = __popc(__ballot_sync(0xffffffffu, bad));
    if (lane_id() == 0 && nb) atomicAdd(n_invalid, (unsigned long long)nb);
}

// after k_face_remap: F' = F - invalid; the scan/compaction that follow see n = F only if something has to move
__global__ void k_face_plan(const unsigned long long* __restrict__ n_invalid, int64_t F_cap, const unsigned long long* __restrict__ F_dev,
                            unsigned long long* __restrict__ n_to_compact, unsigned long long* __restrict__ f_out)
{
    const unsigned long long F = (unsigned long long)dev_n(F_cap, F_dev);
    *n_to_compact = (*n_invalid) ? F : 0ull;
    *f_out = F - *n_invalid;
}

static size_t sort_temp_bytes(int64_t V)
{
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)V);
    return bytes;
}

static inline int64_t align256(int64_t x) { return (x + 255) & ~(int64_t)255; }

extern "C" int64_t t3d_canonicalize_workspace_bytes(int64_t V, int64_t F)
{
    const int64_t n = V > F ? V : F;
    int64_t b = 0;
    b += 4 * align256(4 * V);                       // keys_a, keys_b, perm_a, perm_b
    b += 2 * align256(4 * n);                       // flags, positions (vertices then faces)
    b += align256(4 * V);                           // newid
    b += align256((int64_t)sort_temp_bytes(V > 0 ? V : 1));
    b += align256(t3d_scan_workspace_bytes(n, 1));
    b += 256;                                       // totals
    return b;
}

// verts_in (V,3) f32, faces_in (F,3) i32  ->  verts_out (<=V,3) f32 sorted+unique, faces_out (<=F,3) int64 and/or int32
// (either pointer may be null).  counts_u64[0] = V', counts_u64[1] = F' (device).
extern "C" int t3d_mesh_canonicalize(const void* verts_in, int64_t V, const void* faces_in, int64_t F, void* verts_out,
                                     void* faces_out_i64, void* faces_out_i32, void* counts_u64, void* workspace, void* stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (V <= 0 || V > 0x7fffffff || F < 0) { t3d_set_error("t3d_mesh_canonicalize: bad sizes"); return 2; }
    const int64_t n = V > F ? V : F;
    char* ws = (char*)workspace;
    uint32_t* keys_a = (uint32_t*)ws; ws += align256(4 * V);
    uint32_t* keys_b = (uint32_t*)ws; ws += align256(4 * V);
    uint32_t* perm_a = (uint32_t*)ws; ws += align256(4 * V);
    uint32_t* perm_b = (uint32_t*)ws; ws += align256(4 * V);
    uint32_t* flags = (uint32_t*)ws; ws += align256(4 * n);
    uint32_t* pos = (uint32_t*)ws; ws += align256(4 * n);
    uint32_t* newid = (uint32_t*)ws; ws += align256(4 * V);
    size_t temp_bytes = sort_temp_bytes(V);
    void* temp = ws; ws += align256((int64_t)temp_bytes);
    void* scan_ws = ws; ws += align256(t3d_scan_workspace_bytes(n, 1));
    unsigned long long* totals = (unsigned long long*)ws;
    unsigned long long* counts = (unsigned long long*)counts_u64;
    const unsigned gv = (unsigned)((V + 255) / 256);
    const float* vin = (const float*)verts_in;

    // stable LSD over the three columns: x (least significant), y, z
    uint32_t *pin = nullptr, *pout = perm_a, *pspare = perm_b;
    for (int pass = 0; pass < 3; ++pass) {
        const int col = 2 - pass;
        // keys of the current order; first pass also creates the identity permutation (in pspare)
        k_make_keys<<<gv, 256, 0, st>>>(vin, V, col, pin, keys_a, pass == 0 ? pspare : nullptr);
        const uint32_t* vals_in = (pass == 0) ? pspare : pin;
        T3D_CUDA(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, (const uint32_t*)keys_a, keys_b, vals_in, pout, (int)V, 0, 32, st));
        // rotate buffers: pout becomes the current permutation
        uint32_t* old_in = pin;
        pin = pout;
        pout = (pass == 0) ? pspare : old_in;
        if (pass == 0) pspare = nullptr;
    }
    const uint32_t* perm = pin;
    k_unique_heads<<<gv, 256, 0, st>>>(vin, perm, V, flags);
    if (t3d_exclusive_scan_u32_dev(flags, pos, V, V, 1, 0, 0, nullptr, totals, scan_ws, stream)) return 1;
    T3D_CUDA(cudaMemcpyAsync(counts, totals, 8, cudaMemcpyDeviceToDevice, st));
    k_scatter_unique<<<gv, 256, 0, st>>>(vin, perm, flags, pos, V, (float*)verts_out, newid);
    if (F > 0) {
        const unsigned gf = (unsigned)((F + 255) / 256);
        k_face_valid<<<gf, 256, 0, st>>>((const int32_t*)faces_in, F, newid, flags);
        if (t3d_exclusive_scan_u32_dev(flags, pos, F, F, 1, 0, 0, nullptr, totals, scan_ws, stream)) return 1;
        T3D_CUDA(cudaMemcpyAsync(counts + 1, totals, 8, cudaMemcpyDeviceToDevice, st));
        k_face_compact<<<gf, 256, 0, st>>>((const int32_t*)faces_in, F, newid, flags, pos, (long long*)faces_out_i64,
                                           (int32_t*)faces_out_i32);
    } else {
        T3D_CUDA(cudaMemsetAsync(counts + 1, 0, 8, st));
    }
    T3D_CHECK_LAUNCH("t3d_mesh_canonicalize");
    t3d_count_launches(F > 0 ? 7 : 5);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// fast canonical mesh for meshes emitted by t3d_mc_emit_dev.  The raw vertex order is [x-edge | y-edge | z-edge] blocks,
// each in raster order of the owning voxel, so among vertices with equal (z, y) float keys the x keys are already
// ascending (equal (z,y) keys across blocks would need a vertex coordinate to round onto a grid plane).  One STABLE
// radix sort on the 64-bit key (z key << 32 | y key) therefore yields np.unique's lexicographic order.  The result is
// verified on the device: counts_u64[2] != 0 means an adjacent pair was out of order and the caller must fall back
// to t3d_mesh_canonicalize (three-key sort, valid for any input).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_make_keys64(const float* __restrict__ verts, int64_t V_cap, const unsigned long long* __restrict__ V_dev,
                                                     unsigned long long* __restrict__ keys, uint32_t* __restrict__ iota)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V_cap) return;
    // slots beyond the true vertex count sort to the end
    keys[i] = (i < dev_n(V_cap, V_dev)) ? (((unsigned long long)float_key(verts[3 * i]) << 32) | float_key(verts[3 * i + 1]))
                                        : 0xffffffffffffffffull;
    iota[i] = (uint32_t)i;
}

// head flags of the sorted sequence + strict lexicographic order check (z, y, x)
__global__ void __launch_bounds__(256) k_heads_checked(const float* __restrict__ verts, const uint32_t* __restrict__ perm, int64_t V_cap,
                                                       const unsigned long long* __restrict__ V_dev, uint32_t* __restrict__ head,
                                                       unsigned long long* __restrict__ bad)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dev_n(V_cap, V_dev)) return;
    uint32_t h = 1;
    if (i > 0) {
        const float* a = verts + 3 * (int64_t)perm[i];
        const float* b = verts + 3 * (int64_t)perm[i - 1];
        const uint32_t az = float_key(a[0]), ay = float_key(a[1]), ax = float_key(a[2]);
        const uint32_t bz = float_key(b[0]), by = float_key(b[1]), bx = float_key(b[2]);
        h = (az != bz || ay != by || ax != bx) ? 1u : 0u;
        const bool lt = (az < bz) || (az == bz && (ay < by || (ay == by && ax < bx)));  // current < previous
        if (lt) atomicOr(bad, 1ull);
    }
    head[i] = h;
}

static size_t sort64_temp_bytes(int64_t V)
{
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)V);
    return bytes;
}

extern "C" int64_t t3d_canonicalize_fast_workspace_bytes(int64_t V, int64_t F)
{
    const int64_t n = V > F ? V : F;
    int64_t b = 0;
    b += 2 * align256(8 * V);                       // keys in/out
    b += 2 * align256(4 * V);                       // iota, perm
    b += 2 * align256(4 * n);                       // flags, positions
    b += align256(4 * V);                           // newid
    b += align256((int64_t)sort64_temp_bytes(V > 0 ? V : 1));
    b += align256(t3d_scan_workspace_bytes(n, 1));
    b += 256;
    return b;
}

// np.unique on the sorted sequence in ONE pass: head flags + strict order check, exclusive scan of the heads (decoupled
// look-back, same tile protocol as k_scan_lookback), scatter of the unique vertices and of the old -> new id map.
// n_unique_out receives V'.
#define UQ_ITEMS 4   // fewer items per thread than the plain scan: three floats + an index per item live in registers
#define UQ_TILE (SC_THREADS * UQ_ITEMS)
__global__ void __launch_bounds__(SC_THREADS) k_unique_fused(const float* __restrict__ verts, const uint32_t* __restrict__ perm, int64_t V_cap,
                                                             const unsigned long long* __restrict__ V_dev, float* __restrict__ out_verts,
                                                             uint32_t* __restrict__ newid, unsigned long long* __restrict__ desc, int n_tiles,
                                                             unsigned int* __restrict__ ticket, unsigned long long* __restrict__ bad,
                                                             unsigned long long* __restrict__ n_unique_out,
                                                             const unsigned long long* __restrict__ skip_unless)
{
    // striped arrangement: element e = k * SC_THREADS + tid of the tile, so a warp always touches 32 consecutive sorted
    // positions (coalesced perm reads, neighbouring vertices); keys go through shared memory for the neighbour compare
    if (skip_unless && *skip_unless == 0) return;      // the optimistic pass (k_unique_optimistic) already wrote everything
    const int64_t n = dev_n(V_cap, V_dev);
    volatile unsigned long long* d = desc;
    __shared__ int s_tile;
    __shared__ uint32_t s_kz[UQ_TILE + 1], s_ky[UQ_TILE + 1], s_kx[UQ_TILE + 1];   // [0] = last element of the previous tile
    __shared__ uint32_t s_part[UQ_ITEMS * (SC_THREADS / 32)];                     // heads per (k, warp), then their exclusive scan
    __shared__ unsigned long long s_prefix;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int tile = s_tile;
    const int64_t need = (n + UQ_TILE - 1) / UQ_TILE;
    n_tiles = (int)(need < 1 ? 1 : (need < n_tiles ? need : n_tiles));
    if (tile >= n_tiles) return;
    const int64_t base = (int64_t)tile * UQ_TILE;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t src[UQ_ITEMS];
    float vz[UQ_ITEMS], vy[UQ_ITEMS], vx[UQ_ITEMS];
#pragma unroll
    for (int k = 0; k < UQ_ITEMS; ++k) {
        const int e = k * SC_THREADS + tid;
        if (base + e < n) {
            src[k] = perm[base + e];
            const float* a = verts + 3 * (int64_t)src[k];
            vz[k] = a[0]; vy[k] = a[1]; vx[k] = a[2];
            s_kz[e + 1] = float_key(vz[k]); s_ky[e + 1] = float_key(vy[k]); s_kx[e + 1] = float_key(vx[k]);
        }
    }
    if (tid == 0 && base > 0) {
        const float* b = verts + 3 * (int64_t)perm[base - 1];
        s_kz[0] = float_key(b[0]); s_ky[0] = float_key(b[1]); s_kx[0] = float_key(b[2]);
    }
    __syncthreads();
    uint32_t ball[UQ_ITEMS];
    uint32_t myhead = 0;
    bool out_of_order = false;
#pragma unroll
    for (int k = 0; k < UQ_ITEMS; ++k) {
        const int e = k * SC_THREADS + tid;
        bool h = false;
        if (base + e < n) {
            h = true;
            if (base + e > 0) {
                const uint32_t az = s_kz[e + 1], ay = s_ky[e + 1], ax = s_kx[e + 1], pz = s_kz[e], py = s_ky[e], px = s_kx[e];
                h = (az != pz || ay != py || ax != px);
                out_of_order |= (az < pz) || (az == pz && (ay < py || (ay == py && ax < px)));
            }
        }
        ball[k] = __ballot_sync(0xffffffffu, h);
        myhead |= (h ? 1u : 0u) << k;
        if (lane == 0) s_part[k * (SC_THREADS / 32) + warp] = __popc(ball[k]);
    }
    if (out_of_order) atomicOr(bad, 1ull);
    __syncthreads();
    if (tid < 32) {
        // exclusive scan of the partial counts (UQ_ITEMS * 8 of them, spread over the lanes), tile aggregate, look-back
        constexpr int PER_LANE = UQ_ITEMS * (SC_THREADS / 32) / 32;
        static_assert(PER_LANE >= 1 && PER_LANE * 32 == UQ_ITEMS * (SC_THREADS / 32), "partials must spread evenly over a warp");
        uint32_t pv[PER_LANE], psum = 0;
#pragma unroll
        for (int t = 0; t < PER_LANE; ++t) { pv[t] = s_part[PER_LANE * lane + t]; psum += pv[t]; }
        const uint32_t incl = warp_incl_scan(psum);
        const uint32_t agg = __shfl_sync(0xffffffffu, incl, 31);
        uint32_t runp = incl - psum;
#pragma unroll
        for (int t = 0; t < PER_LANE; ++t) { s_part[PER_LANE * lane + t] = runp; runp += pv[t]; }
        unsigned long long prefix = 0;
        if (tile == 0) {
            if (tid == 0) { d[0] = SC_FLAG_P | (unsigned long long)agg; }
        } else {
            if (tid == 0) { d[tile] = SC_FLAG_A | (unsigned long long)agg; }
            int idx = tile - 1 - tid;
            while (true) {
                unsigned long long w = (idx >= 0) ? d[idx] : SC_FLAG_P;
                while (__any_sync(0xffffffffu, (w >> 62) == 0)) {
                    if ((w >> 62) == 0) w = (idx >= 0) ? d[idx] : SC_FLAG_P;
                }
                const uint32_t is_p = __ballot_sync(0xffffffffu, (w >> 62) == 2);
                const int first_p = is_p ? (__ffs(is_p) - 1) : 32;
                unsigned long long val = (tid <= first_p) ? (w & SC_VALUE_MASK) : 0ull;
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) val += __shfl_xor_sync(0xffffffffu, val, off);
                prefix += val;
                if (is_p) break;
                idx -= 32;
            }
            if (tid == 0) { d[tile] = SC_FLAG_P | ((prefix + agg) & SC_VALUE_MASK); }
        }
        if (tid == 0) {
            s_prefix = prefix;
            if (tile == n_tiles - 1) *n_unique_out = prefix + agg;
        }
    }
    __syncthreads();
    const uint32_t tile_prefix = (uint32_t)s_prefix;
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int k = 0; k < UQ_ITEMS; ++k) {
        const int e = k * SC_THREADS + tid;
        if (base + e < n) {
            const uint32_t h = (myhead >> k) & 1u;
            // unique index = (heads up to and including this element) - 1
            const uint32_t u = tile_prefix + s_part[k * (SC_THREADS / 32) + warp] + __popc(ball[k] & lt) + h - 1u;
            newid[src[k]] = u;
            if (h) {
                float* o = out_verts + 3 * (int64_t)u;
                o[0] = vz[k]; o[1] = vy[k]; o[2] = vx[k];
            }
        }
    }
}

// The same np.unique under the assumption that NO two vertices coincide (the rule on a marching-cubes mesh: duplicates need a
// field value of exactly 0.5 at a grid point): then the unique index of a vertex is its sorted position and there is nothing
// to scan -- one streaming pass: gather the vertex, write it and its new id, compare it with its predecessor.  Any equal pair
// raises *dup and the exact kernel above (enqueued right behind, returning at once while *dup == 0) redoes the step.
__global__ void __launch_bounds__(256) k_unique_optimistic(const float* __restrict__ verts, const uint32_t* __restrict__ perm, int64_t V_cap,
                                                           const unsigned long long* __restrict__ V_dev, float* __restrict__ out_verts,
                                                           uint32_t* __restrict__ newid, unsigned long long* __restrict__ bad,
                                                           unsigned long long* __restrict__ n_unique_out, unsigned long long* __restrict__ dup)
{
    const int64_t n = dev_n(V_cap, V_dev);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *n_unique_out = (unsigned long long)n;
    const bool ok = i < n;
    uint32_t src = 0, kz = 0, ky = 0, kx = 0;
    if (ok) {
        src = perm[i];
        const float* a = verts + 3 * (int64_t)src;
        const float z = a[0], y = a[1], x = a[2];
        float* o = out_verts + 3 * i;
        o[0] = z; o[1] = y; o[2] = x;
        newid[src] = (uint32_t)i;
        kz = float_key(z); ky = float_key(y); kx = float_key(x);
    }
    // predecessor: the lane below, or (lane 0) one more gather
    uint32_t pz = __shfl_up_sync(0xffffffffu, kz, 1), py = __shfl_up_sync(0xffffffffu, ky, 1), px = __shfl_up_sync(0xffffffffu, kx, 1);
    if ((threadIdx.x & 31) == 0 && ok && i > 0) {
        const float* b = verts + 3 * (int64_t)perm[i - 1];
        pz = float_key(b[0]); py = float_key(b[1]); px = float_key(b[2]);
    }
    if (ok && i > 0) {
        if (kz == pz && ky == py && kx == px) atomicOr(dup, 1ull);
        else if ((kz < pz) || (kz == pz && (ky < py || (ky == py && kx < px)))) atomicOr(bad, 1ull);
    }
}

// everything after the sorted permutation is known: head flags + order check, unique scatter, face remap
// The single-enqueue pipeline emits the faces on its side stream while the vertices are being ordered here: it registers
// the event "faces emitted" and the tail waits for it right before the first kernel that reads the faces (the kernels before
// that -- layer sort, positions, unique -- only need the vertices).  One-shot: consumed by the next canonical_tail of this thread.
static thread_local cudaEvent_t g_faces_ready = nullptr;
void t3d_canon_faces_ready_event(cudaEvent_t e) { g_faces_ready = e; }
// true if the registered event was not consumed (the caller then waits for it itself); clears it
bool t3d_canon_faces_ready_pending() { const bool p = g_faces_ready != nullptr; g_faces_ready = nullptr; return p; }

static int canonical_tail(const float* vin, const uint32_t* perm, int64_t V, const unsigned long long* V_dev, const void* faces_in,
                          int64_t F, const unsigned long long* F_dev, void* verts_out, void* faces_out_i64, void* faces_out_i32,
                          unsigned long long* counts, uint32_t* flags, uint32_t* pos, uint32_t* newid, void* scan_ws,
                          void* scan_ws_faces, unsigned long long* totals, cudaStream_t st)
{
    void* stream = (void*)st;
    {
        // workspace as in t3d_exclusive_scan_u32_dev: [tile descriptors][ticket], zeroed per use
        const int64_t nb = (V + UQ_TILE - 1) / UQ_TILE;
        const size_t desc_bytes = (size_t)nb * 8;
        if (t3d_zero_async(scan_ws, desc_bytes + 64, st)) return 1;
        unsigned long long* dup = totals + 8;
        if (t3d_zero_async(dup, 8, st)) return 1;
        k_unique_optimistic<<<(unsigned)((V + 255) / 256), 256, 0, st>>>(vin, perm, V, V_dev, (float*)verts_out, newid, counts + 2, counts, dup);
        t3d_count_launches(1);
        k_unique_fused<<<(unsigned)nb, SC_THREADS, 0, st>>>(vin, perm, V, V_dev, (float*)verts_out, newid, (unsigned long long*)scan_ws,
                                                           (int)nb, (unsigned int*)((char*)scan_ws + desc_bytes), counts + 2, counts, dup);
    }
    if (g_faces_ready) {
        T3D_CUDA(cudaStreamWaitEvent(st, g_faces_ready, 0));
        g_faces_ready = nullptr;
    }
    if (F > 0) {
        // totals[1] = invalid faces, totals[2] = faces the compaction has to look at (0 when nothing is invalid)
        const unsigned gf = (unsigned)((F + 255) / 256);
        if (t3d_zero_async(totals + 1, 16, st)) return 1;
        k_face_remap<<<gf, 256, 0, st>>>((const int32_t*)faces_in, F, newid, flags, (long long*)faces_out_i64, (int32_t*)faces_out_i32,
                                         totals + 1, F_dev);
        k_face_plan<<<1, 1, 0, st>>>(totals + 1, F, F_dev, totals + 2, counts + 1);
        if (t3d_exclusive_scan_u32_dev(flags, pos, F, F, 1, 0, 0, totals + 2, totals + 3, scan_ws_faces, stream)) return 1;
        const unsigned gc = gf < (unsigned)(T3D_NUM_SMS * 8) ? gf : (unsigned)(T3D_NUM_SMS * 8);
        k_face_compact<<<gc, 256, 0, st>>>((const int32_t*)faces_in, F, newid, flags, pos, (long long*)faces_out_i64,
                                           (int32_t*)faces_out_i32, totals + 2);
    } else {
        T3D_CUDA(cudaMemsetAsync(counts + 1, 0, 8, st));
    }
    return 0;
}

// same outputs as t3d_mesh_canonicalize; counts_u64[0] = V', [1] = F', [2] = 0 if the fast ordering was verified.
// V_dev_u64 / F_dev_u64 (optional, device uint64): true sizes when V / F are only capacities.
extern "C" int t3d_mesh_canonicalize_fast_dev(const void* verts_in, int64_t V, const void* V_dev_u64, const void* faces_in, int64_t F,
                                              const void* F_dev_u64, void* verts_out, void* faces_out_i64, void* faces_out_i32,
                                              void* counts_u64, void* workspace, void* stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (V <= 0 || V > 0x7fffffff || F < 0) { t3d_set_error("t3d_mesh_canonicalize_fast_dev: bad sizes"); return 2; }
    const unsigned long long* V_dev = (const unsigned long long*)V_dev_u64;
    const unsigned long long* F_dev = (const unsigned long long*)F_dev_u64;
    const int64_t n = V > F ? V : F;
    char* ws = (char*)workspace;
    unsigned long long* keys_a = (unsigned long long*)ws; ws += align256(8 * V);
    unsigned long long* keys_b = (unsigned long long*)ws; ws += align256(8 * V);
    uint32_t* iota = (uint32_t*)ws; ws += align256(4 * V);
    uint32_t* perm = (uint32_t*)ws; ws += align256(4 * V);
    uint32_t* flags = (uint32_t*)ws; ws += align256(4 * n);
    uint32_t* pos = (uint32_t*)ws; ws += align256(4 * n);
    uint32_t* newid = (uint32_t*)ws; ws += align256(4 * V);
    size_t temp_bytes = sort64_temp_bytes(V);
    void* temp = ws; ws += align256((int64_t)temp_bytes);
    void* scan_ws = ws; ws += align256(t3d_scan_workspace_bytes(n, 1));
    unsigned long long* totals = (unsigned long long*)ws;
    unsigned long long* counts = (unsigned long long*)counts_u64;
    const unsigned gv = (unsigned)((V + 255) / 256);
    const float* vin = (const float*)verts_in;
    T3D_CUDA(cudaMemsetAsync(counts + 2, 0, 8, st));
    k_make_keys64<<<gv, 256, 0, st>>>(vin, V, V_dev, keys_a, iota);
    T3D_CUDA(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, (const unsigned long long*)keys_a, keys_b, (const uint32_t*)iota, perm,
                                             (int)V, 0, 64, st));
    if (canonical_tail(vin, perm, V, V_dev, faces_in, F, F_dev, verts_out, faces_out_i64, faces_out_i32, counts, flags, pos, newid,
                       scan_ws, scan_ws, totals, st)) return 1;
    T3D_CHECK_LAUNCH("t3d_mesh_canonicalize_fast_dev");
    t3d_count_launches(F > 0 ? 5 : 3);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// structured canonical order for meshes emitted by t3d_mc_emit_dev (vertex keys available).
//
// Raw order = [x-edge | y-edge | z-edge] blocks, each in raster order of the owning grid point (zc, yc, xc).  A vertex
// has one fractional coordinate; give every coordinate a level (2c on a grid line, 2c+1 strictly inside cell c).
// np.unique's order (z, y, x floats) is the order by (z level, z float, y level, y float, x level) as long as the
// coordinate transform is monotone, which fixes almost everything without sorting:
//   * x-edge vertices are already in canonical order among themselves;
//   * y-edge vertices only need ordering inside their (plane, row gap) segment (a handful of vertices): ranked by counting;
//   * z-edge vertices need ONE stable sort by (layer, z float) -- a third of the vertices, one segment per layer (below);
//   * the final position of a vertex = its rank in its own block + how many vertices of the other two blocks precede it;
//     those counts are per-row / per-plane prefix counts, read from the scanned per-active-word counts of the emit pass.
// Exception G0: with the z map's clamp (surface_extractor.py:100-103) every vertex at or below un-padded plane 0 gets
// z = 0, so the vertices of the closing cap under slice 0 interleave with those of plane 0 by (y, x): that group (empty
// unless the object touches slice 0) is ordered by one small generic (y,x)-key sort of its own (cap_g0 entries).
// As with the fast path the result is verified on the device (counts[2]): rounding that breaks the level model, a
// group larger than cap_g0 or more z-edge vertices than cap_z leave counts[2] != 0 and the caller falls back.
// ------------------------------------------------------------------------------------------------
struct CanonS {
    const float* verts;
    const unsigned long long* vkeys;
    const unsigned long long* sizes;   // {n_active, n_x, n_y, n_z, n_t}
    uint32_t cap_verts, cap_z, cap_g0;
    int Zs, Hs;                        // planes / rows per plane of the (local, padded) sign volume
    int ncr;                           // bitmap chunks per row (t3d_mc_flags)
    const uint32_t* chunkbase;         // active words before each chunk
    const uint32_t* aw_base;           // 4 arrays (x, y, z vertices, triangles before each active word), `stride` apart
    uint32_t stride;
    int g_plane;                       // local plane index of un-padded plane 0 (= shift - z_offset); < 0: no clamp group here
    int z_offset; float shift;         // as in t3d_mc_vertices_dev: global plane of local plane 0, un-pad shift
    const double* cum; const double* adj; int n_cum;
    int zkey_bits;                     // 32: absolute z keys; less: key relative to the layer's lower plane, that many bits
    unsigned long long* zkeys;
    uint32_t* zval;
    const uint32_t* zperm;             // z block sorted by (layer, z float)
    unsigned long long* gkeys;
    uint32_t* gval;
    const uint32_t* gperm;             // clamp group sorted by (y, x)
    uint32_t* perm;                    // out: sorted position -> raw vertex id
    unsigned long long* n_g0_out;
};

// Number of x- / y- / z-edge vertices (AX = 0 / 1 / 2) owned by grid rows before `row` (rows in raster order, row =
// plane * Hs + y): the emit order is row-major over active words, so this is the scanned count at the first active word
// at or after the start of the row.
template <int AX>
__device__ __forceinline__ uint32_t before_row(const CanonS& c, int64_t row)
{
    const uint32_t na = (uint32_t)c.sizes[0];
    const uint32_t r = row >= (int64_t)c.Zs * c.Hs ? na : c.chunkbase[row * c.ncr];
    return r >= na ? (uint32_t)c.sizes[1 + AX] : c.aw_base[(int64_t)AX * c.stride + r];
}

// sizes of the clamp group per block (0 when the group needs no merging)
__device__ __forceinline__ void g0_sizes(const CanonS& c, uint32_t& gX, uint32_t& gY, uint32_t& gZ)
{
    gX = gY = gZ = 0;
    if (c.g_plane < 0) return;
    const int64_t r_plane = (int64_t)min(c.g_plane, c.Zs) * c.Hs, r_next = (int64_t)min(c.g_plane + 1, c.Zs) * c.Hs;
    const uint32_t z_below = before_row<2>(c, r_plane);                               // z-edge vertices in layers below plane g_plane
    const uint32_t xy_below = before_row<0>(c, r_plane) + before_row<1>(c, r_plane);  // x/y-edge vertices on planes below it
    if (z_below == 0 && xy_below == 0) return;                                        // only plane g_plane itself: the level model holds
    gX = before_row<0>(c, r_next); gY = before_row<1>(c, r_next); gZ = z_below;
}

// z coordinate the vertex transform gives to a vertex lying exactly on local plane k (same arithmetic as vertex_body)
__device__ __forceinline__ float plane_z(const CanonS& c, int k)
{
    float fz = __fsub_rn(__double2float_rn((double)(k + c.z_offset)), c.shift);
    if (c.n_cum > 0) {
        if (fz < 0.0f) fz = 0.0f;
        else if (fz >= (float)(c.n_cum - 1)) fz = __double2float_rn(c.cum[c.n_cum - 1]);
        else {
            const float fl = floorf(fz);
            const int lo = (int)fl;
            const float fr = __fsub_rn(fz, fl);
            fz = __double2float_rn(__dadd_rn(c.cum[lo], __dmul_rn((double)fr, c.adj[min(lo, c.n_cum - 2)])));
        }
    }
    return fz;
}

// ------------------------------------------------------------------------------------------------
// Ordering of the z-edge vertices without a library sort.  They are emitted in raster order of their owning grid point,
// so the vertices of one cube layer are contiguous: the (layer, z float) order is a SEGMENTED sort, one independent
// segment per layer, by the 32-bit (or narrower) layer-relative z key alone.  One CTA per layer runs a stable LSD radix
// sort (8-bit digits) over its segment, ping-ponging between two global buffers:
//   count   : every warp histograms its contiguous sub-range of the segment into its own 256 shared-memory bins;
//   offsets : digit-major exclusive scan over (digit, warp) -> where each warp's elements of each digit start;
//   scatter : every warp walks its sub-range in order, 32 elements per step; lanes with equal digits find each other with
//             match.any, rank themselves by lane order and advance the warp's offset for that digit -> stable.
// Layers are independent (no grid-wide synchronisation, no library), a typical layer (a few thousand vertices) costs a few
// microseconds and all layers run at once; keys are generated on the fly in pass 0.  The result is the permutation
// k_canon_positions expects (zperm[rank in the z block] = index in the z block).
// ------------------------------------------------------------------------------------------------
#define ZS_WARPS 16
#define ZS_THREADS (32 * ZS_WARPS)

__device__ __forceinline__ uint32_t canon_zkey(const CanonS& c, uint32_t i, uint32_t nx, uint32_t ny, uint32_t gZ)
{
    if (i < gZ) return 0u;     // clamp group: ordered elsewhere (k_gsort); keep raster order here
    const uint32_t raw = nx + ny + i;
    const int k = (int)(c.vkeys[raw] >> 42);
    uint32_t zk = float_key(c.verts[3 * (int64_t)raw]);
    if (c.zkey_bits < 32) {
        // relative to the layer's lower plane; anything outside the promised span saturates (and fails the order check)
        const uint32_t base = float_key(plane_z(c, k));
        zk = zk >= base ? zk - base : 0u;
        const uint32_t lim = (1u << c.zkey_bits) - 1u;
        zk = zk > lim ? lim : zk;
    }
    return zk;
}

// Stable LSD radix sort (8-bit digits) of ONE segment by ONE CTA of ZS_THREADS threads.  key_of(i) generates the key of
// element i in pass 0 (keys are materialised in keyA); out[rank] = value_of(i).  keyA/keyB/idxA/idxB: the segment's slices
// of the ping-pong buffers.  `passes` digits are sorted, least significant first.
template <int ZS_U, typename KeyT, typename KeyFn, typename ValFn>
__device__ __forceinline__ void cta_radix_sort_u(uint32_t n, int passes, KeyFn key_of, ValFn value_of, KeyT* keyA, KeyT* keyB, uint32_t* idxA,
                                               uint32_t* idxB, uint32_t* out)
{
    __shared__ uint32_t s_hist[ZS_WARPS][256];
    __shared__ uint32_t s_tot[256];
    __shared__ uint32_t s_carry[8];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    // contiguous sub-range of every warp, a multiple of 32 elements long
    const uint32_t per = (((n + ZS_WARPS - 1) / ZS_WARPS) + 31u) & ~31u;
    const uint32_t ws = min(n, (uint32_t)w * per), we = min(n, ws + per);
    const KeyT* kin = keyA; const uint32_t* iin = idxA;
    KeyT* kout = keyB; uint32_t* iout = idxB;
    for (int p = 0; p < passes; ++p) {
        const int shift = 8 * p;
        const bool first = p == 0, last = p == passes - 1;
        for (int i = tid; i < ZS_WARPS * 256; i += ZS_THREADS) (&s_hist[0][0])[i] = 0;
        __syncthreads();
        // ---- count (pass 0 also materialises the keys)
        // (ZS_U elements per lane are fetched before any is consumed: one exposed memory latency per ZS_U elements -- with one
        // element per trip both loops of a pass ran at one global-memory round trip per 32 elements per warp)
        for (uint32_t i0 = ws + lane; i0 < we; i0 += 32 * ZS_U) {
            KeyT kk[ZS_U];
#pragma unroll
            for (int u = 0; u < ZS_U; ++u) {
                const uint32_t i = i0 + 32 * u;
                if (i < we) { if (first) { kk[u] = key_of(i); keyA[i] = kk[u]; } else kk[u] = kin[i]; }
            }
#pragma unroll
            for (int u = 0; u < ZS_U; ++u)
                if (i0 + 32 * u < we) atomicAdd(&s_hist[w][(uint32_t)(kk[u] >> shift) & 255u], 1u);
        }
        __syncthreads();
        // ---- offsets: digit-major exclusive scan over (digit, warp)
        if (tid < 256) {
            uint32_t t = 0;
            for (int ww = 0; ww < ZS_WARPS; ++ww) t += s_hist[ww][tid];
            s_tot[tid] = t;
        }
        __syncthreads();
        if (tid < 256) {       // the first 8 warps: exclusive scan of the 256 digit totals (named barrier 1)
            const uint32_t v = s_tot[tid];
            const uint32_t incl = warp_incl_scan(v);
            if (lane == 31) s_carry[w] = incl;
            asm volatile("bar.sync 1, 256;" ::: "memory");
            uint32_t carry = 0;
            for (int ww = 0; ww < w; ++ww) carry += s_carry[ww];
            uint32_t run = carry + incl - v;
            for (int ww = 0; ww < ZS_WARPS; ++ww) { const uint32_t h = s_hist[ww][tid]; s_hist[ww][tid] = run; run += h; }
        }
        __syncthreads();
        // ---- stable scatter
        for (uint32_t c0 = ws; c0 < we; c0 += 32 * ZS_U) {
            KeyT kk[ZS_U];
            uint32_t ii[ZS_U];
#pragma unroll
            for (int u = 0; u < ZS_U; ++u) {
                const uint32_t i = c0 + 32 * u + lane;
                kk[u] = 0; ii[u] = 0;
                if (i < we) {
                    kk[u] = first ? keyA[i] : kin[i];
                    ii[u] = first ? value_of(i) : iin[i];
                }
            }
#pragma unroll
            for (int u = 0; u < ZS_U; ++u) {
                if (c0 + 32 * u >= we) break;                      // (warp-uniform)
                const uint32_t i = c0 + 32 * u + lane;
                const bool ok = i < we;
                const KeyT key = kk[u];
                const uint32_t idx = ii[u];
                const uint32_t d = ok ? ((uint32_t)(key >> shift) & 255u) : 0xffffffffu;
                const uint32_t peers = __match_any_sync(0xffffffffu, d);
                const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
                uint32_t pos = 0;
                if (ok) pos = s_hist[w][d] + rank;
                __syncwarp();
                if (ok && rank == 0) s_hist[w][d] += __popc(peers);      // the lowest lane of each digit group advances the offset
                __syncwarp();
                if (ok) {
                    if (last) out[pos] = idx;
                    else { kout[pos] = key; iout[pos] = idx; }
                }
            }
        }
        __syncthreads();
        // ping-pong (pass 0 read keyA / implicit values and wrote B)
        const KeyT* tk = kin; const uint32_t* ti = iin;
        kin = kout; iin = iout;
        kout = (KeyT*)tk; iout = (uint32_t*)ti;
    }
}

// ZS_U = elements per lane fetched before any is consumed.  Long segments want 8 (one exposed memory latency per 8 elements: the
// 30..60 thousand z-edge vertices of a 4096 x 4096 layer sort 1.3x faster), short ones 1 (a few thousand elements per layer at
// 1024 x 1024: the batched variant needs 64 registers instead of 40 and loses occupancy: 57 against 41 us).  Picked per launch
// from the average layer length.
template <int ZS_U>
__global__ void __launch_bounds__(ZS_THREADS) k_zsort_layers(CanonS c, uint32_t* __restrict__ keyA, uint32_t* __restrict__ keyB,
                                                            uint32_t* __restrict__ idxA, uint32_t* __restrict__ idxB,
                                                            uint32_t* __restrict__ zperm)
{
    const uint32_t nx = (uint32_t)c.sizes[1], ny = (uint32_t)c.sizes[2], nz = (uint32_t)c.sizes[3];
    if ((unsigned long long)nx + ny + nz > c.cap_verts || nz > c.cap_z) return;
    const int layer = blockIdx.x;
    uint32_t s = before_row<2>(c, (int64_t)layer * c.Hs), e = before_row<2>(c, (int64_t)(layer + 1) * c.Hs);
    if (e > nz) e = nz;
    if (s >= e) return;
    const uint32_t n = e - s;
    uint32_t gX, gY, gZ;
    g0_sizes(c, gX, gY, gZ);
    if (n == 1 || e <= gZ) {       // nothing to order (single vertex, or a layer of the clamp group)
        for (uint32_t i = s + threadIdx.x; i < e; i += ZS_THREADS) zperm[i] = i;
        return;
    }
    cta_radix_sort_u<ZS_U, uint32_t>(n, (c.zkey_bits + 7) / 8, [&](uint32_t i) { return canon_zkey(c, s + i, nx, ny, gZ); },
                                     [&](uint32_t i) { return s + i; }, keyA + s, keyB + s, idxA + s, idxB + s, zperm + s);
}

// the clamp group (vertices the z map clamps onto z = 0, see above): one CTA orders it by its 64-bit (y, x) key;
// gperm[rank] = raw vertex id.  A group larger than cap_g0 is left alone (the order check then fails, the caller retries).
__global__ void __launch_bounds__(ZS_THREADS) k_gsort(CanonS c, unsigned long long* __restrict__ keyA, unsigned long long* __restrict__ keyB,
                                                     uint32_t* __restrict__ idxA, uint32_t* __restrict__ idxB, uint32_t* __restrict__ gperm)
{
    const uint32_t nx = (uint32_t)c.sizes[1], ny = (uint32_t)c.sizes[2], nz = (uint32_t)c.sizes[3];
    if ((unsigned long long)nx + ny + nz > c.cap_verts) return;
    uint32_t gX, gY, gZ;
    g0_sizes(c, gX, gY, gZ);
    const uint32_t n = gX + gY + gZ;
    if (n == 0 || n > c.cap_g0) return;
    auto raw_of = [&](uint32_t t) -> uint32_t { return t < gX ? t : t < gX + gY ? nx + (t - gX) : nx + ny + (t - gX - gY); };
    if (n == 1) { if (threadIdx.x == 0) gperm[0] = raw_of(0); return; }
    cta_radix_sort_u<1, unsigned long long>(n, 8, [&](uint32_t t) {
        const float* v = c.verts + 3 * (int64_t)raw_of(t);
        return ((unsigned long long)float_key(v[1]) << 32) | float_key(v[2]);
    }, raw_of, keyA, keyB, idxA, idxB, gperm);
}

__global__ void __launch_bounds__(256) k_canon_positions(CanonS c)
{
    __shared__ uint32_t s_g[3];
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t nx = (uint32_t)c.sizes[1], ny = (uint32_t)c.sizes[2], nz = (uint32_t)c.sizes[3];
    const unsigned long long V64 = (unsigned long long)nx + ny + nz;
    if (V64 > c.cap_verts) return;
    if (threadIdx.x == 0) g0_sizes(c, s_g[0], s_g[1], s_g[2]);
    __syncthreads();
    if (i >= (uint32_t)V64) return;
    if (nz > c.cap_z) { c.perm[i] = i; return; }       // no z order available: identity, the order check will fail
    const uint32_t gX = s_g[0], gY = s_g[1], gZ = s_g[2];
    const uint32_t nG = gX + gY + gZ;
    if (i == 0 && c.n_g0_out) *c.n_g0_out = nG;
    // positions [0, nG): the clamp group in (y, x) order (block order when its sort was not provisioned)
    if (i < nG) c.perm[i] = (nG <= c.cap_g0) ? c.gperm[i] : (i < gX ? i : i < gX + gY ? nx + (i - gX) : nx + ny + (i - gX - gY));
    if (i < nx) {                                       // x-edge vertex: after the y-edge vertices of earlier rows and the z-edge
        if (i < gX) return;                             // vertices of lower layers
        const unsigned long long key = c.vkeys[i];
        const int k = (int)(key >> 42), j = (int)((key >> 22) & 0xfffffu);
        c.perm[i + before_row<1>(c, (int64_t)k * c.Hs + j) + before_row<2>(c, (int64_t)k * c.Hs)] = i;
    } else if (i < nx + ny) {                           // y-edge vertex: rank inside its (plane, row gap) segment by counting
        const uint32_t iy = i - nx;
        if (iy < gY) return;
        const unsigned long long key = c.vkeys[i];
        const int k = (int)(key >> 42), j = (int)((key >> 22) & 0xfffffu);
        const int64_t row = (int64_t)k * c.Hs + j;
        const uint32_t lo = before_row<1>(c, row), hi = before_row<1>(c, row + 1);
        const uint32_t mine = float_key(c.verts[3 * (int64_t)i + 1]);
        uint32_t r = 0;
        for (uint32_t e = lo; e < hi; ++e) {
            const uint32_t ke = float_key(c.verts[3 * (int64_t)(nx + e) + 1]);
            r += (ke < mine || (ke == mine && e < iy)) ? 1u : 0u;
        }
        c.perm[before_row<0>(c, row + 1) + lo + r + before_row<2>(c, (int64_t)k * c.Hs)] = i;
    } else {                                            // z block: this thread takes sorted rank R
        const uint32_t R = i - nx - ny;
        if (R < gZ) return;
        const uint32_t raw = nx + ny + c.zperm[R];
        const int64_t next_plane = ((int64_t)(c.vkeys[raw] >> 42) + 1) * c.Hs;
        c.perm[before_row<0>(c, next_plane) + before_row<1>(c, next_plane) + R] = raw;
    }
}

extern "C" int64_t t3d_canonicalize_structured_workspace_bytes(int64_t V, int64_t F, uint32_t cap_z, uint32_t cap_g0, int Zs)
{
    const int64_t n = V > F ? V : F;
    int64_t b = 0;
    b += 2 * align256(8 * (int64_t)cap_z) + 2 * align256(4 * (int64_t)cap_z);      // z keys in/out, values in/out
    b += 2 * align256(8 * (int64_t)cap_g0) + 2 * align256(4 * (int64_t)cap_g0);    // clamp group keys / values
    b += align256(4 * V);                                                          // perm
    b += 2 * align256(4 * n);                                                      // flags, positions
    b += align256(4 * V);                                                          // newid
    b += align256(4 * (int64_t)cap_g0 + 256);                                      // k_gsort's second value buffer
    b += 2 * align256(t3d_scan_workspace_bytes(n, 1)) + 256;   // zero tail: unique descriptors, face-scan workspace, totals
    return b;
}

// Where the raw -> canonical map of a canonicalisation lives in its workspace, for consumers enqueued after it (vertex normals):
// out4 = byte offsets of {newid (u32 per raw vertex: canonical slot), perm (u32 per sorted position: raw id), a u32 scratch of
// at least V entries that is dead once the call has finished (the face flags), the unique pass's "equal pair seen" flag
// (u64; -1: the generic path has none, every sorted run may merge)}.
// kind: 0 = t3d_mesh_canonicalize (V, F), 1 = the fast variants (V, F), 2 = the structured variant (V, F, cap_z, cap_g0, Zs).
extern "C" int t3d_canonical_map_offsets(int kind, int64_t V, int64_t F, uint32_t cap_z, uint32_t cap_g0, int Zs, int64_t* out4)
{
    if (V <= 0 || F < 0 || !out4 || kind < 0 || kind > 2) { t3d_set_error("t3d_canonical_map_offsets: bad arguments"); return 2; }
    const int64_t n = V > F ? V : F;
    int64_t o = 0;
    if (kind == 0) {
        out4[1] = 2 * align256(4 * V);                           // perm_a: the order after the three passes
        o = 4 * align256(4 * V);
        out4[2] = o; o += 2 * align256(4 * n);
        out4[0] = o;
        out4[3] = -1;
        return 0;
    }
    if (kind == 1) {
        o = 2 * align256(8 * V) + align256(4 * V);
        out4[1] = o; o += align256(4 * V);
        out4[2] = o; o += 2 * align256(4 * n);
        out4[0] = o; o += align256(4 * V);
        o += align256((int64_t)sort64_temp_bytes(V));
        o += align256(t3d_scan_workspace_bytes(n, 1));
    } else {
        o = 2 * align256(8 * (int64_t)cap_z) + 2 * align256(4 * (int64_t)cap_z) + 2 * align256(8 * (int64_t)cap_g0) +
            2 * align256(4 * (int64_t)cap_g0);
        out4[1] = o; o += align256(4 * V);
        out4[2] = o; o += 2 * align256(4 * n);
        out4[0] = o; o += align256(4 * V);
        o += align256(4 * (int64_t)cap_g0 + 256);
        o += 2 * align256(t3d_scan_workspace_bytes(n, 1));
    }
    out4[3] = o + 8 * 8;                                         // canonical_tail: dup = totals + 8
    (void)Zs;
    return 0;
}

// the part of the workspace the call needs zeroed on entry (it does so itself unless the range was zeroed up front and
// registered, see t3d_zero_async): [offset, offset + size) from the start of the workspace
void t3d_canonicalize_structured_zero_range(int64_t V, int64_t F, uint32_t cap_z, uint32_t cap_g0, int Zs, int64_t* offset,
                                            int64_t* size)
{
    const int64_t n = V > F ? V : F;
    *size = 2 * align256(t3d_scan_workspace_bytes(n, 1)) + 256;
    *offset = t3d_canonicalize_structured_workspace_bytes(V, F, cap_z, cap_g0, Zs) - *size;
}

// verts_in / vkeys: capacity V_cap, true block sizes in sizes_u64 = {n_active, n_x, n_y, n_z, n_t} (device); V_dev_u64 = n_x+n_y+n_z
// and F_dev_u64 = n_t (device).  Zs: planes of the marched (local) sign volume; z_offset / unpad_shift / n_cum as passed to
// t3d_mc_vertices_dev.  counts_u64: [0] V' [1] F' [2] != 0: order not verified, fall back; n_g0_u64 (optional): size of the
// clamp group (a caller seeing [2] != 0 with *n_g0 > cap_g0 retries with a larger cap_g0).
extern "C" int t3d_mesh_canonicalize_structured_dev(const void* verts_in, const void* vkeys_u64, int64_t V_cap, const void* sizes_u64,
                                                    const void* V_dev_u64, int Zs, int Hs, int Ws, const void* chunkbase_u32,
                                                    const void* aw_base_u32, uint32_t aw_stride, int z_offset, int unpad_shift,
                                                    const void* cum_f64, const void* adj_f64, int n_cum, int zkey_bits,
                                                    uint32_t cap_z, uint32_t cap_g0, const void* faces_in, int64_t F_cap,
                                                    const void* F_dev_u64, void* verts_out, void* faces_out_i64, void* faces_out_i32,
                                                    void* counts_u64, void* n_g0_u64, void* workspace, int phases, void* stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (zkey_bits <= 0 || zkey_bits > 32) zkey_bits = 32;
    if (V_cap <= 0 || V_cap > 0x7fffffff || F_cap < 0 || Zs <= 0 || Hs <= 0 || Ws <= 0 || cap_z == 0 || (phases & 3) == 0) {
        t3d_set_error("t3d_mesh_canonicalize_structured: bad sizes");
        return 2;
    }
    const int64_t V = V_cap, F = F_cap, n = V > F ? V : F;
    char* ws = (char*)workspace;
    CanonS c;
    c.verts = (const float*)verts_in;
    c.vkeys = (const unsigned long long*)vkeys_u64;
    c.sizes = (const unsigned long long*)sizes_u64;
    c.cap_verts = (uint32_t)V; c.cap_z = cap_z; c.cap_g0 = cap_g0;
    c.Zs = Zs; c.Hs = Hs;
    c.ncr = (t3d_wpr(Ws) + 31) >> 5;
    c.chunkbase = (const uint32_t*)chunkbase_u32;
    c.aw_base = (const uint32_t*)aw_base_u32;
    c.stride = aw_stride;
    c.g_plane = (n_cum > 0 && unpad_shift > 0) ? unpad_shift - z_offset : -1;
    c.z_offset = z_offset; c.shift = unpad_shift ? 1.0f : 0.0f;
    c.cum = (const double*)cum_f64; c.adj = (const double*)adj_f64; c.n_cum = n_cum;
    c.zkey_bits = zkey_bits;
    unsigned long long* zkeys_b; uint32_t* zperm; unsigned long long* gkeys_b; uint32_t* gperm;
    c.zkeys = (unsigned long long*)ws; ws += align256(8 * (int64_t)cap_z);
    zkeys_b = (unsigned long long*)ws; ws += align256(8 * (int64_t)cap_z);
    c.zval = (uint32_t*)ws; ws += align256(4 * (int64_t)cap_z);
    zperm = (uint32_t*)ws; ws += align256(4 * (int64_t)cap_z);
    c.gkeys = (unsigned long long*)ws; ws += align256(8 * (int64_t)cap_g0);
    gkeys_b = (unsigned long long*)ws; ws += align256(8 * (int64_t)cap_g0);
    c.gval = (uint32_t*)ws; ws += align256(4 * (int64_t)cap_g0);
    gperm = (uint32_t*)ws; ws += align256(4 * (int64_t)cap_g0);
    c.perm = (uint32_t*)ws; ws += align256(4 * V);
    uint32_t* flags = (uint32_t*)ws; ws += align256(4 * n);
    uint32_t* pos = (uint32_t*)ws; ws += align256(4 * n);
    uint32_t* newid = (uint32_t*)ws; ws += align256(4 * V);
    void* temp = ws; ws += align256(4 * (int64_t)cap_g0 + 256);             // k_gsort's second value buffer
    void* scan_ws = ws; ws += align256(t3d_scan_workspace_bytes(n, 1));
    void* scan_ws_f = ws; ws += align256(t3d_scan_workspace_bytes(n, 1));
    unsigned long long* totals = (unsigned long long*)ws;
    unsigned long long* counts = (unsigned long long*)counts_u64;
    c.zperm = zperm; c.gperm = gperm;
    c.n_g0_out = (unsigned long long*)n_g0_u64;
    if (phases & 1) {
        // one CTA per cube layer: segmented stable radix sort of the layer's z-edge vertices (no library)
        uint32_t* keyA = (uint32_t*)c.zkeys;
        uint32_t* keyB = keyA + cap_z;
        uint32_t* idxA = (uint32_t*)zkeys_b;
        uint32_t* idxB = idxA + cap_z;
        if ((int64_t)cap_z >= 4096 * (int64_t)Zs) k_zsort_layers<8><<<Zs, ZS_THREADS, 0, st>>>(c, keyA, keyB, idxA, idxB, zperm);
        else k_zsort_layers<1><<<Zs, ZS_THREADS, 0, st>>>(c, keyA, keyB, idxA, idxB, zperm);
        t3d_count_launches(1);
    }
    if (phases & 2) {
        if (t3d_zero_async(counts + 2, 8, st)) return 1;
        if (cap_g0 > 0) {
            // one CTA: stable radix sort of the clamp group by (y, x); gval / `temp` serve as the second value / key buffers
            k_gsort<<<1, ZS_THREADS, 0, st>>>(c, c.gkeys, gkeys_b, c.gval, (uint32_t*)temp, gperm);
        }
        k_canon_positions<<<(unsigned)((V + 255) / 256), 256, 0, st>>>(c);
        if (canonical_tail(c.verts, c.perm, V, (const unsigned long long*)V_dev_u64, faces_in, F, (const unsigned long long*)F_dev_u64,
                           verts_out, faces_out_i64, faces_out_i32, counts, flags, pos, newid, scan_ws, scan_ws_f, totals, st)) return 1;
        t3d_count_launches((F > 0 ? 5 : 3) + (cap_g0 > 0 ? 1 : 0));
    }
    T3D_CHECK_LAUNCH("t3d_mesh_canonicalize_structured");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// mesh measures: signed volume sum_f v0.(v1 x v2)/6 and area sum_f 0.5|(v1-v0)x(v2-v0)|, float64 terms and
// float64 accumulation, fixed reduction order (warp-shuffle trees, then one block over the block partials)
// ------------------------------------------------------------------------------------------------
template <typename IdxT>
__global__ void __launch_bounds__(256) k_mesh_measure(const float* __restrict__ verts, const IdxT* __restrict__ faces, int64_t F_cap,
                                                      double* __restrict__ partials, const unsigned long long* __restrict__ F_dev = nullptr)
{
    const int64_t F = dev_n(F_cap, F_dev);
    double vol = 0.0, area = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < F; i += (int64_t)gridDim.x * blockDim.x) {
        const float* a = verts + 3 * (int64_t)faces[3 * i];
        const float* b = verts + 3 * (int64_t)faces[3 * i + 1];
        const float* c = verts + 3 * (int64_t)faces[3 * i + 2];
        const double ax = a[0], ay = a[1], az = a[2], bx = b[0], by = b[1], bz = b[2], cx = c[0], cy = c[1], cz = c[2];
        const double nx = by * cz - bz * cy, ny = bz * cx - bx * cz, nz = bx * cy - by * cx;
        vol += (ax * nx + ay * ny + az * nz) / 6.0;
        const double ux = bx - ax, uy = by - ay, uz = bz - az, vx = cx - ax, vy = cy - ay, vz = cz - az;
        const double px = uy * vz - uz * vy, py = uz * vx - ux * vz, pz = ux * vy - uy * vx;
        area += 0.5 * sqrt(px * px + py * py + pz * pz);
    }
    vol = warp_sum(vol); area = warp_sum(area);
    __shared__ double sv[8], sa[8];
    if (lane_id() == 0) { sv[threadIdx.x >> 5] = vol; sa[threadIdx.x >> 5] = area; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = 0, a = 0;
        for (int k = 0; k < 8; ++k) { v += sv[k]; a += sa[k]; }
        partials[2 * blockIdx.x] = v; partials[2 * blockIdx.x + 1] = a;
    }
}

__global__ void __launch_bounds__(256) k_reduce_partials(const double* __restrict__ partials, int n, double* __restrict__ out)
{
    double v = 0, a = 0;
    for (int i = threadIdx.x; i < n; i += 256) { v += partials[2 * i]; a += partials[2 * i + 1]; }
    v = warp_sum(v); a = warp_sum(a);
    __shared__ double sv[8], sa[8];
    if (lane_id() == 0) { sv[threadIdx.x >> 5] = v; sa[threadIdx.x >> 5] = a; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double tv = 0, ta = 0;
        for (int k = 0; k < 8; ++k) { tv += sv[k]; ta += sa[k]; }
        out[0] = tv; out[1] = ta;
    }
}

#define MM_BLOCKS (T3D_NUM_SMS * 4)

extern "C" int64_t t3d_mesh_measure_workspace_bytes(void) { return (int64_t)MM_BLOCKS * 2 * 8; }

// out_f64[0] = signed volume, out_f64[1] = area (device).  F_dev_u64 (optional, device uint64): the true face count when F is
// only a capacity.
extern "C" int t3d_mesh_measure_dev(const void* verts_f32, const void* faces, int64_t F, const void* F_dev_u64, int faces_are_i64,
                                    void* out_f64, void* workspace, void* stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long* F_dev = (const unsigned long long*)F_dev_u64;
    if (F <= 0) { T3D_CUDA(cudaMemsetAsync(out_f64, 0, 16, st)); return 0; }
    int blocks = (int)((F + 255) / 256);
    if (blocks > MM_BLOCKS) blocks = MM_BLOCKS;
    if (faces_are_i64)
        k_mesh_measure<long long><<<blocks, 256, 0, st>>>((const float*)verts_f32, (const long long*)faces, F, (double*)workspace, F_dev);
    else
        k_mesh_measure<int32_t><<<blocks, 256, 0, st>>>((const float*)verts_f32, (const int32_t*)faces, F, (double*)workspace, F_dev);
    k_reduce_partials<<<1, 256, 0, st>>>((const double*)workspace, blocks, (double*)out_f64);
    T3D_CHECK_LAUNCH("t3d_mesh_measure_dev");
    t3d_count_launches(2);
    return 0;
}
