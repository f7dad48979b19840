// t3d_voxel.cu -- VoxelProcessor / VolumeCalculator kernels (sm_100a).
//
// Reference semantics (file:line into the reference repository):
//   pack        : image_loader.py:108 (`img >= threshold`) + np.stack, voxel_processor.py:46
//   fill_holes  : scipy.ndimage.binary_fill_holes on slice 0 / Z-1, voxel_processor.py:60-70
//   gap_fill    : the z loop of _close_volume_ends, voxel_processor.py:72-75 (== 3-point z stencil)
//   morph       : skimage binary_opening / binary_closing, voxel_processor.py:87-91
//   stats       : np.sum per slice (volume_calculator.py:31-33) and np.where min/max (:62-79)
//   point cloud : np.where + subsample, voxel_processor.py:99-108
//
// All kernels are HBM/L2-bandwidth bound integer work on the bit-packed occupancy; no tensor cores.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "t3d_common.cuh"

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

extern "C" void t3d_set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char* t3d_last_error(void) { return g_err; }
static long long g_launches = 0;
extern "C" void t3d_count_launches(int n) { g_launches += n; }
extern "C" int64_t t3d_launch_count(void) { return g_launches; }

struct ZeroRange { const char* p; size_t n; };
static thread_local ZeroRange g_zero[8];
static thread_local int g_nzero = 0;
void t3d_prezero_register(const void* p, size_t n) { if (g_nzero < 8) g_zero[g_nzero++] = {(const char*)p, n}; }
void t3d_prezero_clear(void) { g_nzero = 0; }
int t3d_zero_async(void* p, size_t n, cudaStream_t st)
{
    for (int k = 0; k < g_nzero; ++k)
        if ((const char*)p >= g_zero[k].p && (const char*)p + n <= g_zero[k].p + g_zero[k].n) return 0;   // zeroed up front
    T3D_CUDA(cudaMemsetAsync(p, 0, n, st));
    return 0;
}

int t3d_num_sms(void)
{
    static int sms[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 148; }
    int& n = sms[dev & 63];
    if (n <= 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) { cudaGetLastError(); v = 148; }
        n = v;
    }
    return n;
}

bool t3d_first_use_on_device(int slot)
{
    static bool done[T3D_ONCE_SLOTS][64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = 0; }
    bool& d = done[slot][dev & 63];
    const bool first = !d;
    d = true;
    return first;
}

extern "C" int t3d_version(void) { return 100; }
extern "C" int64_t t3d_words_per_row(int W) { return t3d_wpr(W); }

// ------------------------------------------------------------------------------------------------
// pack: uint8 (Z,H,W) -> bits.  Fast path: W % 32 == 0 and 16-byte aligned input; each warp turns
// 1024 contiguous bytes into 32 contiguous words per iteration with fully coalesced 128-bit loads.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_flat(const uint8_t* __restrict__ src, uint32_t* __restrict__ dst,
                                                   int64_t n_words, uint32_t thr4)
{
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t l = lane_id();
    const int64_t n_chunks = n_words >> 5;  // chunks of 32 words = 1024 bytes
    for (int64_t c = warp; c < n_chunks; c += n_warps) {
        const uint8_t* p = src + (c << 10);
        const uint4 a = ld_stream_u4(p + 16 * l);
        const uint4 b = ld_stream_u4(p + 512 + 16 * l);
        const uint32_t ha = ge16(a, thr4), hb = ge16(b, thr4);
        const int s0 = (2 * l) & 31;
        const uint32_t a0 = __shfl_sync(0xffffffffu, ha, s0), a1 = __shfl_sync(0xffffffffu, ha, s0 + 1);
        const uint32_t b0 = __shfl_sync(0xffffffffu, hb, s0), b1 = __shfl_sync(0xffffffffu, hb, s0 + 1);
        dst[(c << 5) + l] = (l < 16) ? (a0 | (a1 << 16)) : (b0 | (b1 << 16));
    }
    // tail words (n_words % 32): one thread per word
    const int64_t tail0 = n_chunks << 5;
    const int64_t t = tail0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_words) {
        const uint4* p = reinterpret_cast<const uint4*>(src + (t << 5));
        dst[t] = ge16(p[0], thr4) | (ge16(p[1], thr4) << 16);
    }
}

// generic path: any W, any alignment; one thread per output word
__global__ void __launch_bounds__(256) k_pack_generic(const uint8_t* __restrict__ src, uint32_t* __restrict__ dst,
                                                      int64_t n_rows, int W, int wpr, int thr)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * wpr) return;
    const int64_t row = i / wpr;
    const int w = (int)(i - row * wpr);
    const uint8_t* p = src + row * W + (w << 5);
    const int n = min(32, W - (w << 5));
    uint32_t v = 0;
    for (int k = 0; k < n; ++k) v |= (uint32_t)(p[k] >= thr) << k;
    dst[i] = v;
}

extern "C" int t3d_pack_masks(const void* masks_u8, int Z, int H, int W, int threshold, void* bits, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_pack_masks: empty volume"); return 2; }
    if (threshold < 0) threshold = 0;
    if (threshold > 256) threshold = 256;
    cudaStream_t st = (cudaStream_t)stream;
    const int wpr = t3d_wpr(W);
    const int64_t rows = (int64_t)Z * H;
    if ((W & 127) == 0 && ((uintptr_t)masks_u8 & 15) == 0 && threshold >= 1 && threshold <= 255) {
        const int64_t n_words = rows * wpr;
        const uint32_t thr4 = 0x01010101u * (uint32_t)threshold;
        int64_t blocks = (n_words / 32 + 7) / 8;           // one warp-iteration per 32 words
        const int64_t cap = (int64_t)T3D_NUM_SMS * 16;     // persistent-ish: 16 CTAs of 8 warps per SM
        if (blocks > cap) blocks = cap;
        if (blocks < 1) blocks = 1;
        k_pack_flat<<<(unsigned)blocks, 256, 0, st>>>((const uint8_t*)masks_u8, (uint32_t*)bits, n_words, thr4);
    } else {
        const int64_t n = rows * wpr;
        k_pack_generic<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const uint8_t*)masks_u8, (uint32_t*)bits, rows, W,
                                                                    wpr, threshold);
    }
    T3D_CHECK_LAUNCH("t3d_pack_masks");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// unpack: bits -> uint8 0/1 (numpy bool) for the API-visible volumes
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_unpack_flat(const uint32_t* __restrict__ src, uint8_t* __restrict__ dst,
                                                     int64_t n_words)
{
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t l = lane_id();
    const int64_t n_chunks = (n_words + 31) >> 5;
    for (int64_t c = warp; c < n_chunks; c += n_warps) {
        const int64_t wi = (c << 5) + l;
        const uint32_t w = wi < n_words ? src[wi] : 0u;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            // lane writes 16 bytes at offset 16*l of this 512-byte half: bits of word (16*half + l/2), half-word l&1
            const uint32_t ww = __shfl_sync(0xffffffffu, w, 16 * half + (l >> 1));
            const uint32_t h = (ww >> (16 * (l & 1))) & 0xffffu;
            uint4 o;
            o.x = expand4(h & 15u); o.y = expand4((h >> 4) & 15u);
            o.z = expand4((h >> 8) & 15u); o.w = expand4((h >> 12) & 15u);
            const int64_t word_of_lane = (c << 5) + 16 * half + (l >> 1);
            if (word_of_lane < n_words) st_stream_u4(dst + (c << 10) + 512 * half + 16 * l, o);
        }
    }
}

__global__ void __launch_bounds__(256) k_unpack_generic(const uint32_t* __restrict__ src, uint8_t* __restrict__ dst,
                                                        int64_t n_rows, int W, int wpr)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * wpr) return;
    const int64_t row = i / wpr;
    const int w = (int)(i - row * wpr);
    const uint32_t v = src[i];
    uint8_t* p = dst + row * W + (w << 5);
    const int n = min(32, W - (w << 5));
    for (int k = 0; k < n; ++k) p[k] = (v >> k) & 1u;
}

extern "C" int t3d_unpack_bits(const void* bits, int Z, int H, int W, void* out_u8, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_unpack_bits: empty volume"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int wpr = t3d_wpr(W);
    const int64_t rows = (int64_t)Z * H;
    const int64_t n = rows * wpr;
    if ((W & 127) == 0 && ((uintptr_t)out_u8 & 15) == 0) {
        int64_t blocks = ((n + 31) / 32 + 7) / 8;
        const int64_t cap = (int64_t)T3D_NUM_SMS * 16;
        if (blocks > cap) blocks = cap;
        if (blocks < 1) blocks = 1;
        k_unpack_flat<<<(unsigned)blocks, 256, 0, st>>>((const uint32_t*)bits, (uint8_t*)out_u8, n);
    } else {
        k_unpack_generic<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const uint32_t*)bits, (uint8_t*)out_u8, rows, W, wpr);
    }
    T3D_CHECK_LAUNCH("t3d_unpack_bits");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// 2-D hole filling of one bit plane (in place): complement of the 4-connected flood fill of the
// background started from outside the image.  One CTA of 1024 threads per plane; every iteration
// closes reachability along whole rows (carry-lookahead over words) and along whole columns
// (segmented carry-lookahead over rows), so convex-ish objects converge in two iterations.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t fill_up(uint32_t m, uint32_t s)  // flood s within m towards bit 31
{
    s |= m & (s << 1);  m &= m << 1;
    s |= m & (s << 2);  m &= m << 2;
    s |= m & (s << 4);  m &= m << 4;
    s |= m & (s << 8);  m &= m << 8;
    s |= m & (s << 16);
    return s;
}
__device__ __forceinline__ uint32_t fill_dn(uint32_t m, uint32_t s)  // towards bit 0
{
    s |= m & (s >> 1);  m &= m >> 1;
    s |= m & (s >> 2);  m &= m >> 2;
    s |= m & (s >> 4);  m &= m >> 4;
    s |= m & (s >> 8);  m &= m >> 8;
    s |= m & (s >> 16);
    return s;
}

// closure of `reach` along rows, both directions.  A warp owns 32 consecutive rows: it stages a 32-row x 16-word tile
// of the mask and of `reach` in shared memory with coalesced loads (row pitch 17 words: conflict-free when lane = row),
// every lane then runs the carry chain of ITS row over the 16 words, and the tile is written back coalesced.  The
// carry of each row crosses tiles in a register.
#define FH_TW 16
#define FH_PITCH 17

__device__ __forceinline__ void rows_closure_tile(const uint32_t* __restrict__ m, uint32_t* __restrict__ r, int nw, int nwv,
                                                  int y0, int H, uint32_t* tm, uint32_t* tr)
{
    const uint32_t l = lane_id();
    const int rsub = l >> 4, wsub = l & 15;
    const int n_tiles = (nwv + FH_TW - 1) / FH_TW;
    for (int dir = 0; dir < 2; ++dir) {
        uint32_t carry = 0;
        for (int t = 0; t < n_tiles; ++t) {
            const int c = dir == 0 ? t : n_tiles - 1 - t;
            const int w = c * FH_TW + wsub;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int rr = 2 * j + rsub, y = y0 + rr;
                const bool ok = (y < H) && (w < nwv);
                tm[rr * FH_PITCH + wsub] = ok ? m[(int64_t)y * nw + w] : 0u;
                tr[rr * FH_PITCH + wsub] = ok ? r[(int64_t)y * nw + w] : 0u;
            }
            __syncwarp();
            uint32_t* mr = tm + l * FH_PITCH;
            uint32_t* rr_ = tr + l * FH_PITCH;
            if (dir == 0) {
#pragma unroll
                for (int k = 0; k < FH_TW; ++k) {
                    const uint32_t mm = mr[k];
                    const uint32_t f = fill_up(mm, rr_[k] | (carry & mm & 1u));
                    carry = f >> 31;
                    rr_[k] = f;
                }
            } else {
#pragma unroll
                for (int k = FH_TW - 1; k >= 0; --k) {
                    const uint32_t mm = mr[k];
                    const uint32_t f = fill_dn(mm, rr_[k] | ((carry << 31) & mm));
                    carry = f & 1u;
                    rr_[k] = f;
                }
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int rr = 2 * j + rsub, y = y0 + rr;
                if (y < H && w < nwv) r[(int64_t)y * nw + w] = tr[rr * FH_PITCH + wsub];
            }
            __syncwarp();
        }
    }
}

#define FH_THREADS 1024
#define FH_MAXSEG 64

__global__ void __launch_bounds__(FH_THREADS) k_fill_holes(uint32_t* bits_planes, int64_t plane_stride_words,
                                                           uint32_t* scratch, int H, int W, int nw)
{
    // plane handled by this CTA; scratch layout: [plane][0: mask m][1: reach r], each H*nw words
    uint32_t* bits = bits_planes + (int64_t)blockIdx.x * plane_stride_words;
    const int64_t pw = (int64_t)H * nw;
    uint32_t* m = scratch + (int64_t)blockIdx.x * 2 * pw;
    uint32_t* r = m + pw;
    const int tid = threadIdx.x;
    const int warp = tid >> 5;

    // background mask + seeds (background pixels on the image border touch the "outside")
    for (int64_t i = tid; i < pw; i += FH_THREADS) {
        const int y = (int)(i / nw), w = (int)(i - (int64_t)y * nw);
        const uint32_t vm = valid_mask(w, W);
        const uint32_t bg = ~bits[i] & vm;
        uint32_t seed = 0;
        if (y == 0 || y == H - 1) seed = bg;
        if (w == 0) seed |= bg & 1u;
        if (w == ((W - 1) >> 5)) seed |= bg & (1u << ((W - 1) & 31));
        m[i] = bg;
        r[i] = seed;
    }
    __syncthreads();

    extern __shared__ uint32_t tile[];  // per warp: mask tile + reach tile, 32 rows x FH_PITCH words each
    // column segments: thread (seg, col) sweeps rows [seg*L, seg*L+L)
    __shared__ uint32_t sG[FH_MAXSEG][32];  // used in column tiles of 32 word-columns
    __shared__ uint32_t sP[FH_MAXSEG][32];
    const int nseg = min(FH_MAXSEG, min(FH_THREADS / 32, H));  // 32 segments
    const int L = (H + nseg - 1) / nseg;

    for (int iter = 0; iter < 4 * (H + W) + 8; ++iter) {
        // A round = row closure then column closure.  The row closure is idempotent, so the fixpoint is reached as
        // soon as a column closure changes nothing: only the column phase feeds `changed`.
        int changed = 0;
        // ---- rows
        for (int y0 = warp * 32; y0 < H; y0 += (FH_THREADS / 32) * 32)
            rows_closure_tile(m, r, nw, (W + 31) >> 5, y0, H, tile + warp * 2 * 32 * FH_PITCH,
                              tile + warp * 2 * 32 * FH_PITCH + 32 * FH_PITCH);
        __syncthreads();
        // ---- columns, 32 word-columns at a time: thread = (seg = warp, col = lane)
        for (int c0 = 0; c0 < nw; c0 += 32) {
            const int c = c0 + (tid & 31), seg = warp;
            const bool act = (c < nw) && (seg < nseg);
            const int y0 = seg * L, y1 = min(H, y0 + L);
            for (int dir = 0; dir < 2; ++dir) {
                // pass 1: segment summary with zero carry-in
                uint32_t G = 0, P = 0xffffffffu;
                if (act && y0 < y1) {
                    if (dir == 0) for (int y = y0; y < y1; ++y) { const uint32_t mm = m[(int64_t)y * nw + c]; G = r[(int64_t)y * nw + c] | (G & mm); P &= mm; }
                    else          for (int y = y1 - 1; y >= y0; --y) { const uint32_t mm = m[(int64_t)y * nw + c]; G = r[(int64_t)y * nw + c] | (G & mm); P &= mm; }
                } else { P = 0xffffffffu; G = 0; }
                if (seg < FH_MAXSEG) { sG[seg][tid & 31] = G; sP[seg][tid & 31] = (act && y0 < y1) ? P : 0xffffffffu; }
                __syncthreads();
                // pass 2: carry into this segment
                uint32_t cin = 0;
                if (act) {
                    if (dir == 0) for (int s = 0; s < seg; ++s) cin = sG[s][tid & 31] | (sP[s][tid & 31] & cin);
                    else          for (int s = nseg - 1; s > seg; --s) cin = sG[s][tid & 31] | (sP[s][tid & 31] & cin);
                }
                // pass 3: final sweep (rows fetched eight at a time ahead of the dependent chain)
                if (act && y0 < y1) {
                    uint32_t carry = cin;
                    const int n = y1 - y0;
                    for (int k0 = 0; k0 < n; k0 += 8) {
                        uint32_t mm[8], rr[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            const int kk = k0 + k;
                            const int y = dir == 0 ? y0 + kk : y1 - 1 - kk;
                            const bool ok = kk < n;
                            mm[k] = ok ? m[(int64_t)y * nw + c] : 0u;
                            rr[k] = ok ? r[(int64_t)y * nw + c] : 0u;
                        }
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            const int kk = k0 + k;
                            if (kk < n) {
                                const int y = dir == 0 ? y0 + kk : y1 - 1 - kk;
                                const uint32_t nv = rr[k] | (carry & mm[k]);
                                if (nv != rr[k]) { r[(int64_t)y * nw + c] = nv; changed = 1; }
                                carry = nv;
                            }
                        }
                    }
                }
                __syncthreads();
            }
        }
        if (!__syncthreads_or(changed)) break;
    }
    // holes = background never reached
    for (int64_t i = tid; i < pw; i += FH_THREADS) bits[i] |= m[i] & ~r[i];
}

extern "C" int64_t t3d_fill_holes_scratch_bytes(int n_planes, int H, int W)
{
    return (int64_t)n_planes * 2 * H * t3d_wpr(W) * 4;
}

extern "C" int t3d_fill_holes_2d(void* bits, int n_planes, int64_t plane_stride_words, int H, int W, void* scratch,
                                 void* stream)
{
    if (n_planes <= 0) return 0;
    if (H <= 0 || W <= 0) { t3d_set_error("t3d_fill_holes_2d: empty plane"); return 2; }
    const size_t smem = (size_t)(FH_THREADS / 32) * 2 * 32 * FH_PITCH * sizeof(uint32_t);  // 136 KB
    if (t3d_first_use_on_device(T3D_ONCE_FILL_HOLES_ATTR))   // function attributes are per device
        T3D_CUDA(cudaFuncSetAttribute(k_fill_holes, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_fill_holes<<<n_planes, FH_THREADS, smem, (cudaStream_t)stream>>>((uint32_t*)bits, plane_stride_words,
                                                                      (uint32_t*)scratch, H, W, t3d_wpr(W));
    T3D_CHECK_LAUNCH("t3d_fill_holes_2d");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// z gap fill: out[z] = f[z] | (f[z-1] & f[z+1]) for 1 <= z <= Z-2, copy for z = 0, Z-1
// (voxel_processor.py:72-75; the np.any guards are redundant and the loop is not a recurrence,
// SURVEY.md V3).  `lo` / `hi` are optional neighbour planes for z-slab sharding: when given, local
// plane 0 / Z-1 is an interior plane of the global stack and uses them as f[-1] / f[Z].
// Optionally accumulates per-slice popcounts of the result.  128-bit accesses, two per thread in flight.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_gap_fill(const uint4* __restrict__ in, uint4* __restrict__ out,
                                                  const uint4* __restrict__ lo, const uint4* __restrict__ hi, int Z,
                                                  int64_t pw4, unsigned long long* __restrict__ counts)
{
    const int z = blockIdx.y;
    const uint4* c = in + (int64_t)z * pw4;
    const uint4* a = (z > 0) ? c - pw4 : lo;
    const uint4* b = (z < Z - 1) ? c + pw4 : hi;
    uint4* o = out + (int64_t)z * pw4;
    uint32_t cnt = 0;
    const bool fill = (a != nullptr) && (b != nullptr);
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < pw4; i += 2 * stride) {
        const int64_t j = i + stride;
        const bool two = j < pw4;
        uint4 v0 = c[i], v1 = two ? c[j] : make_uint4(0, 0, 0, 0);
        if (fill) {
            const uint4 a0 = a[i], b0 = b[i];
            v0 = or4(v0, and4(a0, b0));
            if (two) { const uint4 a1 = a[j], b1 = b[j]; v1 = or4(v1, and4(a1, b1)); }
        }
        o[i] = v0;
        if (two) o[j] = v1;
        cnt += popc4(v0) + popc4(v1);
    }
    if (counts) {
        cnt = warp_sum(cnt);
        __shared__ uint32_t s[8];
        if (lane_id() == 0) s[threadIdx.x >> 5] = cnt;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long t = 0;
            for (int k = 0; k < 8; ++k) t += s[k];
            if (t) atomicAdd(counts + z, t);
        }
    }
}

extern "C" int t3d_gap_fill(const void* in_bits, void* out_bits, const void* lo_plane, const void* hi_plane, int Z, int H,
                            int W, void* slice_counts_u64, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_gap_fill: empty volume"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t pw4 = (int64_t)H * (t3d_wpr(W) / 4);
    if (slice_counts_u64 && t3d_zero_async(slice_counts_u64, sizeof(unsigned long long) * Z, st)) return 1;
    int bx = (int)min((int64_t)32, (pw4 + 511) / 512);
    dim3 grid(bx, Z);
    k_gap_fill<<<grid, 256, 0, st>>>((const uint4*)in_bits, (uint4*)out_bits, (const uint4*)lo_plane, (const uint4*)hi_plane, Z,
                                     pw4, (unsigned long long*)slice_counts_u64);
    T3D_CHECK_LAUNCH("t3d_gap_fill");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Fused create_voxel_data: `img >= threshold` + np.stack + the z loop of _close_volume_ends + np.sum per slice + the
// np.where extrema, in ONE pass over the uint8 stack (voxel_processor.py:46-52, 72-75; volume_calculator.py:62-79).
// A warp owns 1024 consecutive bytes (32 packed words) of the (y,x) plane and marches along z through a chunk of planes
// with the packed words of planes z-1, z, z+1 in registers: out[z] = w[z] | (w[z-1] & w[z+1]).  Every mask byte is read
// once (plus one halo plane per chunk end), the bit volume is written once, nothing is re-read.
// The two end planes need scipy.ndimage.binary_fill_holes first (voxel_processor.py:60-70): k_pack_gap treats them as
// raw and k_close_ends_fixup afterwards rewrites planes 0, 1, Z-2, Z-1 from the hole-filled end planes (and counts them).
// Extrema are accumulated in a form that works on zero-initialised memory: {INT_MAX - min, max + 1} under atomicMax.
// ------------------------------------------------------------------------------------------------
#define PG_ZC 128   // most planes a chunk may have

struct PackGapArgs {
    const uint8_t* src;
    uint32_t* dst;
    int Z, nw;                    // nw: words per row (= W/32 on this path)
    long long plane_words, plane_bytes;
    uint32_t thr4;
    int zc;                       // planes per chunk (<= PG_ZC)
    int skip_ends;                // planes 0, 1, Z-2, Z-1 are not counted here (k_close_ends_fixup counts them)
    int z_bias;                   // added to the z extrema (a sub-stack of a z-slab reports planes of the slab)
    unsigned long long* counts;   // Z per-slice counts (zeroed by the caller) or null
    unsigned int* bbox_t;         // 6 transformed extrema {z, y, x} x {INT_MAX - min, max + 1} (zeroed by the caller) or null
};

// `byte >= threshold` for the 16 bytes of a uint4 -> 16 bits, threshold 1..255, with the constants of ThrK:
// low 7 bits by a carry that cannot leave the byte ((v & 0x7f) + (0x80 - (t & 0x7f)) sets bit 7 iff low7(v) >= low7(t)), then
// bit 7 of the result is MAJ(carry, v, ~t) at bit 7 (t < 128: carry | v7, t >= 128: carry & v7) -- four ALU operations per
// four bytes where the emulated SIMD compare took about ten; the four result bits are gathered by one multiply and the four
// nibbles of the uint4 are chained by funnel shifts.
struct ThrK { uint32_t add7, n7; };
__device__ __forceinline__ ThrK make_thrk(uint32_t thr4)
{
    ThrK k;
    k.add7 = 0x80808080u - (thr4 & 0x7f7f7f7fu);
    k.n7 = ~thr4 & 0x80808080u;
    return k;
}
__device__ __forceinline__ uint32_t ge4_top(uint32_t v, const ThrK& k)      // result nibble in bits 28..31 (garbage below)
{
    const uint32_t c = (v & 0x7f7f7f7fu) + k.add7;
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(r) : "r"(c), "r"(v), "r"(k.n7));   // MAJ(c, v, n7) (kept as ONE operation)
    return (r & 0x80808080u) * 0x00204081u;
}
__device__ __forceinline__ uint32_t ge16k(const uint4& v, const ThrK& k)
{
    uint32_t acc = ge4_top(v.w, k) >> 28;
    acc = __funnelshift_l(ge4_top(v.z, k), acc, 4);
    acc = __funnelshift_l(ge4_top(v.y, k), acc, 4);
    acc = __funnelshift_l(ge4_top(v.x, k), acc, 4);
    return acc;
}

// FULL: the plane is a whole number of 1024-byte spans (no partial span: no validity predicates in the loop)
template <bool FULL>
__global__ void __launch_bounds__(256) k_pack_gap(PackGapArgs a)
{
    __shared__ unsigned int s_cnt[PG_ZC];
    __shared__ unsigned int s_bb[6];
    const int tid = threadIdx.x, warp = tid >> 5;
    const uint32_t l = lane_id();
    if (tid < PG_ZC) s_cnt[tid] = 0;
    if (tid < 6) s_bb[tid] = 0;
    __syncthreads();
    const long long span = (long long)blockIdx.x * 8 + warp;     // 1024 bytes = 32 words of a plane
    const int za = blockIdx.y * a.zc, zb = min(a.Z, za + a.zc);
    const long long wi = span * 32 + l;                           // this lane's word of the plane
    const bool wvalid = FULL || wi < a.plane_words;
    const long long boff = span * 1024 + 16 * l;                  // this lane's first 16 mask bytes
    const bool va = FULL || boff + 16 <= a.plane_bytes, vb = FULL || boff + 512 + 16 <= a.plane_bytes;
    const ThrK tk = make_thrk(a.thr4);
    const int s0 = (2 * l) & 31;
    const uint32_t sel = l < 16 ? 0x5410u : 0x7632u;             // which halves of the two shuffled words make this lane's word
    // raw 2 x 16 mask bytes of this lane for plane z, and their conversion to the lane's packed word: split so that the
    // loads of later planes are in flight while an earlier one is converted (three planes of loads per warp)
    auto load_raw = [&](int z, uint4& x, uint4& y) {
        const uint8_t* p = a.src + (long long)z * a.plane_bytes + boff;
        const uint4 zero = make_uint4(0, 0, 0, 0);
        x = va ? ld_stream_u4(p) : zero;
        y = vb ? ld_stream_u4(p + 512) : zero;
    };
    auto to_word = [&](const uint4& x, const uint4& y) -> uint32_t {
        const uint32_t hab = ge16k(x, tk) | (ge16k(y, tk) << 16);                // bits of bytes [16l, 16l+16) and [512+16l, ...)
        const uint32_t x0 = __shfl_sync(0xffffffffu, hab, s0), x1 = __shfl_sync(0xffffffffu, hab, s0 + 1);
        return __byte_perm(x0, x1, sel);
    };
    uint32_t acc = 0;
    int zmin = 0x7fffffff, zmax = -1;
    if (span * 1024 < a.plane_bytes) {   // (warp-uniform; the last CTA of a plane may hold warps beyond it)
        uint4 r0x, r0y, r1x, r1y, r2x, r2y;      // raw planes z+1, z+2, z+3 (a ring, rotated by the 3-way unrolled loop)
        const int p_hi = min(zb, a.Z - 1);        // last plane this chunk reads
        uint32_t prev = 0u;
        if (za > 0) { load_raw(za - 1, r0x, r0y); prev = to_word(r0x, r0y); }
        load_raw(za, r0x, r0y);
        uint32_t cur = to_word(r0x, r0y);
        if (za + 1 <= p_hi) load_raw(za + 1, r0x, r0y);
        if (za + 2 <= p_hi) load_raw(za + 2, r1x, r1y);
        if (za + 3 <= p_hi) load_raw(za + 3, r2x, r2y);
        uint32_t* dp = a.dst + (long long)za * a.plane_words + wi;
        // one plane: rx/ry hold raw plane z+1 on entry and raw plane z+4 on exit
        auto step = [&](int z, uint4& rx, uint4& ry) {
            const bool hn = z + 1 < a.Z;
            const uint32_t next = hn ? to_word(rx, ry) : 0u;
            if (z + 4 <= p_hi) load_raw(z + 4, rx, ry);
            uint32_t v = cur;
            if (z > 0 && hn) v |= prev & next;
            if (wvalid) *dp = v;
            dp += a.plane_words;
            acc |= v;
            const unsigned wc = __reduce_add_sync(0xffffffffu, (unsigned)__popc(v));
            if (wc) {
                zmin = min(zmin, z);
                zmax = z;
                const bool counted = !(a.skip_ends && (z < 2 || z >= a.Z - 2));
                if (l == 0 && counted) atomicAdd(&s_cnt[z - za], wc);
            }
            prev = cur;
            cur = next;
        };
        for (int z = za; z < zb; z += 3) {
            step(z, r0x, r0y);
            if (z + 1 < zb) step(z + 1, r1x, r1y);
            if (z + 2 < zb) step(z + 2, r2x, r2y);
        }
    }
    if (a.bbox_t && zmax >= 0) {         // (warp-uniform)
        int ymin = 0x7fffffff, ymax = -1, xmin = 0x7fffffff, xmax = -1;
        if (acc) {
            const int y = (int)(wi / a.nw), w = (int)(wi - (long long)y * a.nw);
            ymin = ymax = y;
            xmin = (w << 5) + __ffs(acc) - 1;
            xmax = (w << 5) + 31 - __clz(acc);
        }
        ymin = __reduce_min_sync(0xffffffffu, ymin); ymax = __reduce_max_sync(0xffffffffu, ymax);
        xmin = __reduce_min_sync(0xffffffffu, xmin); xmax = __reduce_max_sync(0xffffffffu, xmax);
        if (l == 0) {
            atomicMax(&s_bb[0], (unsigned)(0x7fffffff - (zmin + a.z_bias))); atomicMax(&s_bb[1], (unsigned)(zmax + a.z_bias + 1));
            atomicMax(&s_bb[2], (unsigned)(0x7fffffff - ymin)); atomicMax(&s_bb[3], (unsigned)(ymax + 1));
            atomicMax(&s_bb[4], (unsigned)(0x7fffffff - xmin)); atomicMax(&s_bb[5], (unsigned)(xmax + 1));
        }
    }
    __syncthreads();
    if (a.counts && tid < zb - za && s_cnt[tid]) atomicAdd(a.counts + za + tid, (unsigned long long)s_cnt[tid]);
    if (a.bbox_t && tid < 6 && s_bb[tid]) atomicMax(a.bbox_t + tid, s_bb[tid]);
}

struct EndsFixArgs {
    const uint8_t* src;
    const uint32_t* f0;           // hole-filled plane 0
    const uint32_t* fT;           // hole-filled plane Z-1
    uint32_t* dst;
    int Z;
    long long plane_words, plane_bytes;
    uint32_t thr4;
    unsigned long long* counts;
};

// planes 0, 1, Z-2, Z-1 of the closed grid from the hole-filled end planes (Z >= 3; one thread per word; a word is 32
// consecutive mask bytes because W % 128 == 0 on this path)
__global__ void __launch_bounds__(256) k_close_ends_fixup(EndsFixArgs a)
{
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long pw = a.plane_words;
    const int Z = a.Z;
    unsigned c[4] = {0, 0, 0, 0};   // planes 0, 1, Z-2, Z-1
    if (i < pw) {
        auto raw = [&](int z) -> uint32_t {
            const uint4* p = reinterpret_cast<const uint4*>(a.src + (long long)z * a.plane_bytes + 32 * i);
            return ge16(p[0], a.thr4) | (ge16(p[1], a.thr4) << 16);
        };
        const uint32_t b = a.f0[i], t = a.fT[i];
        a.dst[i] = b;
        a.dst[(long long)(Z - 1) * pw + i] = t;
        c[0] = __popc(b); c[3] = __popc(t);
        const uint32_t v1 = raw(1) | (b & ((Z - 1 == 2) ? t : raw(2)));
        a.dst[pw + i] = v1;
        c[1] = __popc(v1);
        if (Z - 2 != 1) {
            const uint32_t vT = raw(Z - 2) | (((Z - 3 == 0) ? b : raw(Z - 3)) & t);
            a.dst[(long long)(Z - 2) * pw + i] = vT;
            c[2] = __popc(vT);
        }
    }
    if (!a.counts) return;
    __shared__ unsigned s[4];
    if (threadIdx.x < 4) s[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned w = __reduce_add_sync(0xffffffffu, c[k]);
        if (lane_id() == 0 && w) atomicAdd(&s[k], w);
    }
    __syncthreads();
    if (threadIdx.x < 4 && s[threadIdx.x]) {
        const int zz = threadIdx.x == 0 ? 0 : threadIdx.x == 1 ? 1 : threadIdx.x == 2 ? Z - 2 : Z - 1;
        atomicAdd(a.counts + zz, (unsigned long long)s[threadIdx.x]);
    }
}

bool t3d_pack_gap_supported(const void* masks_u8, int Z, int H, int W, int threshold)
{
    return Z >= 3 && H > 0 && (W & 127) == 0 && ((uintptr_t)masks_u8 & 15) == 0 && threshold >= 1 && threshold <= 255;
}

// masks -> gap-filled grid `out` (end planes still raw), per-slice counts (zeroed by the caller; planes 0, 1, Z-2, Z-1
// left out when skip_ends) and transformed extrema (6 uint32 zeroed by the caller, may be null)
int t3d_pack_gap_launch(const void* masks_u8, int Z, int H, int W, int threshold, void* out, unsigned long long* counts,
                        unsigned int* bbox_t, int skip_ends, cudaStream_t st, int z_bias)
{
    PackGapArgs a;
    a.z_bias = z_bias;
    a.src = (const uint8_t*)masks_u8; a.dst = (uint32_t*)out;
    a.Z = Z; a.nw = t3d_wpr(W);
    a.plane_words = (long long)H * a.nw; a.plane_bytes = (long long)H * W;
    a.thr4 = 0x01010101u * (uint32_t)threshold;
    const long long n_spans = (a.plane_bytes + 1023) / 1024;
    // about one wave of resident warps (64 per SM); chunks of 16..PG_ZC planes (each chunk re-reads two halo planes)
    long long chunks = ((long long)T3D_NUM_SMS * 64 + n_spans - 1) / n_spans;
    if (chunks < 1) chunks = 1;
    int zc = (int)((Z + chunks - 1) / chunks);
    if (zc < 16) zc = 16;
    if (zc > PG_ZC) zc = PG_ZC;
    a.zc = zc;
    a.skip_ends = skip_ends;
    a.counts = counts; a.bbox_t = bbox_t;
    dim3 grid((unsigned)((n_spans + 7) / 8), (unsigned)((Z + zc - 1) / zc));
    if (a.plane_bytes % 1024 == 0) k_pack_gap<true><<<grid, 256, 0, st>>>(a);
    else k_pack_gap<false><<<grid, 256, 0, st>>>(a);
    T3D_CHECK_LAUNCH("t3d_pack_gap");
    t3d_count_launches(1);
    return 0;
}

extern "C" int t3d_pack_gap(const void* masks_u8, int Z, int H, int W, int threshold, void* bits, void* counts_u64, void* bbox_u32x6,
                            void* stream)
{
    if (!t3d_pack_gap_supported(masks_u8, Z, H, W, threshold)) {
        t3d_set_error("t3d_pack_gap: needs Z >= 3, W %% 128 == 0, a 16-byte aligned stack and 1 <= threshold <= 255");
        return 2;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // counts / extrema are ACCUMULATED (atomics): the caller zeroes them, as t3d_reconstruct does with its one up-front zeroing kernel
    return t3d_pack_gap_launch(masks_u8, Z, H, W, threshold, bits, (unsigned long long*)counts_u64, (unsigned int*)bbox_u32x6, 0, st);
}

// extrema of the set voxels of `n_planes` planes in k_pack_gap's transformed form ({INT_MAX - min, max + 1} under atomicMax on
// zero-initialised memory); plane p of the call is plane z_bias + p of the slab.  One CTA per (plane, band of rows).
__global__ void __launch_bounds__(256) k_bbox_t_planes(const uint32_t* __restrict__ bits, int H, int nw, int z_bias, unsigned int* __restrict__ bbox_t)
{
    const int z = blockIdx.y;
    const uint32_t* p = bits + (long long)z * H * nw;
    const int rows_per = (H + gridDim.x - 1) / gridDim.x;
    const int ya = blockIdx.x * rows_per, yb = min(H, ya + rows_per);
    int ymin = 0x7fffffff, ymax = -1, xmin = 0x7fffffff, xmax = -1;
    for (long long i = (long long)ya * nw + threadIdx.x; i < (long long)yb * nw; i += 256) {
        const uint32_t v = p[i];
        if (v) {
            const int y = (int)(i / nw), w = (int)(i - (long long)y * nw);
            ymin = min(ymin, y); ymax = max(ymax, y);
            xmin = min(xmin, (w << 5) + __ffs(v) - 1);
            xmax = max(xmax, (w << 5) + 31 - __clz(v));
        }
    }
    ymin = __reduce_min_sync(0xffffffffu, ymin); ymax = __reduce_max_sync(0xffffffffu, ymax);
    xmin = __reduce_min_sync(0xffffffffu, xmin); xmax = __reduce_max_sync(0xffffffffu, xmax);
    if ((threadIdx.x & 31) == 0 && ymax >= 0) {
        atomicMax(bbox_t + 0, (unsigned)(0x7fffffff - (z + z_bias))); atomicMax(bbox_t + 1, (unsigned)(z + z_bias + 1));
        atomicMax(bbox_t + 2, (unsigned)(0x7fffffff - ymin)); atomicMax(bbox_t + 3, (unsigned)(ymax + 1));
        atomicMax(bbox_t + 4, (unsigned)(0x7fffffff - xmin)); atomicMax(bbox_t + 5, (unsigned)(xmax + 1));
    }
}

int t3d_bbox_t_planes_launch(const uint32_t* bits, int n_planes, int H, int W, int z_bias, unsigned int* bbox_t, cudaStream_t st)
{
    if (n_planes <= 0) return 0;
    dim3 grid((unsigned)min(8, H), (unsigned)n_planes);
    k_bbox_t_planes<<<grid, 256, 0, st>>>(bits, H, t3d_wpr(W), z_bias, bbox_t);
    T3D_CHECK_LAUNCH("t3d_bbox_t_planes");
    t3d_count_launches(1);
    return 0;
}

int t3d_close_ends_fixup_launch(const void* masks_u8, int Z, int H, int W, int threshold, const void* filled0, const void* filledT,
                                void* out, unsigned long long* counts, cudaStream_t st)
{
    EndsFixArgs a;
    a.src = (const uint8_t*)masks_u8; a.f0 = (const uint32_t*)filled0; a.fT = (const uint32_t*)filledT; a.dst = (uint32_t*)out;
    a.Z = Z; a.plane_words = (long long)H * t3d_wpr(W); a.plane_bytes = (long long)H * W;
    a.thr4 = 0x01010101u * (uint32_t)threshold;
    a.counts = counts;
    k_close_ends_fixup<<<(unsigned)((a.plane_words + 255) / 256), 256, 0, st>>>(a);
    T3D_CHECK_LAUNCH("t3d_close_ends_fixup");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// 6-connected binary morphology.  Stage s of a call is an erosion (bit s of erode_mask set; out-of-volume = 1)
// or a dilation (out-of-volume = 0): exactly skimage's binary_erosion / binary_dilation with the default cross
// footprint (SURVEY.md 8a-3).  opening then closing = stages E,D,D,E = erode_mask 0b1001.
//
// One launch per stage.  A thread owns one uint4 column (128 voxels) of one plane and marches down `my` rows with the
// y neighbours in a register window; all addresses are running pointers (one add per row and stream), so a row costs
// 3 x 128-bit loads (next row, z-1, z+1) + 2 scalar loads (x neighbours, L1 hits), 8 funnel shifts, 12 LOP3 and one
// 128-bit store.  The output may live in a differently strided buffer: the last stage of the fused pipeline writes
// straight into the padded layout the marching-cubes kernels read (RING: it also clears the pad words of its rows).
// ------------------------------------------------------------------------------------------------
#define MY 8

struct MorphArgs {
    const uint32_t* in;          // compact (Z, H, nw) volume
    uint32_t* out;               // word (plane z0, row 0, word 0) of the output
    int Z, H, W, nw;
    int z0, nz;                  // planes [z0, z0 + nz) are computed
    int out_rs;                  // output row stride (words)
    long long out_ps;            // output plane stride (words)
    int lanes_x, pz_per_block, my;
    int ring_tail;               // RING: uint4s of zeros appended after the nw real words of every output row (0 or 1)
    unsigned long long* counts;  // COUNT: counts[z - z0] += set voxels of output plane z
};

// a row of border values for each kind of stage: neighbours outside the volume are read from here through pointers that
// do not advance, so the inner loop carries no predicated loads (each would cost four register moves for its default)
__device__ __align__(16) const uint32_t g_border_row[8] = {0u, 0u, 0u, 0u, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};

template <bool ER, bool FIX, bool COUNT, bool RING>
__global__ void __launch_bounds__(256, 4) k_morph(MorphArgs a)
{
    const int lx = threadIdx.x % a.lanes_x, pz = threadIdx.x / a.lanes_x;
    const int nw4 = a.nw >> 2, nwv = (a.W + 31) >> 5;
    const int w4 = blockIdx.x * a.lanes_x + lx, zi = blockIdx.z * a.pz_per_block + pz, y0 = blockIdx.y * a.my;
    extern __shared__ unsigned int s_cnt[];
    if (COUNT) {
        if ((int)threadIdx.x < a.pz_per_block) s_cnt[threadIdx.x] = 0;
        __syncthreads();
    }
    if (pz < a.pz_per_block && w4 < nw4 && zi < a.nz) {
        const int z = a.z0 + zi;
        const uint4 vm = valid_mask4(w4, a.W);
        // words beyond the volume (tail bits, padding words) read as the border value of this stage
        const bool fix = FIX && ER && (4 * w4 + 4 > (a.W >> 5));
        const uint4 fixm = fix ? make_uint4(~vm.x, ~vm.y, ~vm.z, ~vm.w) : make_uint4(0, 0, 0, 0);
        auto ld4 = [&](const uint32_t* p) -> uint4 {
            uint4 v = *reinterpret_cast<const uint4*>(p);
            if (FIX && ER) v = or4(v, fixm);
            return v;
        };
        const uint32_t* border = g_border_row + (ER ? 4 : 0);
        const bool has_l = (w4 > 0), has_r = (4 * w4 + 4 < nwv);
        const bool fix_r = FIX && ER && has_r && (4 * w4 + 5 >= nwv);   // the right neighbour is the partial last word
        const uint32_t fix_r_bits = fix_r ? ~valid_mask(4 * w4 + 4, a.W) : 0u;
        const long long in_ps = (long long)a.H * a.nw;
        const uint32_t* pc = a.in + (long long)z * in_ps + (long long)y0 * a.nw + 4 * w4;   // row (z, y)
        // neighbours: running pointers with a step of one row, or the border row with a step of zero
        const uint32_t* pm = (z > 0) ? pc - in_ps : border;
        const uint32_t* pp = (z + 1 < a.Z) ? pc + in_ps : border;
        const uint32_t* pl = has_l ? pc - 1 : border;
        const uint32_t* pr = has_r ? pc + 4 : border;
        const int sm = (z > 0) ? a.nw : 0, sp = (z + 1 < a.Z) ? a.nw : 0, sl = has_l ? a.nw : 0, sr = has_r ? a.nw : 0;
        uint32_t* po = a.out + (long long)zi * a.out_ps + (long long)y0 * a.out_rs + 4 * w4;
        uint4 prev = ld4(y0 > 0 ? pc - a.nw : border);
        uint4 cur = ld4(pc);
        const int y1 = min(a.H, y0 + a.my);
        uint32_t cnt = 0;
#pragma unroll 4
        for (int y = y0; y < y1; ++y) {
            const uint4 next = ld4((y + 1 < a.H) ? pc + a.nw : border);
            const uint4 zm = ld4(pm);
            const uint4 zp = ld4(pp);
            const uint32_t l = *pl;
            const uint32_t r = *pr | fix_r_bits;
            const uint4 xm = shl1_4(cur, l), xp = shr1_4(cur, r);
            uint4 v;
            if (ER) v = and4(and4(and4(cur, xm), and4(xp, prev)), and4(and4(next, zm), zp));
            else v = or4(or4(or4(cur, xm), or4(xp, prev)), or4(or4(next, zm), zp));
            v = and4(v, vm);
            *reinterpret_cast<uint4*>(po) = v;
            if (RING) {   // pad words of the padded layout: 4 zero words in front of every row, the tail behind it
                if (w4 == 0) *reinterpret_cast<uint4*>(po - 4) = make_uint4(0, 0, 0, 0);
                if (w4 == nw4 - 1 && a.ring_tail) *reinterpret_cast<uint4*>(po + 4) = make_uint4(0, 0, 0, 0);
            }
            if (COUNT) cnt += popc4(v);
            prev = cur;
            cur = next;
            pc += a.nw; pm += sm; pp += sp; pl += sl; pr += sr; po += a.out_rs;
        }
        if (COUNT && cnt) atomicAdd(&s_cnt[pz], cnt);
    }
    if (COUNT) {
        __syncthreads();
        const int zz = blockIdx.z * a.pz_per_block + threadIdx.x;
        if ((int)threadIdx.x < a.pz_per_block && zz < a.nz && s_cnt[threadIdx.x])
            atomicAdd(a.counts + zz, (unsigned long long)s_cnt[threadIdx.x]);
    }
}

// one stage: planes [z0, z0 + nz) of the compact volume `in` -> out (see MorphArgs)
int t3d_morph_stage(const uint32_t* in, uint32_t* out, int Z, int H, int W, int z0, int nz, int out_rs, long long out_ps,
                    bool erode, bool ring, int ring_tail, unsigned long long* counts, cudaStream_t st)
{
    MorphArgs a;
    a.in = in; a.out = out; a.Z = Z; a.H = H; a.W = W; a.nw = t3d_wpr(W);
    a.z0 = z0; a.nz = nz; a.out_rs = out_rs; a.out_ps = out_ps;
    const int nw4 = a.nw / 4;
    a.lanes_x = nw4 < 256 ? nw4 : 256;
    a.pz_per_block = 256 / a.lanes_x;
    a.my = MY;
    a.ring_tail = ring_tail;
    a.counts = counts;
    dim3 grid((nw4 + a.lanes_x - 1) / a.lanes_x, (H + a.my - 1) / a.my, (nz + a.pz_per_block - 1) / a.pz_per_block);
    const size_t smem = counts ? sizeof(unsigned int) * a.pz_per_block : 0;
    const bool fixw = (W & 127) != 0;
#define T3D_MORPH_LAUNCH(ER, FIX, COUNT, RING) k_morph<ER, FIX, COUNT, RING><<<grid, 256, smem, st>>>(a)
    if (ring) {
        if (erode) { if (fixw) { if (counts) T3D_MORPH_LAUNCH(true, true, true, true); else T3D_MORPH_LAUNCH(true, true, false, true); }
                     else { if (counts) T3D_MORPH_LAUNCH(true, false, true, true); else T3D_MORPH_LAUNCH(true, false, false, true); } }
        else { if (counts) T3D_MORPH_LAUNCH(false, false, true, true); else T3D_MORPH_LAUNCH(false, false, false, true); }
    } else {
        if (erode) { if (fixw) { if (counts) T3D_MORPH_LAUNCH(true, true, true, false); else T3D_MORPH_LAUNCH(true, true, false, false); }
                     else { if (counts) T3D_MORPH_LAUNCH(true, false, true, false); else T3D_MORPH_LAUNCH(true, false, false, false); } }
        else { if (counts) T3D_MORPH_LAUNCH(false, false, true, false); else T3D_MORPH_LAUNCH(false, false, false, false); }
    }
#undef T3D_MORPH_LAUNCH
    T3D_CHECK_LAUNCH("t3d_morph_stage");
    t3d_count_launches(1);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Opening + closing (stages E, D, D, E) in ONE pass over the volume: the grid is read once and the result written once,
// instead of four reads and four writes (the four-launch chain above moves 8 x the volume through DRAM).
//
// A CTA owns a band of `ty` rows (full row width) and marches along z through a chunk of planes.  A thread owns M4_R
// consecutive rows of one uint4 column (128 voxels) and carries, for every stage s, two registers per row:
//     Xp_s = the stage's input at the previous plane,   Q_s = op_s(in-plane cross of the previous plane, input two planes back)
// so that when input plane t arrives
//     stage 0 output (t-1) = op_0(Q_0, I(t))   -> is stage 1's input plane t-1
//     stage 1 output (t-2) = op_1(Q_1, that)   -> stage 2's input ...          stage 3 output (t-4) goes to global memory
// entirely in registers.  Only the in-plane neighbours (rows above / below the thread's rows; the x neighbours come from
// warp shuffles) need another thread's data: the four new input planes are exchanged through shared memory, double
// buffered, ONE barrier per plane.  Input planes arrive through a cp.async ring M4_PF deep.
// Halo: 4 rows above / below the band and 4 planes before / after the chunk are recomputed; rows / planes outside the
// volume hold the neutral element of the stage that reads them (skimage's border rule: erosion sees 1, dilation 0).
// Requires W % 128 == 0 and a row of nw4 = W / 128 uint4 with 32 % nw4 == 0 (W = 128 .. 4096 in powers of two).
// ------------------------------------------------------------------------------------------------
#define M4_R 2
#define M4_PF 4
#define M4_ZC_MAX 128
#define M4_EM 9u          // stage s is an erosion when bit s is set: E, D, D, E

struct Morph4Args {
    const uint32_t* in;          // compact (Z, H, 4 * nw4) volume
    uint32_t* out;               // word (plane z0, row 0, word 0) of the output
    int Z, H, nw4;
    int z0, nz;                  // planes [z0, z0 + nz) are written
    int out_rs;
    long long out_ps;
    int ty, zc;                  // band height, planes per chunk
    int ring_tail;
    unsigned long long* counts;  // counts[z - z0] += set voxels of output plane z (or null)
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v)
{
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void cp_async16s(uint32_t saddr, const void* gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(saddr), "l"(gsrc) : "memory");
}

__global__ void __launch_bounds__(512, 1) k_morph4(Morph4Args a)
{
    extern __shared__ __align__(16) uint32_t m4_smem[];
    __shared__ unsigned int s_cnt[M4_ZC_MAX];
    const int nw4 = a.nw4;
    const uint32_t row_b = 16u * nw4;                            // bytes of a tile row
    const int tid = threadIdx.x, x4 = tid % nw4, rg = tid / nw4;
    const int rows = a.ty + 8;
    const int yl0 = rg * M4_R;                                   // first tile row of this thread
    const int y0 = blockIdx.x * a.ty - 4;                        // volume row of tile row 0
    const int za = a.z0 + blockIdx.y * a.zc, zb = min(a.z0 + a.nz, za + a.zc);
    const uint32_t tile_b = (uint32_t)rows * row_b;
    // shared memory (byte addresses of this thread's first uint4): ring [M4_PF] input planes, xbuf [2][3] inputs of stages 1..3
    const uint32_t me = (uint32_t)__cvta_generic_to_shared(m4_smem) + (uint32_t)yl0 * row_b + 16u * x4;
    const uint32_t xb0 = me + M4_PF * tile_b;
    for (int i = tid; i < M4_ZC_MAX; i += blockDim.x) s_cnt[i] = 0;
    __syncthreads();

    const uint4 ones = splat4(0xffffffffu), zeros = splat4(0u);
    bool rowin[M4_R], rowst[M4_R];
    uint32_t rowout[M4_R];                                       // all ones: the row lies outside the volume
#pragma unroll
    for (int r = 0; r < M4_R; ++r) {
        const int yl = yl0 + r, y = y0 + yl;
        rowin[r] = y >= 0 && y < a.H;
        rowst[r] = rowin[r] && yl >= 4 && yl < 4 + a.ty;
        rowout[r] = rowin[r] ? 0u : 0xffffffffu;
    }
    const long long in_ps = (long long)a.H * 4 * nw4;
    const int t0 = za - 4, t_last = zb + 3;
    const uint32_t* gnext = a.in + (long long)t0 * in_ps + (long long)(y0 + yl0) * 4 * nw4 + 4 * x4;   // this thread's rows of the next plane to fetch
    int pnext = t0;
    const int p_hi = min(a.Z - 1, t_last);

    auto issue = [&](uint32_t saddr) {                           // input plane pnext -> ring slot at saddr
        const bool need = pnext >= 0 && pnext <= p_hi;
#pragma unroll
        for (int r = 0; r < M4_R; ++r) {
            if (need && rowin[r]) cp_async16s(saddr + r * row_b, gnext + r * 4 * nw4);
            else sts128(saddr + r * row_b, (M4_EM & 1u) ? ones : zeros);
        }
        cp_async_commit();
        gnext += in_ps;
        ++pnext;
    };

    uint4 Q[4][M4_R], Xp[4][M4_R];
#pragma unroll
    for (int s = 0; s < 4; ++s)
#pragma unroll
        for (int r = 0; r < M4_R; ++r) { Q[s][r] = zeros; Xp[s][r] = zeros; }

#pragma unroll
    for (int k = 0; k < M4_PF - 1; ++k) issue(me + k * tile_b);
    uint32_t slot_a = me;                                        // ring slot of plane t
    uint32_t slot_w = me + (M4_PF - 1) * tile_b;                 // ring slot the next fetch goes to
    uint32_t xb = xb0, xb_other = xb0 + 3 * tile_b;
    const bool up_ok = yl0 > 0, dn_ok = yl0 + M4_R < rows;
    const unsigned full = 0xffffffffu;
    const uint32_t lfix = x4 == 0 ? 0x80000000u : 0u, rfix = x4 == nw4 - 1 ? 1u : 0u;   // the bit an x neighbour outside the row supplies
    // output pointers of this thread's rows at plane t0 - 4 (advanced every step; dereferenced inside [za, zb) only)
    uint32_t* po = a.out + (long long)(t0 - 4 - a.z0) * a.out_ps + (long long)(y0 + yl0) * a.out_rs + 4 * x4;
    const bool pad_l = x4 == 0, pad_r = x4 == nw4 - 1 && a.ring_tail;
#pragma unroll 2
    for (int t = t0; t <= t_last; ++t) {
        cp_async_wait<M4_PF - 2>();                              // this thread's part of plane t has landed
        uint4 Xn[4][M4_R];
#pragma unroll
        for (int r = 0; r < M4_R; ++r) Xn[0][r] = lds128(slot_a + r * row_b);
        // the chain along z, in registers: stage s turns its new input plane t - s into its output plane t - s - 1
        const int zo = t - 4;
        const bool st_plane = zo >= za && zo < zb;
        uint32_t cnt = 0;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const bool er = (M4_EM >> s) & 1u;
            const int q = t - s - 1;                             // plane of this stage's output = next stage's input
            const uint32_t pout = (q >= 0 && q < a.Z) ? 0u : 0xffffffffu;
#pragma unroll
            for (int r = 0; r < M4_R; ++r) {
                uint4 y = er ? and4(Q[s][r], Xn[s][r]) : or4(Q[s][r], Xn[s][r]);
                if (s < 3) {
                    // outside the volume: the neutral element of the stage that reads it (one LOP3 with the line above)
                    const uint32_t o = pout | rowout[r];
                    const bool ern = (M4_EM >> (s + 1)) & 1u;
                    if (ern) y = or4(y, splat4(o)); else y = and4(y, splat4(~o));
                    Xn[s < 3 ? s + 1 : 3][r] = y;
                } else if (st_plane && rowst[r]) {
                    uint32_t* pr = po + (long long)r * a.out_rs;
                    *reinterpret_cast<uint4*>(pr) = y;
                    if (pad_l) *reinterpret_cast<uint4*>(pr - 4) = zeros;                 // pad words of the padded layout
                    if (pad_r) *reinterpret_cast<uint4*>(pr + 4) = zeros;
                    cnt += popc4(y);
                }
            }
        }
        po += a.out_ps;
        if (a.counts && st_plane) {
            cnt = __reduce_add_sync(full, cnt);
            if ((tid & 31) == 0 && cnt) atomicAdd(&s_cnt[zo - za], cnt);
        }
        // exchange: the new input planes of stages 1..3 (stage 0's is the ring slot itself)
#pragma unroll
        for (int s = 1; s < 4; ++s)
#pragma unroll
            for (int r = 0; r < M4_R; ++r) sts128(xb + (s - 1) * tile_b + r * row_b, Xn[s][r]);
        __syncthreads();
        issue(slot_w);                                           // into the slot read one step ago
        // in-plane cross of the new planes, folded with the previous plane into Q
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const bool er = (M4_EM >> s) & 1u;
            const uint4 nt = er ? ones : zeros;
            const uint32_t base = s == 0 ? slot_a : xb + (s - 1) * tile_b;
            const uint4 up = up_ok ? lds128(base - row_b) : nt;
            const uint4 dn = dn_ok ? lds128(base + M4_R * row_b) : nt;
#pragma unroll
            for (int r = 0; r < M4_R; ++r) {
                const uint4 c = Xn[s][r];
                uint32_t l = __shfl_up_sync(full, c.w, 1), rr = __shfl_down_sync(full, c.x, 1);
                if (er) { l |= lfix; rr |= rfix; } else { l &= ~lfix; rr &= ~rfix; }
                const uint4 above = r == 0 ? up : Xn[s][r > 0 ? r - 1 : 0];
                const uint4 below = r == M4_R - 1 ? dn : Xn[s][r < M4_R - 1 ? r + 1 : 0];
                const uint4 xm = shl1_4(c, l), xp = shr1_4(c, rr);
                uint4 P;
                if (er) P = and4(and4(and4(c, xm), and4(xp, above)), and4(below, Xp[s][r]));
                else P = or4(or4(or4(c, xm), or4(xp, above)), or4(below, Xp[s][r]));
                Q[s][r] = P;
                Xp[s][r] = c;
            }
        }
        slot_w = slot_a;
        slot_a = slot_a == me + (M4_PF - 1) * tile_b ? me : slot_a + tile_b;
        const uint32_t tmp = xb; xb = xb_other; xb_other = tmp;
    }
    cp_async_wait<0>();
    if (a.counts) {
        __syncthreads();
        for (int i = tid; i < zb - za; i += blockDim.x)
            if (s_cnt[i]) atomicAdd(a.counts + (za - a.z0) + i, (unsigned long long)s_cnt[i]);
    }
}

// can the one-pass kernel take this volume?  (else the four-launch chain runs)
bool t3d_morph4_eligible(int Z, int H, int W)
{
    if ((W & 127) || W > 4096 || W < 512) return false;
    const int nw4 = W / 128;
    return (32 % nw4) == 0 && Z >= 1 && H >= 1;
}

// E, D, D, E of planes [z0, z0 + nz) of the compact volume `in` (Z planes) -> out (row stride out_rs, plane stride out_ps words),
// with the pad words of the padded layout cleared (see k_morph RING) and per-plane counts accumulated
int t3d_morph4_launch(const uint32_t* in, uint32_t* out, int Z, int H, int W, int z0, int nz, int out_rs, long long out_ps, int ring_tail,
                      unsigned long long* counts, cudaStream_t st)
{
    Morph4Args a;
    a.in = in; a.out = out; a.Z = Z; a.H = H; a.nw4 = W / 128;
    a.z0 = z0; a.nz = nz; a.out_rs = out_rs; a.out_ps = out_ps; a.ring_tail = ring_tail; a.counts = counts;
    const int nw = 4 * a.nw4;
    // Tile rows: at most 512 threads (rows / M4_R row groups x nw4 columns) and (M4_PF + 6) tiles in ~200 KB of shared memory,
    // a multiple of the rows one warp covers.  Band height and chunk length are picked by a small cost model: a CTA runs
    // zc + 8 steps whose duration grows with the tile rows (throughput) but not below a per-step latency floor; the CTAs of
    // one SM share its throughput.  Tall bands / long chunks waste less halo, short ones fill the machine.
    const int warp_rows = M4_R * (32 / a.nw4);
    int rows_max = 512 / a.nw4 * M4_R;
    const int by_smem = (200 * 1024) / ((M4_PF + 6) * nw * 4);
    if (rows_max > by_smem) rows_max = by_smem;
    rows_max -= rows_max % warp_rows;
    if (rows_max < 9 || rows_max < warp_rows) { t3d_set_error("t3d_morph4: tile does not fit"); return 2; }
    const int sms = T3D_NUM_SMS;
    int rows = 0, zc = 0;
    double best = 1e300;
    for (int rr = rows_max; rr >= 16 && rr >= warp_rows; rr -= warp_rows) {
        const int ty = rr - 8, bands = (H + ty - 1) / ty, thr = rr / M4_R * a.nw4;
        int per_sm = 512 / thr;
        const int smem_fit = (int)((220 * 1024) / ((size_t)(M4_PF + 6) * rr * nw * 4));
        if (per_sm > smem_fit) per_sm = smem_fit;
        if (per_sm < 1) continue;
        static const int zcs[] = {16, 24, 32, 48, 64, 96, 128};
        for (int zi = 0; zi < 7; ++zi) {
            const int c = zcs[zi];
            if (c > M4_ZC_MAX) continue;
            const long long ctas = (long long)bands * ((nz + c - 1) / c);
            const double load = (double)((ctas + sms - 1) / sms) * rr;                                   // tile rows per SM per step
            const double floor_ = 48.0 * (double)((ctas + (long long)sms * per_sm - 1) / ((long long)sms * per_sm));
            const double cost = (load > floor_ ? load : floor_) * (c + 8);
            if (cost < best) { best = cost; rows = rr; zc = c; }
        }
    }
    if (rows == 0) { t3d_set_error("t3d_morph4: no tile configuration"); return 2; }
    a.ty = rows - 8;
    const int bands = (H + a.ty - 1) / a.ty;
    a.zc = zc;
    const int threads = rows / M4_R * a.nw4;
    const size_t smem = (size_t)(M4_PF + 6) * rows * nw * 4;
    if (t3d_first_use_on_device(T3D_ONCE_MORPH4_ATTR))
        T3D_CUDA(cudaFuncSetAttribute(k_morph4, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    dim3 grid(bands, (nz + zc - 1) / zc);
    k_morph4<<<grid, threads, smem, st>>>(a);
    T3D_CHECK_LAUNCH("t3d_morph4");
    t3d_count_launches(1);
    return 0;
}

extern "C" int64_t t3d_morph_scratch_bytes(int Z, int H, int W, int n_stages)
{
    return n_stages > 1 ? (int64_t)Z * H * t3d_wpr(W) * 4 * (n_stages > 2 ? 2 : 1) : 0;
}

// scratch: t3d_morph_scratch_bytes (intermediate stages ping-pong there); in/out must not alias.
extern "C" int t3d_morph(const void* in_bits, void* out_bits, int Z, int H, int W, int n_stages, unsigned erode_mask,
                         void* slice_counts_u64, void* scratch, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_morph: empty volume"); return 2; }
    if (n_stages < 1 || n_stages > 32) { t3d_set_error("t3d_morph: n_stages must be 1..32"); return 2; }
    if (in_bits == out_bits) { t3d_set_error("t3d_morph: in-place is not supported"); return 2; }
    if (n_stages > 1 && !scratch) { t3d_set_error("t3d_morph: scratch required for more than one stage"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int nw = t3d_wpr(W);
    const int64_t vol_words = (int64_t)Z * H * nw;
    if (slice_counts_u64 && t3d_zero_async(slice_counts_u64, sizeof(unsigned long long) * Z, st)) return 1;
    uint32_t* tmp[2] = {(uint32_t*)scratch, (uint32_t*)scratch + vol_words};
    const uint32_t* src = (const uint32_t*)in_bits;
    for (int s = 0; s < n_stages; ++s) {
        const bool last = (s == n_stages - 1);
        uint32_t* dst = last ? (uint32_t*)out_bits : tmp[s & 1];
        unsigned long long* cnt = last ? (unsigned long long*)slice_counts_u64 : nullptr;
        if (int rc = t3d_morph_stage(src, dst, Z, H, W, 0, Z, nw, (long long)H * nw, (erode_mask >> s) & 1u, false, 0, cnt, st)) return rc;
        src = dst;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// per-slice popcounts + bounding box of the set voxels (warp-shuffle tree reductions)
// bbox = {zmin, zmax, ymin, ymax, xmin, xmax}; empty volume leaves {INT_MAX, -1, ...}
// ------------------------------------------------------------------------------------------------
__global__ void k_stats_init(unsigned long long* counts, int Z, int* bbox)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (counts && i < Z) counts[i] = 0;
    if (bbox && i < 6) bbox[i] = (i & 1) ? -1 : 0x7fffffff;
}

#define ST_YSPLIT 4

__global__ void __launch_bounds__(256) k_stats(const uint32_t* __restrict__ bits, int H, int nw,
                                               unsigned long long* __restrict__ counts, int* __restrict__ bbox)
{
    const int z = blockIdx.z;
    const int w = blockIdx.x * 32 + threadIdx.x;
    const int rows_per = (H + ST_YSPLIT - 1) / ST_YSPLIT;
    const int ya = blockIdx.y * rows_per, yb = min(H, ya + rows_per);
    const uint32_t* p = bits + (int64_t)z * H * nw;
    unsigned long long cnt = 0;
    int ymin = 0x7fffffff, ymax = -1, xmin = 0x7fffffff, xmax = -1;
    if (w < nw) {
        for (int y = ya + threadIdx.y; y < yb; y += 8) {
            const uint32_t v = p[(int64_t)y * nw + w];
            if (v) {
                cnt += __popc(v);
                ymin = min(ymin, y); ymax = max(ymax, y);
                xmin = min(xmin, (w << 5) + __ffs(v) - 1);
                xmax = max(xmax, (w << 5) + 31 - __clz(v));
            }
        }
    }
    cnt = warp_sum(cnt);
    ymin = warp_min(ymin); xmin = warp_min(xmin); ymax = warp_max(ymax); xmax = warp_max(xmax);
    __shared__ unsigned long long sc[8];
    __shared__ int sb[8][4];
    const int wi = threadIdx.y;
    if (threadIdx.x == 0) { sc[wi] = cnt; sb[wi][0] = ymin; sb[wi][1] = ymax; sb[wi][2] = xmin; sb[wi][3] = xmax; }
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        for (int k = 1; k < 8; ++k) {
            cnt += sc[k]; ymin = min(ymin, sb[k][0]); ymax = max(ymax, sb[k][1]);
            xmin = min(xmin, sb[k][2]); xmax = max(xmax, sb[k][3]);
        }
        if (cnt) {
            if (counts) atomicAdd(counts + z, cnt);
            if (bbox) {
                atomicMin(bbox + 0, z); atomicMax(bbox + 1, z);
                atomicMin(bbox + 2, ymin); atomicMax(bbox + 3, ymax);
                atomicMin(bbox + 4, xmin); atomicMax(bbox + 5, xmax);
            }
        }
    }
}

extern "C" int t3d_volume_stats(const void* bits, int Z, int H, int W, void* slice_counts_u64, void* bbox_i32x6,
                                void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_volume_stats: empty volume"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int nw = t3d_wpr(W);
    const int n_init = Z > 6 ? Z : 6;
    k_stats_init<<<(n_init + 255) / 256, 256, 0, st>>>((unsigned long long*)slice_counts_u64, Z, (int*)bbox_i32x6);
    dim3 grid((nw + 31) / 32, ST_YSPLIT, Z), block(32, 8);
    k_stats<<<grid, block, 0, st>>>((const uint32_t*)bits, H, nw, (unsigned long long*)slice_counts_u64, (int*)bbox_i32x6);
    T3D_CHECK_LAUNCH("t3d_volume_stats");
    t3d_count_launches(2);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// point cloud (voxel_processor.py:99-127): np.where order (C order), every `sub`-th set voxel,
// z -> cum[z] + depth[z]/2, y*mm_y, x*mm_x, float64 (N,3).
// Two kernels: per-row popcounts (then an exclusive scan by the caller, t3d_scan_u32) and emission.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_row_popc(const uint32_t* __restrict__ bits, int64_t n_rows, int nw,
                                                  uint32_t* __restrict__ row_counts)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n_rows) return;
    uint32_t c = 0;
    for (int w = lane_id(); w < nw; w += 32) c += __popc(bits[row * nw + w]);
    c = warp_sum(c);
    if (lane_id() == 0) row_counts[row] = c;
}

__global__ void __launch_bounds__(256) k_point_cloud(const uint32_t* __restrict__ bits, int64_t n_rows, int H, int nw,
                                                     const unsigned long long* __restrict__ row_base, int sub,
                                                     const double* __restrict__ zc_mm, double mm_y, double mm_x,
                                                     double* __restrict__ out)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n_rows) return;
    const int z = (int)(row / H), y = (int)(row - (int64_t)z * H);
    unsigned long long base = row_base[row];
    const uint32_t l = lane_id();
    for (int w0 = 0; w0 < nw; w0 += 32) {
        const int w = w0 + l;
        uint32_t v = (w < nw) ? bits[row * nw + w] : 0u;
        const uint32_t c = __popc(v);
        const uint32_t incl = warp_incl_scan(c);
        unsigned long long idx = base + incl - c;
        while (v) {
            const int b = __ffs(v) - 1;
            v &= v - 1;
            if (idx % (unsigned)sub == 0) {
                double* o = out + 3 * (idx / (unsigned)sub);
                o[0] = zc_mm[z];
                o[1] = (double)y * mm_y;
                o[2] = (double)((w << 5) + b) * mm_x;
            }
            ++idx;
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
}

extern "C" int t3d_row_popcounts(const void* bits, int Z, int H, int W, void* row_counts_u32, void* stream)
{
    const int64_t rows = (int64_t)Z * H;
    if (rows <= 0) return 0;
    k_row_popc<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const uint32_t*)bits, rows,
                                                                                      t3d_wpr(W), (uint32_t*)row_counts_u32);
    T3D_CHECK_LAUNCH("t3d_row_popcounts");
    t3d_count_launches(1);
    return 0;
}

extern "C" int t3d_point_cloud_emit(const void* bits, int Z, int H, int W, const void* row_base_u64, int subsample,
                                    const void* z_centre_mm_f64, double mm_per_pixel_y, double mm_per_pixel_x,
                                    void* out_f64, void* stream)
{
    const int64_t rows = (int64_t)Z * H;
    if (rows <= 0) return 0;
    if (subsample < 1) subsample = 1;
    k_point_cloud<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint32_t*)bits, rows, H, t3d_wpr(W), (const unsigned long long*)row_base_u64, subsample,
        (const double*)z_centre_mm_f64, mm_per_pixel_y, mm_per_pixel_x, (double*)out_f64);
    T3D_CHECK_LAUNCH("t3d_point_cloud_emit");
    t3d_count_launches(1);
    return 0;
}
