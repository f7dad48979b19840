// t3d_common.cuh -- shared helpers for the sm_100a kernels behind include/t3d.h.
//
// Volume layout everywhere: C-contiguous (Z, H, W); occupancy is bit-packed along x, LSB first:
//   word(z, y, w) bit i  <=>  voxel (z, y, x = 32*w + i),   row stride = words_per_row(W) = ceil(W/32) rounded up
//   to a multiple of 4 words, so every row starts 16-byte aligned and kernels move uint4 (128 voxels) per thread.
// Invariant: bits at x >= W (tail of the last word and the padding words) are zero.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

// number of SMs of the current device (queried once per device; 148 on a B200); grids of the persistent-style kernels
// are sized in multiples of it
int t3d_num_sms(void);
#define T3D_NUM_SMS (t3d_num_sms())
// per-device "done once" flags for state that lives per device (constant memory, function attributes): returns true the
// first time it is called for (slot, current device)
bool t3d_first_use_on_device(int slot);
enum { T3D_ONCE_FILL_HOLES_ATTR = 0, T3D_ONCE_MC_LUTS = 1, T3D_ONCE_SORT_ATTR = 2, T3D_ONCE_MORPH4_ATTR = 3, T3D_ONCE_SLOTS = 8 };

extern "C" void t3d_set_error(const char* fmt, ...);
extern "C" void t3d_count_launches(int n);  // bookkeeping for bench.py's gpu_launches (our kernels only)
// Zeroing of small counters / scan descriptors / bitmaps.  The single-enqueue entry points (t3d_pipeline.cu) zero every
// such buffer of a step with ONE kernel up front and register the ranges; t3d_zero_async then skips the ranges it finds
// registered (each memset would be its own node on the critical path of the captured graph) and memsets anything else.
int t3d_zero_async(void* p, size_t n, cudaStream_t st);
void t3d_prezero_register(const void* p, size_t n);
void t3d_prezero_clear(void);
void t3d_canonicalize_structured_zero_range(int64_t V, int64_t F, uint32_t cap_z, uint32_t cap_g0, int Zs, int64_t* offset,
                                            int64_t* size);

#define T3D_CHECK_LAUNCH(name)                                                                   \
    do {                                                                                         \
        cudaError_t e__ = cudaGetLastError();                                                    \
        if (e__ != cudaSuccess) {                                                                \
            t3d_set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));               \
            return 1;                                                                            \
        }                                                                                        \
    } while (0)

#define T3D_CUDA(call)                                                                           \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            t3d_set_error("%s failed: %s", #call, cudaGetErrorString(e__));                      \
            return 1;                                                                            \
        }                                                                                        \
    } while (0)

static inline int t3d_wpr(int W) { return (((W + 31) >> 5) + 3) & ~3; }
static inline int t3d_wvalid(int W) { return (W + 31) >> 5; }  // words that hold at least one voxel

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

// mask of valid bits (x < W) of word w in a row of width W
__device__ __forceinline__ uint32_t valid_mask(int w, int W)
{
    const int rem = W - (w << 5);
    if (rem >= 32) return 0xffffffffu;
    if (rem <= 0) return 0u;
    return (1u << rem) - 1u;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ int warp_min(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int warp_max(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// inclusive warp scan (Kogge-Stone over shuffles)
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v)
{
    const uint32_t l = lane_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (l >= (uint32_t)o) v += t;
    }
    return v;
}

// streaming 128-bit loads/stores (no L1 allocation: every input byte is touched once)
__device__ __forceinline__ uint4 ld_stream_u4(const void* p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream_u4(void* p, uint4 v)
{
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
                 "r"(v.z), "r"(v.w)
                 : "memory");
}

// 4 bytes -> 4 bits: bit k = (byte k >= thr)
__device__ __forceinline__ uint32_t ge4(uint32_t v, uint32_t thr4)
{
    const uint32_t m = __vcmpgeu4(v, thr4) & 0x80808080u;  // bit 7 of each byte
    return (m * 0x00204081u) >> 28;
}
// 16 bytes -> 16 bits
__device__ __forceinline__ uint32_t ge16(uint4 v, uint32_t thr4)
{
    return ge4(v.x, thr4) | (ge4(v.y, thr4) << 4) | (ge4(v.z, thr4) << 8) | (ge4(v.w, thr4) << 12);
}
// 4 bits -> 4 bytes of 0/1
__device__ __forceinline__ uint32_t expand4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }

__device__ __forceinline__ uint4 and4(uint4 a, uint4 b) { return make_uint4(a.x & b.x, a.y & b.y, a.z & b.z, a.w & b.w); }
__device__ __forceinline__ uint4 or4(uint4 a, uint4 b) { return make_uint4(a.x | b.x, a.y | b.y, a.z | b.z, a.w | b.w); }
__device__ __forceinline__ uint4 splat4(uint32_t v) { return make_uint4(v, v, v, v); }
__device__ __forceinline__ uint32_t popc4(uint4 a) { return __popc(a.x) + __popc(a.y) + __popc(a.z) + __popc(a.w); }
// valid-bit masks of the four words of uint4 column w4 in a row of width W
__device__ __forceinline__ uint4 valid_mask4(int w4, int W)
{
    return make_uint4(valid_mask(4 * w4, W), valid_mask(4 * w4 + 1, W), valid_mask(4 * w4 + 2, W), valid_mask(4 * w4 + 3, W));
}
// x-1 / x+1 neighbours of the 128 voxels of a uint4: l = word to the left of .x, r = word to the right of .w
__device__ __forceinline__ uint4 shl1_4(uint4 c, uint32_t l)
{
    return make_uint4(__funnelshift_l(l, c.x, 1), __funnelshift_l(c.x, c.y, 1), __funnelshift_l(c.y, c.z, 1), __funnelshift_l(c.z, c.w, 1));
}
__device__ __forceinline__ uint4 shr1_4(uint4 c, uint32_t r)
{
    return make_uint4(__funnelshift_r(c.x, c.y, 1), __funnelshift_r(c.y, c.z, 1), __funnelshift_r(c.z, c.w, 1), __funnelshift_r(c.w, r, 1));
}

// Sizes that only the device knows (number of active words, vertices, faces ...) are passed as a capacity plus an
// optional pointer to the true value in device memory, so that a whole step can be enqueued (and graph-captured)
// without a host round trip.  n = min(cap, *p) when p is given, else cap.
__device__ __forceinline__ int64_t dev_n(int64_t cap, const unsigned long long* p)
{
    if (!p) return cap;
    const unsigned long long v = *p;
    return v < (unsigned long long)cap ? (int64_t)v : cap;
}

// ---- internal launchers shared between translation units (t3d_voxel.cu) -----------------------------------------------
// one 6-connected erosion / dilation stage: planes [z0, z0 + nz) of the compact volume `in` -> `out` (pointing at the word
// of plane z0, row 0, word 0) with its own row / plane strides.  ring: the output is the padded-storage layout, the
// stage also clears the 4 pad words in front of every row it writes and ring_tail (0 / 1) uint4 behind it.
int t3d_morph_stage(const uint32_t* in, uint32_t* out, int Z, int H, int W, int z0, int nz, int out_rs, long long out_ps,
                    bool erode, bool ring, int ring_tail, unsigned long long* counts, cudaStream_t st);
// the four stages E, D, D, E in one pass (k_morph4, t3d_voxel.cu): eligibility of a volume and the launch; arguments as for a
// ring + counts t3d_morph_stage
bool t3d_morph4_eligible(int Z, int H, int W);
int t3d_morph4_launch(const uint32_t* in, uint32_t* out, int Z, int H, int W, int z0, int nz, int out_rs, long long out_ps, int ring_tail,
                      unsigned long long* counts, cudaStream_t st);
// one-shot: the next canonicalisation of this thread waits for `e` before its first kernel that reads the faces (t3d_surface.cu)
void t3d_canon_faces_ready_event(cudaEvent_t e);
bool t3d_canon_faces_ready_pending();
// fused pack + z gap fill + per-slice counts + extrema (see t3d_voxel.cu)
bool t3d_pack_gap_supported(const void* masks_u8, int Z, int H, int W, int threshold);
int t3d_pack_gap_launch(const void* masks_u8, int Z, int H, int W, int threshold, void* out, unsigned long long* counts,
                        unsigned int* bbox_t, int skip_ends, cudaStream_t st, int z_bias = 0);
// extrema of a few planes in the same transformed form (plane p of the call = plane z_bias + p)
int t3d_bbox_t_planes_launch(const uint32_t* bits, int n_planes, int H, int W, int z_bias, unsigned int* bbox_t, cudaStream_t st);
int t3d_close_ends_fixup_launch(const void* masks_u8, int Z, int H, int W, int threshold, const void* filled0, const void* filledT,
                                void* out, unsigned long long* counts, cudaStream_t st);
