// t3d_pipeline.cu -- the whole hot path as ONE enqueue: mask stack -> voxel grid -> smoothing -> canonical mesh + volumes.
//
// Order of work = the reference orchestrator's (tomography_3d_reconstruction.py:88-140, 194-229), every stage one of
// the kernels of this library.  Nothing here synchronises with the host: data-dependent sizes (active words, vertices,
// faces) stay in device memory, all buffers are capacity-sized by the caller and nothing is written beyond a
// capacity (the overflow flags in the result block tell the caller to retry with larger capacities).  The call can
// therefore be captured in a CUDA graph and replayed with a single launch; hole filling of the two end slices and the
// bounding-box reduction run on an internal side stream, forked and joined with events (also capturable).
#include <stdint.h>

#include <stdlib.h>

#include <nvtx3/nvToolsExt.h>

#include "t3d.h"
#include "t3d_field.cuh"

// NVTX ranges per stage of the enqueue (host side: they bracket the launches of a stage, and show up in an Nsight Systems
// trace of a step next to the kernels they enqueue; header-only NVTX3, a no-op without an attached tool)
struct NvtxRange {
    bool open;
    explicit NvtxRange(const char* name) : open(true) { nvtxRangePushA(name); }
    void end() { if (open) { nvtxRangePop(); open = false; } }
    ~NvtxRange() { end(); }
};

// result block (uint64 slots); keep in sync with include/t3d.h and pipeline.py
enum {
    R_NACTIVE = 0, R_NX = 1, R_NY = 2, R_NZ = 3, R_NT = 4, R_VCANON = 5, R_FCANON = 6, R_UNVERIFIED = 7, R_OVERFLOW = 8,
    R_NAMBIGUOUS = 9, R_NEXACT = 10, R_VOLUME_F64 = 11, R_AREA_F64 = 12, R_BBOX_I32X6 = 13 /* 3 slots */, R_VRAW = 16, R_NEXC = 17,
    R_NGHOST = 18, R_NLEAD = 19, R_NG0 = 25,
    R_COUNTS = 32  /* Zx raw per-slice counts, then Zx smoothed per-slice counts */
};

#define EXC_CAP (1u << 20)  // capacity of the list of sign words that need the exact field evaluation
#define SURF_HALO 3         // smoothed planes the surface stage reads beyond the owned ones (Gaussian radius 2 + upper cube corner)

#define S_XPAD 128          // zero voxels in front of every row of the padded-storage sign volume (4 words: rows stay 16-byte aligned)

static inline int64_t al(int64_t x) { return (x + 255) & ~(int64_t)255; }

// Opening then closing (stages E,D,D,E) leaves no voxel whose six face neighbours all disagree with it: an opened set is a
// union of crosses (every member touches another member), closing only adds voxels next to the dilated set, and a cleared
// voxel with six set neighbours would have survived the closing's erosion.  With the zero pad ring around it the sign of
// (gaussian(0.5) - 0.5) is then the padded occupancy itself (see t3d_surface.cu), so the last erosion writes the sign
// volume directly, in a padded STORAGE layout: (Zl+2, H+2, wpr(W + S_XPAD + 1)) with the occupancy at plane 1, row 1,
// word 4 -- no separate field-sign pass, no separately stored smoothed volume.
static bool fast_surface(int n_stages, unsigned erode_mask, int pad, int Zx, int H, int W)
{
    return pad == 1 && n_stages == 4 && (erode_mask & 15u) == 9u && Zx >= 2 && H >= 2 && W >= 2;
}

struct Layout {
    int64_t bitsA, bitsB, bitsC, morph, fill, sign, exc, ballots, chunkbase, scan1, aw_idx, aw_cnt, aw_base, scan2, vkeys, verts_raw,
        faces_raw, canon, measure, total;
};

// Zx: planes of the voxel buffers (own slices + halos); Zl: planes the surface stage reads
static Layout make_layout(int Zx, int Zl, int H, int W, int pad, uint32_t capNA, uint32_t capV, uint32_t capF, uint32_t capZ,
                          uint32_t capG0, int n_stages, bool own_bitsA, bool fast)
{
    Layout L;
    const int64_t nw = t3d_words_per_row(W), vol = (int64_t)Zx * H * nw * 4;
    const int Zp = Zl + 2 * pad, Hp = H + 2 * pad, Wp = fast ? W + S_XPAD + 1 : W + 2 * pad;
    const int64_t nwp = t3d_words_per_row(Wp), n_chunks = t3d_mc_num_chunks(Zp, Hp, Wp);
    int64_t o = 0;
    L.bitsA = o; o += own_bitsA ? al(vol) : 0;
    L.bitsB = o; o += al(vol);
    L.bitsC = o; o += fast ? 0 : al(vol);       // smoothed volume (the fast path writes it straight into the sign volume)
    L.morph = o; o += al(t3d_morph_scratch_bytes(Zx, H, W, n_stages));
    L.fill = o; o += al(t3d_fill_holes_scratch_bytes(2, H, W));
    L.sign = o; o += al((int64_t)Zp * Hp * nwp * 4);
    L.exc = o; o += al((int64_t)EXC_CAP * 8);
    L.ballots = o; o += al(n_chunks * 4);
    L.chunkbase = o; o += al(n_chunks * 4);
    L.scan1 = o; o += al(t3d_scan_workspace_bytes(n_chunks, 1));
    L.aw_idx = o; o += al((int64_t)capNA * 4);
    L.aw_cnt = o; o += al((int64_t)capNA * 16);
    L.aw_base = o; o += al((int64_t)capNA * 16);
    L.scan2 = o; o += al(t3d_scan_workspace_bytes(capNA, 4));
    L.vkeys = o; o += al((int64_t)capV * 8);
    L.verts_raw = o; o += al((int64_t)capV * 12);
    L.faces_raw = o; o += al((int64_t)capF * 12);
    L.canon = o; o += al(capZ ? t3d_canonicalize_structured_workspace_bytes(capV, capF, capZ, capG0, Zp)
                              : t3d_canonicalize_fast_workspace_bytes(capV, capF));
    L.measure = o; o += al(t3d_mesh_measure_workspace_bytes());
    L.total = o;
    return L;
}

extern "C" int64_t t3d_reconstruct_workspace_bytes(int Z, int H, int W, int add_padding, int n_stages, uint32_t cap_active,
                                                   uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0)
{
    // (sized for whichever of the two surface paths needs more; which one runs also depends on the erode mask)
    const int pad = add_padding ? 1 : 0;
    const int64_t a = make_layout(Z, Z, H, W, pad, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, n_stages, true, false).total;
    const int64_t b = make_layout(Z, Z, H, W, pad, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, n_stages, true, true).total;
    return a > b ? a : b;
}

extern "C" int64_t t3d_reconstruct_results_len(int Z) { return R_COUNTS + 2 * (int64_t)Z; }

static inline int imin(int a, int b) { return a < b ? a : b; }

extern "C" int64_t t3d_reconstruct_slab_workspace_bytes(int halo_lo, int n_own, int halo_hi, int H, int W, int add_padding,
                                                        int n_stages, uint32_t cap_active, uint32_t cap_verts, uint32_t cap_faces,
                                                        uint32_t cap_zverts, uint32_t cap_g0)
{
    const int Zx = halo_lo + n_own + halo_hi, Zl = imin(SURF_HALO, halo_lo) + n_own + imin(SURF_HALO, halo_hi);
    const int pad = add_padding ? 1 : 0;
    const int64_t a = make_layout(Zx, Zl, H, W, pad, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, n_stages, false, false).total;
    const int64_t b = make_layout(Zx, Zl, H, W, pad, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, n_stages, false, true).total;
    return a > b ? a : b;
}

__global__ void k_finalize_sizes(unsigned long long* r, unsigned long long capNA, unsigned long long capV, unsigned long long capF,
                                 int bbox_transformed)
{
    if (bbox_transformed) {   // k_pack_gap accumulates {INT_MAX - min, max + 1}: back to {min (INT_MAX if empty), max (-1 if empty)}
        unsigned int* t = (unsigned int*)(r + R_BBOX_I32X6);
        int* b = (int*)(r + R_BBOX_I32X6);
        for (int k = 0; k < 3; ++k) {
            const unsigned lo = t[2 * k], hi = t[2 * k + 1];
            b[2 * k] = 0x7fffffff - (int)lo;
            b[2 * k + 1] = (int)hi - 1;
        }
    }
    unsigned long long of8 = (r[R_NEXC] > EXC_CAP) ? 8ull : 0ull;
    const unsigned long long v = r[R_NX] + r[R_NY] + r[R_NZ];
    r[R_VRAW] = v;
    unsigned long long of = 0;
    if (r[R_NACTIVE] > capNA) of |= 1;
    if (v > capV) of |= 2;
    if (r[R_NT] > capF) of |= 4;
    r[R_OVERFLOW] = of | of8;
    if (of | of8) {
        // the emit kernel writes nothing on overflow: make every later stage see an empty mesh instead of stale indices
        // (the sizes that did not fit are kept in slots 20..24 for the caller's next capacity guess)
        for (int k = 0; k < 5; ++k) { r[20 + k] = r[R_NACTIVE + k]; r[R_NACTIVE + k] = 0; }
        r[R_VRAW] = 0;
    }
}

// Number of canonical vertices whose z equals zq[w] (warp w): the list is sorted by z first, so this is
// upper_bound - lower_bound, found by a 32-ary search (one probe per lane and step).
__global__ void k_count_plane_vertices(const float* __restrict__ verts, const unsigned long long* n_dev, float z_ghost, float z_lead,
                                       int want_ghost, int want_lead, unsigned long long* out_ghost, unsigned long long* out_lead)
{
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool want = w == 0 ? want_ghost != 0 : want_lead != 0;
    unsigned long long* out = w == 0 ? out_ghost : out_lead;
    if (!want) {
        if (lane == 0) *out = 0;
        return;
    }
    const float zq = w == 0 ? z_ghost : z_lead;
    const long long n = (long long)*n_dev;
    long long bound[2];
    for (int upper = 0; upper < 2; ++upper) {
        // smallest i with z[i] >= zq (lower) / z[i] > zq (upper)
        long long lo = 0, hi = n;   // answer in [lo, hi]
        while (hi - lo > 0) {
            const long long span = hi - lo, step = (span + 31) / 32;
            const long long i = lo + (long long)lane * step;
            bool before = false;     // element i is before the answer
            if (i < hi) {
                const float z = verts[3 * i];
                before = upper ? (z <= zq) : (z < zq);
            }
            const unsigned b = __ballot_sync(0xffffffffu, before);
            const int k = __popc(b);   // lanes 0..k-1 are before (monotone)
            if (k == 0) { hi = lo; break; }
            const long long last_before = lo + (long long)(k - 1) * step;
            const long long nlo = last_before + 1;
            const long long nhi = (k < 32 && lo + (long long)k * step < hi) ? lo + (long long)k * step : hi;
            lo = nlo; hi = nhi;
        }
        bound[upper] = lo;
    }
    if (lane == 0) *out = (unsigned long long)(bound[1] - bound[0]);
}

#define N_SIDE_EVENTS 8
struct SideStream {
    cudaStream_t s = nullptr;
    cudaEvent_t e[N_SIDE_EVENTS] = {};
};
static SideStream g_side[64];

static int side_for_current_device(SideStream** out)
{
    int dev = 0;
    T3D_CUDA(cudaGetDevice(&dev));
    SideStream& s = g_side[dev & 63];
    if (!s.s) {
        // highest priority: the side stream carries short dependent chains (hole filling, the z-edge sort) that must not
        // queue behind the large grids of the main stream
        int prio_lo = 0, prio_hi = 0;
        T3D_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        T3D_CUDA(cudaStreamCreateWithPriority(&s.s, cudaStreamNonBlocking, prio_hi));
        for (int k = 0; k < N_SIDE_EVENTS; ++k) T3D_CUDA(cudaEventCreateWithFlags(&s.e[k], cudaEventDisableTiming));
    }
    *out = &s;
    return 0;
}

#define RUN(call) do { if (int rc__ = (call)) return rc__; } while (0)

// every counter / scan descriptor / bitmap a step needs zeroed, in one node of the graph (see t3d_zero_async)
struct ZeroSet {
    uint4* p[6];
    unsigned long long n16[6];   // sizes in 16-byte units
    int n;
};
__global__ void __launch_bounds__(256) k_zero_ranges(ZeroSet z)
{
    for (int k = 0; k < z.n; ++k)
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < z.n16[k];
             i += (unsigned long long)gridDim.x * blockDim.x)
            z.p[k][i] = make_uint4(0, 0, 0, 0);
}
struct PrezeroGuard {
    PrezeroGuard() { t3d_prezero_clear(); }
    ~PrezeroGuard() { t3d_prezero_clear(); }
    ZeroSet z{};
    void add(void* p, size_t bytes)
    {
        const size_t n16 = bytes / 16;       // ranges are 16-byte aligned; a tail that is not a multiple stays a memset
        if (!n16 || z.n >= 6 || ((uintptr_t)p & 15)) return;
        z.p[z.n] = (uint4*)p; z.n16[z.n] = n16; ++z.n;
        t3d_prezero_register(p, n16 * 16);
    }
    int launch(cudaStream_t st)
    {
        if (!z.n) return 0;
        k_zero_ranges<<<T3D_NUM_SMS * 2, 256, 0, st>>>(z);
        T3D_CHECK_LAUNCH("k_zero_ranges");
        t3d_count_launches(1);
        return 0;
    }
};

struct SlabGeom {
    int hl, n, hh;        // halo planes below / own planes / halo planes above in the voxel buffers
    int z_begin, z_end;   // owned planes of the local padded sign volume (-1 = to the end)
    int z_offset;         // global un-padded plane index of local surface plane 0
    int want_ghost, want_lead;
    float z_ghost, z_lead;
};

// zero ring of the padded-storage sign volume: planes 0 and Zs-1, rows 0 and Hs-1 of the planes between them (the pad
// words of the other rows are written by the morphology stage that fills them)
__global__ void __launch_bounds__(256) k_zero_ring(uint4* __restrict__ S, int Zs, int Hs, int nws4)
{
    const long long plane4 = (long long)Hs * nws4;
    const long long nA = 2 * plane4, nB = (long long)(Zs - 2) * 2 * nws4;
    const uint4 zero = make_uint4(0, 0, 0, 0);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nA + nB; i += (long long)gridDim.x * blockDim.x) {
        if (i < nA) {
            S[i < plane4 ? i : (long long)(Zs - 1) * plane4 + (i - plane4)] = zero;
        } else {
            const long long j = i - nA;
            const long long z = 1 + j / (2 * nws4);
            const int r = (int)(j % (2 * nws4));
            S[z * plane4 + (long long)(r < nws4 ? 0 : Hs - 1) * nws4 + (r % nws4)] = zero;
        }
    }
}

// Debug timeline (T3D_STAGE_EVENTS=1, eager launches only): events on the main stream at the stage boundaries of
// reconstruct_core; the elapsed times between them (which include every wait on the side stream) go to stderr after a
// stream synchronize.  Off by default; never active while the stream is being captured.
struct StageMarks {
    enum { N = 12 };
    cudaEvent_t ev[N];
    const char* name[N];
    int n = 0;
    bool on = false;
    void begin(cudaStream_t st)
    {
        static const bool want = getenv("T3D_STAGE_EVENTS") != nullptr;
        on = false;
        if (!want) return;
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return;
        on = true; n = 0;
    }
    void mark(const char* what, cudaStream_t st)
    {
        if (!on || n >= N) return;
        static thread_local cudaEvent_t pool[N] = {};
        if (!pool[n]) cudaEventCreate(&pool[n]);
        ev[n] = pool[n]; name[n] = what;
        cudaEventRecord(ev[n], st);
        ++n;
    }
    void report(cudaStream_t st)
    {
        if (!on) return;
        cudaStreamSynchronize(st);
        fprintf(stderr, "[t3d stages]");
        for (int i = 1; i < n; ++i) { float ms = 0; cudaEventElapsedTime(&ms, ev[i - 1], ev[i]); fprintf(stderr, " %s %.1f us |", name[i], 1e3f * ms); }
        float tot = 0; if (n > 1) cudaEventElapsedTime(&tot, ev[0], ev[n - 1]);
        fprintf(stderr, " total %.1f us\n", 1e3f * tot);
    }
};

// Everything after the voxel grid exists: smoothing, surface, canonical mesh, measures.  `grid` = bit volume of
// Zx = hl + n + hh planes after close_ends (bitsB of the layout), counts already in R[R_COUNTS .. +Zx).
// bbox_state: 0 = compute the bounding box of the owned planes here (side stream), 1 = already in R (int32 x 6),
// 2 = in R in k_pack_gap's transformed form (converted by k_finalize_sizes).
static int reconstruct_core(const uint32_t* grid, const SlabGeom& g, int H, int W, int n_stages, unsigned erode_mask, int pad,
                            const double* weights3_host, const void* cum_f64, const void* adj_f64, int n_cum, double mm_y,
                            double mm_x, int scale_in_f64, uint32_t cap_active, uint32_t cap_verts, uint32_t cap_faces,
                            uint32_t cap_zverts, uint32_t cap_g0, int zkey_bits, void* verts_out_f32, void* faces_out_i64,
                            unsigned long long* R, char* ws, const Layout& L, bool fast, int bbox_state, SideStream* side, cudaStream_t st)
{
    const int Zx = g.hl + g.n + g.hh;
    const int64_t nw = t3d_words_per_row(W), plane_words = (int64_t)H * nw, vol_words = (int64_t)Zx * plane_words;
    const int sl = imin(SURF_HALO, g.hl), sh = imin(SURF_HALO, g.hh), Zl = sl + g.n + sh;
    const int Zp = Zl + 2 * pad, Hp = H + 2 * pad, Wp = fast ? W + S_XPAD + 1 : W + 2 * pad;
    const int64_t n_chunks = t3d_mc_num_chunks(Zp, Hp, Wp);

    // side stream: bounding box of the owned planes of the raw grid (unless the pack kernel already did it) and the zero
    // ring of the padded sign volume; joined before the cube flags / the measures
    NvtxRange r_smooth("t3d:smooth_voxel_data");
    StageMarks marks;
    marks.begin(st);
    marks.mark("start", st);
    (void)t3d_canon_faces_ready_pending();   // (nothing registered by an earlier, failed step)
    T3D_CUDA(cudaEventRecord(side->e[2], st));
    T3D_CUDA(cudaStreamWaitEvent(side->s, side->e[2], 0));
    if (bbox_state == 0)
        RUN(t3d_volume_stats(grid + (int64_t)g.hl * plane_words, g.n, H, W, nullptr, R + R_BBOX_I32X6, side->s));
    OccView view;   // the smoothed occupancy the vertex kernel evaluates the field on
    int x_off = 0;
    if (fast) {
        const int nws = (int)t3d_words_per_row(Wp);
        uint32_t* S = (uint32_t*)(ws + L.sign);
        const long long s_ps = (long long)Hp * nws;
        {
            const long long items = 2 * (long long)Hp * (nws / 4) + (long long)(Zp - 2) * 2 * (nws / 4);
            long long blocks = (items + 255) / 256;
            if (blocks > (long long)T3D_NUM_SMS * 8) blocks = (long long)T3D_NUM_SMS * 8;
            k_zero_ring<<<(unsigned)(blocks < 1 ? 1 : blocks), 256, 0, side->s>>>((uint4*)S, Zp, Hp, nws / 4);
            t3d_count_launches(1);
        }
        T3D_CUDA(cudaEventRecord(side->e[3], side->s));
        // ---- smooth_voxel_data: E, D, D on compact scratch volumes, the last E straight into the padded sign volume
        uint32_t* tA = (uint32_t*)(ws + L.morph);
        uint32_t* tB = tA + vol_words;
        uint32_t* S_origin = S + s_ps + nws + S_XPAD / 32;   // word of (plane 1, row 1, x = S_XPAD)
        const int z0 = g.hl - sl;
        const int ring_tail = (nws - (int)nw - S_XPAD / 32) / 4;
        // (An L2-tiled variant of the four-launch chain -- chunks of planes with the intermediate stages kept in L2 -- was
        // measured slower than the untiled chain at 512x4096x4096, profiles/r02_morph_ztile_sweep_c4slab.txt, and removed.)
        if (t3d_morph4_eligible(Zx, H, W)) {
            // the four stages in one pass: grid read once, sign volume written once
            RUN(t3d_morph4_launch(grid, S_origin, Zx, H, W, z0, Zl, nws, s_ps, ring_tail, R + R_COUNTS + Zx + z0, st));
        } else {
            RUN(t3d_morph_stage(grid, tA, Zx, H, W, 0, Zx, (int)nw, plane_words, true, false, 0, nullptr, st));
            RUN(t3d_morph_stage(tA, tB, Zx, H, W, 0, Zx, (int)nw, plane_words, false, false, 0, nullptr, st));
            RUN(t3d_morph_stage(tB, tA, Zx, H, W, 0, Zx, (int)nw, plane_words, false, false, 0, nullptr, st));
            RUN(t3d_morph_stage(tA, S_origin, Zx, H, W, z0, Zl, nws, s_ps, true, true, ring_tail, R + R_COUNTS + Zx + z0, st));
        }
        view = t3d_make_view_strided(S_origin, Zl, H, W, nws, s_ps, 1, 1, weights3_host);
        x_off = S_XPAD - 1;
        T3D_CUDA(cudaStreamWaitEvent(st, side->e[3], 0));   // ring zeroed
    } else {
        T3D_CUDA(cudaEventRecord(side->e[3], side->s));
        uint32_t* bitsC = (uint32_t*)(ws + L.bitsC);
        // ---- smooth_voxel_data
        const uint32_t* smoothed = grid;
        if (n_stages > 0) {
            RUN(t3d_morph(grid, bitsC, Zx, H, W, n_stages, erode_mask, R + R_COUNTS + Zx, ws + L.morph, st));
            smoothed = bitsC;
        } else {
            T3D_CUDA(cudaMemcpyAsync(R + R_COUNTS + Zx, R + R_COUNTS, sizeof(unsigned long long) * Zx, cudaMemcpyDeviceToDevice, st));
        }
        const uint32_t* surf = smoothed + (int64_t)(g.hl - sl) * plane_words;
        // ---- field sign: pad + gaussian + `> 0.5` (exceptions evaluated exactly)
        RUN(t3d_field_sign_lean(surf, Zl, H, W, pad, weights3_host, ws + L.sign, R + R_NEXACT, ws + L.exc, EXC_CAP, R + R_NEXC, st));
        view = t3d_make_view(surf, Zl, H, W, pad, 1, weights3_host);
    }

    r_smooth.end();
    marks.mark("smooth", st);
    // ---- extract_manifold_surface: two-pass marching cubes, vertices
    NvtxRange r_mc("t3d:extract_manifold_surface");
    RUN(t3d_mc_flags(ws + L.sign, Zp, Hp, Wp, g.z_begin, g.z_end, ws + L.ballots, st));
    marks.mark("flags", st);
    RUN(t3d_exclusive_scan_u32_dev(ws + L.ballots, ws + L.chunkbase, n_chunks, n_chunks, 1, 0, 1, nullptr, R + R_NACTIVE,
                                   ws + L.scan1, st));
    RUN(t3d_mc_words_view_dev(view, x_off, ws + L.sign, Zp, Hp, Wp, g.z_begin, g.z_end, ws + L.ballots, ws + L.chunkbase, cap_active,
                              R + R_NACTIVE, ws + L.aw_idx, ws + L.aw_cnt, R + R_NAMBIGUOUS, st));
    RUN(t3d_exclusive_scan_u32_dev(ws + L.aw_cnt, ws + L.aw_base, cap_active, cap_active, 4, 0, 0, R + R_NACTIVE, R + R_NX,
                                   ws + L.scan2, st));
    k_finalize_sizes<<<1, 1, 0, st>>>(R, cap_active, cap_verts, cap_faces, bbox_state == 2 ? 1 : 0);
    t3d_count_launches(1);
    marks.mark("scan+words+scan", st);
    // Keys, then the vertices on the main stream.  The faces are emitted on the side stream AFTER the vertex kernel (run side
    // by side the two took longer than one after the other: 1.70 ms against 0.77 + 0.76 at 512 x 4096 x 4096) and
    // concurrently with the ordering of the vertices (layer sort, positions, unique: latency-bound kernels that only need the
    // vertices); the canonicalisation waits for the faces right before its face kernels.  The measures follow the faces on
    // the side stream and are joined at the end.
    RUN(t3d_mc_emit_view_dev(view, x_off, ws + L.sign, Zp, Hp, Wp, g.z_begin, g.z_end, ws + L.ballots, ws + L.chunkbase, ws + L.aw_idx,
                             ws + L.aw_base, cap_active, R + R_NACTIVE, cap_verts, cap_faces, ws + L.vkeys, ws + L.faces_raw, 1, st));
    marks.mark("keys", st);
    RUN(t3d_mc_vertices_view_dev(view, x_off, ws + L.vkeys, R + R_NACTIVE, cap_verts, 1, g.z_offset, cum_f64, adj_f64, n_cum, mm_y, mm_x,
                                 scale_in_f64, 7, ws + L.verts_raw, st));
    r_mc.end();
    marks.mark("vertices", st);
    NvtxRange r_canon("t3d:ensure_manifold_mesh+measures");
    T3D_CUDA(cudaEventRecord(side->e[4], st));
    T3D_CUDA(cudaStreamWaitEvent(side->s, side->e[4], 0));
    RUN(t3d_mc_emit_view_dev(view, x_off, ws + L.sign, Zp, Hp, Wp, g.z_begin, g.z_end, ws + L.ballots, ws + L.chunkbase, ws + L.aw_idx,
                             ws + L.aw_base, cap_active, R + R_NACTIVE, cap_verts, cap_faces, ws + L.vkeys, ws + L.faces_raw, 2, side->s));
    T3D_CUDA(cudaEventRecord(side->e[6], side->s));
    // ---- mesh volume / area on the emitted mesh (side stream), canonical mesh
    RUN(t3d_mesh_measure_dev(ws + L.verts_raw, ws + L.faces_raw, cap_faces, R + R_NT, 0, R + R_VOLUME_F64, ws + L.measure, side->s));
    T3D_CUDA(cudaEventRecord(side->e[5], side->s));
    t3d_canon_faces_ready_event(side->e[6]);            // (also orders the earlier work of that stream: the bbox reduction)
    if (cap_zverts)
        RUN(t3d_mesh_canonicalize_structured_dev(ws + L.verts_raw, ws + L.vkeys, cap_verts, R + R_NACTIVE, R + R_VRAW, Zp, Hp, Wp,
                                                 ws + L.chunkbase, ws + L.aw_base, cap_active, g.z_offset, 1, cum_f64, adj_f64, n_cum,
                                                 zkey_bits, cap_zverts, cap_g0, ws + L.faces_raw, cap_faces, R + R_NT, verts_out_f32,
                                                 faces_out_i64, nullptr, R + R_VCANON, R + R_NG0, ws + L.canon, 3, st));
    else
        RUN(t3d_mesh_canonicalize_fast_dev(ws + L.verts_raw, cap_verts, R + R_VRAW, ws + L.faces_raw, cap_faces, R + R_NT,
                                           verts_out_f32, faces_out_i64, nullptr, R + R_VCANON, ws + L.canon, st));
    if (t3d_canon_faces_ready_pending()) T3D_CUDA(cudaStreamWaitEvent(st, side->e[6], 0));   // (a path without face kernels)
    if (g.want_ghost || g.want_lead)
        k_count_plane_vertices<<<1, 64, 0, st>>>((const float*)verts_out_f32, R + R_VCANON, g.z_ghost, g.z_lead, g.want_ghost,
                                                 g.want_lead, R + R_NGHOST, R + R_NLEAD);
    if (g.want_ghost || g.want_lead) t3d_count_launches(1);
    marks.mark("canonicalize", st);
    T3D_CUDA(cudaStreamWaitEvent(st, side->e[5], 0));
    marks.mark("wait measures", st);
    marks.report(st);
    return 0;
}

extern "C" int t3d_reconstruct(const void* masks_u8, int Z, int H, int W, int threshold, int close_ends, int n_stages,
                               unsigned erode_mask, int add_padding, const double* weights3_host, const void* cum_f64,
                               const void* adj_f64, int n_cum, double mm_per_pixel_y, double mm_per_pixel_x, int scale_in_f64,
                               uint32_t cap_active, uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0,
                               int zkey_bits, void* verts_out_f32, void* faces_out_i64, void* results_u64, void* workspace,
                               void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_reconstruct: empty volume"); return 2; }
    if (cap_active == 0 || cap_verts == 0 || cap_faces == 0) { t3d_set_error("t3d_reconstruct: zero capacity"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int pad = add_padding ? 1 : 0;
    const bool fast = fast_surface(n_stages, erode_mask, pad, Z, H, W);
    const Layout L = make_layout(Z, Z, H, W, pad, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, n_stages, true, fast);
    char* ws = (char*)workspace;
    unsigned long long* R = (unsigned long long*)results_u64;
    const int64_t nw = t3d_words_per_row(W), plane_words = (int64_t)H * nw, plane_bytes = (int64_t)H * W;
    uint32_t* bitsA = (uint32_t*)(ws + L.bitsA);
    uint32_t* bitsB = (uint32_t*)(ws + L.bitsB);
    const uint8_t* m = (const uint8_t*)masks_u8;
    SideStream* side;
    RUN(side_for_current_device(&side));
    PrezeroGuard zg;
    {
        const int Zp = Z + 2 * pad, Hp = H + 2 * pad, Wp = fast ? W + S_XPAD + 1 : W + 2 * pad;
        const int64_t n_chunks = t3d_mc_num_chunks(Zp, Hp, Wp);
        zg.add(R, sizeof(unsigned long long) * (R_COUNTS + 2 * (size_t)Z));
        zg.add(ws + L.ballots, (size_t)al(n_chunks * 4));
        zg.add(ws + L.scan1, (size_t)al(t3d_scan_workspace_bytes(n_chunks, 1)));
        zg.add(ws + L.scan2, (size_t)al(t3d_scan_workspace_bytes(cap_active, 4)));
        if (cap_zverts) {
            int64_t off = 0, size = 0;
            t3d_canonicalize_structured_zero_range(cap_verts, cap_faces, cap_zverts, cap_g0, Zp, &off, &size);
            zg.add(ws + L.canon + off, (size_t)size);
        }
        RUN(zg.launch(st));
    }

    // ---- create_voxel_data: pack, fill the holes of the end slices (side stream), z gap fill + per-slice counts
    int bbox_state = 0;
    NvtxRange r_create("t3d:create_voxel_data");
    if (close_ends && t3d_pack_gap_supported(m, Z, H, W, threshold)) {
        // one pass over the masks: pack + gap fill + counts + extrema; the two end planes are packed apart, hole-filled on
        // the side stream meanwhile, and planes 0, 1, Z-2, Z-1 are then rewritten from them
        uint32_t* f0 = bitsA;
        uint32_t* fT = bitsA + plane_words;
        RUN(t3d_pack_masks(m, 1, H, W, threshold, f0, st));
        RUN(t3d_pack_masks(m + (int64_t)(Z - 1) * plane_bytes, 1, H, W, threshold, fT, st));
        T3D_CUDA(cudaEventRecord(side->e[0], st));
        T3D_CUDA(cudaStreamWaitEvent(side->s, side->e[0], 0));
        RUN(t3d_fill_holes_2d(f0, 2, plane_words, H, W, ws + L.fill, side->s));
        T3D_CUDA(cudaEventRecord(side->e[1], side->s));
        RUN(t3d_pack_gap_launch(m, Z, H, W, threshold, bitsB, R + R_COUNTS, (unsigned int*)(R + R_BBOX_I32X6), 1, st));
        T3D_CUDA(cudaStreamWaitEvent(st, side->e[1], 0));
        RUN(t3d_close_ends_fixup_launch(m, Z, H, W, threshold, f0, fT, bitsB, R + R_COUNTS, st));
        bbox_state = 2;
    } else if (close_ends && Z >= 3) {
        RUN(t3d_pack_masks(m, 1, H, W, threshold, bitsA, st));
        RUN(t3d_pack_masks(m + (int64_t)(Z - 1) * plane_bytes, 1, H, W, threshold, bitsA + (int64_t)(Z - 1) * plane_words, st));
        T3D_CUDA(cudaEventRecord(side->e[0], st));
        T3D_CUDA(cudaStreamWaitEvent(side->s, side->e[0], 0));
        RUN(t3d_fill_holes_2d(bitsA, 2, (int64_t)(Z - 1) * plane_words, H, W, ws + L.fill, side->s));
        T3D_CUDA(cudaEventRecord(side->e[1], side->s));
        RUN(t3d_pack_masks(m + plane_bytes, Z - 2, H, W, threshold, bitsA + plane_words, st));
        T3D_CUDA(cudaStreamWaitEvent(st, side->e[1], 0));
        RUN(t3d_gap_fill(bitsA, bitsB, nullptr, nullptr, Z, H, W, R + R_COUNTS, st));
    } else if (close_ends) {
        RUN(t3d_pack_masks(m, Z, H, W, threshold, bitsA, st));
        RUN(t3d_fill_holes_2d(bitsA, 1, 0, H, W, ws + L.fill, st));
        if (Z > 1) RUN(t3d_fill_holes_2d(bitsA + (int64_t)(Z - 1) * plane_words, 1, 0, H, W, ws + L.fill, st));
        RUN(t3d_gap_fill(bitsA, bitsB, nullptr, nullptr, Z, H, W, R + R_COUNTS, st));
    } else {
        RUN(t3d_pack_masks(m, Z, H, W, threshold, bitsB, st));
        RUN(t3d_volume_stats(bitsB, Z, H, W, R + R_COUNTS, nullptr, st));
    }
    r_create.end();
    SlabGeom g = {0, Z, 0, 0, -1, 0, 0, 0, 0.f, 0.f};
    RUN(reconstruct_core(bitsB, g, H, W, n_stages, erode_mask, pad, weights3_host, cum_f64, adj_f64, n_cum, mm_per_pixel_y,
                         mm_per_pixel_x, scale_in_f64, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, zkey_bits, verts_out_f32,
                         faces_out_i64, R, ws, L, fast, bbox_state, side, st));
    T3D_CHECK_LAUNCH("t3d_reconstruct");
    t3d_count_launches(1);
    return 0;
}

// t3d_normals.cu: normals kernel on a strided view (same x_off convention as t3d_mc_vertices_view_dev)
int t3d_mc_normals_view_dev(const OccView& view, int x_off, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts, int unpad_shift,
                            int z_offset, const void* adj_f64, int n_cum, double mm_per_pixel_y, double mm_per_pixel_x,
                            const void* newid_u32, const void* perm_u32, const void* dup_u64, void* winner_u32, void* normals_f32,
                            void* stream);

// Post-step of t3d_reconstruct: field-gradient normals of the step's canonical mesh, enqueued after it on the same stream with
// the same geometry, capacities and workspace.  Everything it reads is still intact when the step ends: the vertex keys, the
// sizes in the result block, the raw -> canonical map of the canonicalisation and the field the vertex kernel evaluated (the
// smoothed occupancy: the padded sign volume on the fast path, bitsC otherwise; neither is written after the vertex kernel).
// The face flags of the canonicalisation's workspace serve as the tie pass's scratch.  normals_out_f32: (cap_verts, 3), rows
// [0, V') valid (V' = results[R_VCANON]); nothing runs when the step overflowed.
extern "C" int t3d_reconstruct_normals(int Z, int H, int W, int n_stages, unsigned erode_mask, int add_padding, const double* weights3_host,
                                       const void* adj_f64, int n_cum, double mm_per_pixel_y, double mm_per_pixel_x, uint32_t cap_active,
                                       uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0, const void* results_u64,
                                       void* workspace, void* normals_out_f32, void* stream)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("t3d_reconstruct_normals: empty volume"); return 2; }
    if (cap_active == 0 || cap_verts == 0 || cap_faces == 0) { t3d_set_error("t3d_reconstruct_normals: zero capacity"); return 2; }
    const int pad = add_padding ? 1 : 0;
    const bool fast = fast_surface(n_stages, erode_mask, pad, Z, H, W);
    const Layout L = make_layout(Z, Z, H, W, pad, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, n_stages, true, fast);
    char* ws = (char*)workspace;
    const unsigned long long* R = (const unsigned long long*)results_u64;
    const int Zp = Z + 2 * pad, Hp = H + 2 * pad, Wp = fast ? W + S_XPAD + 1 : W + 2 * pad;
    OccView view;
    int x_off = 0;
    if (fast) {
        const int nws = (int)t3d_words_per_row(Wp);
        const long long s_ps = (long long)Hp * nws;
        const uint32_t* S_origin = (const uint32_t*)(ws + L.sign) + s_ps + nws + S_XPAD / 32;
        view = t3d_make_view_strided(S_origin, Z, H, W, nws, s_ps, 1, 1, weights3_host);
        x_off = S_XPAD - 1;
    } else {
        const void* smoothed = n_stages > 0 ? ws + L.bitsC : ws + L.bitsB;
        view = t3d_make_view(smoothed, Z, H, W, pad, 1, weights3_host);
    }
    int64_t off[4];
    RUN(t3d_canonical_map_offsets(cap_zverts ? 2 : 1, cap_verts, cap_faces, cap_zverts, cap_g0, Zp, off));
    char* canon = ws + L.canon;
    (void)Hp;
    return t3d_mc_normals_view_dev(view, x_off, ws + L.vkeys, R + R_NACTIVE, cap_verts, 1, 0, adj_f64, n_cum, mm_per_pixel_y,
                                   mm_per_pixel_x, canon + off[0], canon + off[1], canon + off[3], canon + off[2], normals_out_f32,
                                   stream);
}

// ---- z-slab packing: own slices -> planes [halo_lo, halo_lo + n_own) of ext_bits.  The global end slices (fill_first /
// fill_last) are packed first and hole-filled on the side stream while the other slices are packed; t3d_reconstruct_slab
// joins the side stream (join_fill), so the halo exchange in between does not wait for the fill.  (The filled slice is
// part of a halo only if the slab is thinner than the halo; then the fill is joined here.)
// counts of the interior planes [za, zb) and the transformed extrema of the pack kernel -> the result block (zeroed before)
__global__ void k_merge_pre_stats(unsigned long long* __restrict__ r, const unsigned long long* __restrict__ pre, int Zx, int za, int zb)
{
    const int z = blockIdx.x * blockDim.x + threadIdx.x;
    if (z >= za && z < zb) r[R_COUNTS + z] = pre[z];
    if (z < 6) atomicMax((unsigned int*)(r + R_BBOX_I32X6) + z, ((const unsigned int*)(pre + Zx))[z]);
}

// Pre-filled mode (pre_grid_bits / pre_stats_u64 given; t3d_slab_pack_gap_ok says when it applies): the interior of the slab
// -- own planes [SLAB_EDGE, n_own - SLAB_EDGE) -- does not depend on any neighbour's data, so it goes through the one-pass
// kernel of the single-device path (k_pack_gap: threshold + stack + z gap fill + slice counts + extrema, masks read once)
// straight into pre_grid_bits, a (halo_lo + n_own + halo_hi)-plane buffer, with its counts / extrema in pre_stats_u64
// (Zx + 3 uint64).  Only the SLAB_RAW own planes at either end are packed raw into ext_bits: those are what the halo exchange
// sends and what t3d_reconstruct_slab gap-fills together with the received halo planes.
#define SLAB_EDGE 4     // own planes at either end of a slab whose gap fill is left to t3d_reconstruct_slab
#define SLAB_RAW 8      // own planes at either end packed raw into the exchange buffer (>= the halo depth and > SLAB_EDGE)

extern "C" int t3d_slab_pack_gap_ok(const void* masks_u8, int n_own, int H, int W, int threshold)
{
    if (n_own < 2 * SLAB_RAW || H <= 0 || W <= 0) return 0;
    const uint8_t* sub = (const uint8_t*)masks_u8 + (int64_t)(SLAB_EDGE - 2) * H * W;
    return t3d_pack_gap_supported(sub, n_own - 2 * SLAB_EDGE + 4, H, W, threshold) ? 1 : 0;
}

extern "C" int t3d_slab_pack(const void* masks_u8, int n_own, int H, int W, int threshold, int halo_lo, int halo_hi, int fill_first,
                             int fill_last, void* ext_bits, void* fill_scratch, void* pre_grid_bits, void* pre_stats_u64, void* stream)
{
    if (n_own <= 0 || H <= 0 || W <= 0 || halo_lo < 0) { t3d_set_error("t3d_slab_pack: bad slab"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nw = t3d_words_per_row(W), plane_words = (int64_t)H * nw, plane_bytes = (int64_t)H * W;
    const uint8_t* m = (const uint8_t*)masks_u8;
    uint32_t* own = (uint32_t*)ext_bits + (int64_t)halo_lo * plane_words;
    const bool pre = pre_grid_bits != nullptr;
    if (pre) {
        if (!pre_stats_u64 || !t3d_slab_pack_gap_ok(masks_u8, n_own, H, W, threshold)) {
            t3d_set_error("t3d_slab_pack: pre-filled mode needs pre_stats_u64 and a slab t3d_slab_pack_gap_ok accepts");
            return 2;
        }
        const int Zx = halo_lo + n_own + halo_hi, a0 = SLAB_EDGE - 2, zsub = n_own - 2 * SLAB_EDGE + 4;
        unsigned long long* ps = (unsigned long long*)pre_stats_u64;
        T3D_CUDA(cudaMemsetAsync(ps, 0, sizeof(unsigned long long) * ((size_t)Zx + 3), st));
        RUN(t3d_pack_gap_launch(m + (int64_t)a0 * plane_bytes, zsub, H, W, threshold,
                                (uint32_t*)pre_grid_bits + (int64_t)(halo_lo + a0) * plane_words, ps + halo_lo + a0,
                                (unsigned int*)(ps + Zx), 1, st, a0));
    }
    if (fill_last && n_own == 1 && fill_first) fill_last = 0;   // one slice: filled once
    if (!fill_first && !fill_last) {
        if (!pre) return t3d_pack_masks(m, n_own, H, W, threshold, own, st);
        RUN(t3d_pack_masks(m, SLAB_RAW, H, W, threshold, own, st));
        return t3d_pack_masks(m + (int64_t)(n_own - SLAB_RAW) * plane_bytes, SLAB_RAW, H, W, threshold, own + (int64_t)(n_own - SLAB_RAW) * plane_words, st);
    }
    SideStream* side;
    RUN(side_for_current_device(&side));
    const int lo = fill_first ? 1 : 0, hi = fill_last ? n_own - 1 : n_own;   // [lo, hi) = slices that are not filled
    if (fill_first) RUN(t3d_pack_masks(m, 1, H, W, threshold, own, st));
    if (fill_last) RUN(t3d_pack_masks(m + (int64_t)(n_own - 1) * plane_bytes, 1, H, W, threshold, own + (int64_t)(n_own - 1) * plane_words, st));
    T3D_CUDA(cudaEventRecord(side->e[0], st));
    T3D_CUDA(cudaStreamWaitEvent(side->s, side->e[0], 0));
    char* scratch = (char*)fill_scratch;
    if (fill_first && fill_last) {
        RUN(t3d_fill_holes_2d(own, 2, (int64_t)(n_own - 1) * plane_words, H, W, scratch, side->s));
    } else {
        RUN(t3d_fill_holes_2d(fill_first ? own : own + (int64_t)(n_own - 1) * plane_words, 1, 0, H, W, scratch, side->s));
    }
    T3D_CUDA(cudaEventRecord(side->e[1], side->s));
    if (pre) {      // only the raw end ranges [lo, SLAB_RAW) and [n_own - SLAB_RAW, hi)
        RUN(t3d_pack_masks(m + (int64_t)lo * plane_bytes, SLAB_RAW - lo, H, W, threshold, own + (int64_t)lo * plane_words, st));
        const int b0 = n_own - SLAB_RAW;
        RUN(t3d_pack_masks(m + (int64_t)b0 * plane_bytes, hi - b0, H, W, threshold, own + (int64_t)b0 * plane_words, st));
    } else if (hi > lo) RUN(t3d_pack_masks(m + (int64_t)lo * plane_bytes, hi - lo, H, W, threshold, own + (int64_t)lo * plane_words, st));
    const int halo = halo_lo > halo_hi ? halo_lo : halo_hi;
    if (n_own <= halo) T3D_CUDA(cudaStreamWaitEvent(st, side->e[1], 0));
    return 0;
}

// ---- z-slab variant (sharded.py): the caller has packed its own slices into planes [halo_lo, halo_lo + n_own) of
// `ext_bits`, filled the holes of the global end slices and received the halo planes from its z-neighbours.
extern "C" int t3d_reconstruct_slab(const void* ext_bits, int halo_lo, int n_own, int halo_hi, int H, int W, int n_stages,
                                    unsigned erode_mask, int add_padding, int z_begin, int z_end, int z_offset, int want_ghost,
                                    float z_ghost, int want_lead, float z_lead, int join_fill, const double* weights3_host, const void* cum_f64,
                                    const void* adj_f64, int n_cum, double mm_per_pixel_y, double mm_per_pixel_x, int scale_in_f64,
                                    uint32_t cap_active, uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0,
                                    int zkey_bits, void* verts_out_f32, void* faces_out_i64, void* results_u64, void* workspace,
                                    void* pre_grid_bits, const void* pre_stats_u64, void* stream)
{
    if (n_own <= 0 || H <= 0 || W <= 0 || halo_lo < 0 || halo_hi < 0) { t3d_set_error("t3d_reconstruct_slab: bad slab"); return 2; }
    if (pre_grid_bits && (!pre_stats_u64 || n_own < 2 * SLAB_RAW)) { t3d_set_error("t3d_reconstruct_slab: bad pre-filled slab"); return 2; }
    if (cap_active == 0 || cap_verts == 0 || cap_faces == 0) { t3d_set_error("t3d_reconstruct_slab: zero capacity"); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    const int pad = add_padding ? 1 : 0, Zx = halo_lo + n_own + halo_hi;
    const int Zl = imin(SURF_HALO, halo_lo) + n_own + imin(SURF_HALO, halo_hi);
    const bool fast = fast_surface(n_stages, erode_mask, pad, Zx, H, W);
    const Layout L = make_layout(Zx, Zl, H, W, pad, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, n_stages, false, fast);
    char* ws = (char*)workspace;
    unsigned long long* R = (unsigned long long*)results_u64;
    SideStream* side;
    RUN(side_for_current_device(&side));
    PrezeroGuard zg;
    {
        const int Zp = Zl + 2 * pad, Hp = H + 2 * pad, Wp = fast ? W + S_XPAD + 1 : W + 2 * pad;
        const int64_t n_chunks = t3d_mc_num_chunks(Zp, Hp, Wp);
        zg.add(R, sizeof(unsigned long long) * (R_COUNTS + 2 * (size_t)Zx));
        zg.add(ws + L.ballots, (size_t)al(n_chunks * 4));
        zg.add(ws + L.scan1, (size_t)al(t3d_scan_workspace_bytes(n_chunks, 1)));
        zg.add(ws + L.scan2, (size_t)al(t3d_scan_workspace_bytes(cap_active, 4)));
        if (cap_zverts) {
            int64_t off = 0, size = 0;
            t3d_canonicalize_structured_zero_range(cap_verts, cap_faces, cap_zverts, cap_g0, Zp, &off, &size);
            zg.add(ws + L.canon + off, (size_t)size);
        }
        RUN(zg.launch(st));
    }
    if (join_fill) T3D_CUDA(cudaStreamWaitEvent(st, side->e[1], 0));   // hole filling started by t3d_slab_pack
    SlabGeom g = {halo_lo, n_own, halo_hi, z_begin, z_end, z_offset, want_ghost, want_lead, z_ghost, z_lead};
    const uint32_t* grid = (const uint32_t*)(ws + L.bitsB);
    int bbox_state = 0;
    if (pre_grid_bits) {
        // the interior own planes are final in pre_grid_bits (t3d_slab_pack): gap-fill the two ends -- halo planes + SLAB_EDGE own
        // planes each, with the raw plane beyond as the outer neighbour -- and merge the pack kernel's counts / extrema
        const int64_t pw = (int64_t)H * t3d_words_per_row(W);
        const uint32_t* ext = (const uint32_t*)ext_bits;
        uint32_t* pg = (uint32_t*)pre_grid_bits;
        const int zl = halo_lo + SLAB_EDGE, p0 = halo_lo + n_own - SLAB_EDGE;
        RUN(t3d_gap_fill(ext, pg, nullptr, ext + (int64_t)zl * pw, zl, H, W, R + R_COUNTS, st));
        RUN(t3d_gap_fill(ext + (int64_t)p0 * pw, pg + (int64_t)p0 * pw, ext + (int64_t)(p0 - 1) * pw, nullptr, Zx - p0, H, W, R + R_COUNTS + p0, st));
        k_merge_pre_stats<<<(Zx + 255) / 256, 256, 0, st>>>(R, (const unsigned long long*)pre_stats_u64, Zx, zl, p0);
        t3d_count_launches(1);
        unsigned int* bb = (unsigned int*)(R + R_BBOX_I32X6);
        RUN(t3d_bbox_t_planes_launch(pg + (int64_t)halo_lo * pw, SLAB_EDGE, H, W, 0, bb, st));
        RUN(t3d_bbox_t_planes_launch(pg + (int64_t)p0 * pw, SLAB_EDGE, H, W, n_own - SLAB_EDGE, bb, st));
        grid = pg;
        bbox_state = 2;
    } else {
        RUN(t3d_gap_fill(ext_bits, ws + L.bitsB, nullptr, nullptr, Zx, H, W, R + R_COUNTS, st));
    }
    RUN(reconstruct_core(grid, g, H, W, n_stages, erode_mask, pad, weights3_host, cum_f64, adj_f64, n_cum,
                         mm_per_pixel_y, mm_per_pixel_x, scale_in_f64, cap_active, cap_verts, cap_faces, cap_zverts, cap_g0, zkey_bits,
                         verts_out_f32, faces_out_i64, R, ws, L, fast, bbox_state, side, st));
    T3D_CHECK_LAUNCH("t3d_reconstruct_slab");
    t3d_count_launches(1);
    return 0;
}

// Stitching: global face ids = local ids + the number of owned unique vertices of the lower ranks.  `gathered` = the
// all-gathered result blocks (world x stride uint64); only slots R_VCANON / R_NGHOST / R_FCANON are read.
__global__ void k_add_vertex_base(long long* __restrict__ faces, const unsigned long long* __restrict__ gathered, int64_t stride, int rank,
                                  int64_t cap3)
{
    long long base = 0;
    for (int r = 0; r < rank; ++r) base += (long long)(gathered[r * stride + R_VCANON] - gathered[r * stride + R_NGHOST]);
    const int64_t n3 = 3 * (int64_t)gathered[rank * stride + R_FCANON];
    const int64_t n = n3 < cap3 ? n3 : cap3;
    if (base == 0) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) faces[i] += base;
}

extern "C" int t3d_slab_stitch_faces(void* faces_i64, int64_t cap_faces, const void* gathered_results_u64, int64_t stride_u64,
                                     int rank, void* stream)
{
    if (rank < 0 || cap_faces < 0) { t3d_set_error("t3d_slab_stitch_faces: bad arguments"); return 2; }
    if (rank == 0 || cap_faces == 0) return 0;
    k_add_vertex_base<<<T3D_NUM_SMS * 8, 256, 0, (cudaStream_t)stream>>>((long long*)faces_i64, (const unsigned long long*)gathered_results_u64,
                                                               stride_u64, rank, 3 * cap_faces);
    T3D_CHECK_LAUNCH("t3d_slab_stitch_faces");
    t3d_count_launches(1);
    return 0;
}
