// t3d_edt.cu -- exact Euclidean distance transform / signed distance of the packed occupancy (sm_100a).
//
// Additive stage (SURVEY.md 8a-16): the reference has no distance transform; the oracle is
// scipy.ndimage.distance_transform_edt(occ, sampling), i.e. for every set voxel the distance between voxel centres
// to the nearest unset voxel, and sdf = edt(occ) - edt(~occ) (positive inside).
//
// Like scipy the transform propagates the OFFSET to the nearest site (a feature transform) through three separable
// passes, and evaluates sqrt(sum((offset*sampling)^2)) in float64 at the end, so with equal nearest sites the result
// is bit-identical to scipy's:
//   x pass : per row, nearest unset voxel along x straight from the bit words (warp per row, coalesced int16 output)
//   y pass : per (z,x) column, Felzenszwalb/Huttenlocher lower envelope of the parabolas f(j) + ((y-j)*sy)^2
//   z pass : the same along z, then the final distance
// The envelope stacks (site index, left boundary) live in global scratch laid out [stack slot][line] so that the
// threads of a warp (adjacent lines) touch adjacent addresses.
#include <math.h>
#include <stdlib.h>

#include "t3d_common.cuh"

#define EDT_NONE 0x7fff  // int16 sentinel: no site along this line

// ------------------------------------------------------------------------------------------------
// x pass: dx(z,y,x) = signed offset to the nearest site (a voxel whose bit != fg) in the row, EDT_NONE if the row has none
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_edt_x(const uint32_t* __restrict__ bits, int64_t n_rows, int W, int nw, int invert,
                                               int16_t* __restrict__ dx)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n_rows) return;
    const uint32_t l = lane_id();
    const uint32_t* r = bits + row * nw;
    const int nwv = (W + 31) >> 5;
    int16_t* o = dx + row * (int64_t)W;
    // sites = voxels that are NOT foreground (foreground = bit set, or bit clear when invert)
    int left_carry = -0x40000000;  // position of the last site before the current chunk
    for (int w0 = 0; w0 < nwv; w0 += 32) {
        const int w = w0 + l;
        uint32_t s = 0;
        if (w < nwv) {
            const uint32_t v = r[w], vm = valid_mask(w, W);
            s = (invert ? v : ~v) & vm;
        }
        // per-word last / first site positions, then warp scans: nearest site strictly before / after each word
        const int last = s ? (w << 5) + 31 - __clz(s) : -0x40000000;
        const int first = s ? (w << 5) + __ffs(s) - 1 : 0x40000000;
        int pl = last, pf = first;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, pl, d), b = __shfl_down_sync(0xffffffffu, pf, d);
            if (l >= (uint32_t)d) pl = max(pl, a);
            if (l + d < 32) pf = min(pf, b);
        }
        int before = __shfl_up_sync(0xffffffffu, pl, 1);
        if (l == 0) before = -0x40000000;
        before = max(before, left_carry);
        int after = __shfl_down_sync(0xffffffffu, pf, 1);
        if (l == 31) after = 0x40000000;
        // sites beyond this 32-word chunk on the right: scan the remaining words (rows wider than 1024 voxels)
        if (w0 + 32 < nwv) {
            int far = 0x40000000;
            for (int ww = w0 + 32 + l; ww < nwv; ww += 32) {
                const uint32_t v = r[ww], vm = valid_mask(ww, W);
                const uint32_t ss = (invert ? v : ~v) & vm;
                if (ss) far = min(far, (ww << 5) + __ffs(ss) - 1);
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) far = min(far, __shfl_xor_sync(0xffffffffu, far, d));
            after = min(after, far);
        }
        // every lane now emits the 32 voxels of each word of the chunk in turn (coalesced stores)
        for (int k = 0; k < 32 && w0 + k < nwv; ++k) {
            const uint32_t sw = __shfl_sync(0xffffffffu, s, k);
            const int bw = __shfl_sync(0xffffffffu, before, k), aw = __shfl_sync(0xffffffffu, after, k);
            const int x = ((w0 + k) << 5) + l;
            if (x < W) {
                const uint32_t lo = sw & (l == 31 ? 0xffffffffu : ((2u << l) - 1u));   // sites at or before x
                const uint32_t hi = sw & ~((1u << l) - 1u);                             // sites at or after x
                const int pl2 = lo ? ((w0 + k) << 5) + 31 - __clz(lo) : bw;
                const int pr2 = hi ? ((w0 + k) << 5) + __ffs(hi) - 1 : aw;
                const int dl = x - pl2, dr = pr2 - x;
                int best;
                if (pl2 < -0x3fffffff && pr2 > 0x3fffffff) best = EDT_NONE;
                else best = (dl <= dr) ? -dl : dr;
                o[x] = (int16_t)best;
            }
        }
        left_carry = max(left_carry, __shfl_sync(0xffffffffu, pl, 31));
    }
}

// ------------------------------------------------------------------------------------------------
// envelope pass along an axis with `n` samples and element stride `stride_line` between consecutive samples;
// line id -> base offset = (line / inner) * outer_stride + (line % inner)
// in : offsets so far (int16 per component, `ncomp_in` components, component arrays `vol` elements apart)
// out: ncomp_in + 1 components (new component first), or the final float distance
// ------------------------------------------------------------------------------------------------
struct EdtPass {
    const int16_t* in;  // first existing component
    const int16_t* in1; // second existing component (ncomp_in > 1)
    int16_t* out;      // (ncomp_in + 1) component arrays, may be null when dist_out is set
    float* dist_out;   // final float32 distance (z pass)
    int64_t vol;       // elements per component array
    int64_t n_lines, inner, outer_stride, stride;
    int n, ncomp_in;
    double w_new, w0, w1;  // squared sampling of the new axis and of the existing components
    double s_new, s0, s1;  // the samplings themselves (final distance, scipy's arithmetic)
    uint32_t* stack;   // [n][n_lines] entries (site | first sample it serves << 16)
    float sign;        // +1 / -1 applied to dist_out
    int accumulate;    // dist_out += instead of =
};

// Lower envelope of the parabolas f(j) + ((q-j)*s)^2 along one line per thread (Felzenszwalb & Huttenlocher).  Only
// integer positions are ever queried, so a stack entry keeps the FIRST SAMPLE its site serves instead of the real
// intersection abscissa: entry = site | start << 16 (4 bytes instead of 12), the top of the stack lives in registers,
// and "pop while the new site takes over at or before the top's start" is equivalent to the real-valued test for every
// integer query (a site whose interval contains no integer can be dropped).  A tie at an integer position stays with the
// earlier site, as in the real-valued sweep (`boundary < q` to advance).
// The kernel is issue-bound (ncu: ~60 % SM throughput, DRAM at 1.3 TB/s), so the loop bodies are kept lean: pass
// parameters in registers, pointers advanced instead of re-derived, the parabola terms carried incrementally, the pass
// kind (one or two existing components, offsets or final distance) fixed at compile time.
#define EDT_THREADS 128

template <int NCOMP>
__device__ __forceinline__ bool site_cost(const int16_t* __restrict__ in0, const int16_t* __restrict__ in1, int64_t off, double w0,
                                          double w1, double& f)
{
    const int a = in0[off];
    if (a == EDT_NONE) return false;
    f = (double)(a * a) * w0;
    if (NCOMP > 1) {
        const int b = in1[off];
        f += (double)(b * b) * w1;
    }
    return true;
}

template <int NCOMP, bool FINAL>
__global__ void __launch_bounds__(EDT_THREADS) k_edt_envelope(EdtPass p)
{
    const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= p.n_lines) return;
    const int64_t L = p.n_lines, stride = p.stride;
    const int64_t base = (line / p.inner) * p.outer_stride + (line % p.inner);
    const int n = p.n;
    const double w_new = p.w_new, w0 = p.w0, w1 = p.w1, two_w = 2.0 * p.w_new, nd = (double)p.n;
    const int16_t* __restrict__ in0 = p.in + base;
    const int16_t* __restrict__ in1 = NCOMP > 1 ? p.in1 + base : nullptr;
    uint32_t* __restrict__ st = p.stack + line;     // entry k of this line at st[k * L]
    int k = -1;            // index of the top entry; entries below the top are in st[], the top is in registers:
    int vk = 0, bk = 0;    //   site, first sample it serves,
    double gk = 0.0, vkd = 0.0;   // f(vk) + vk^2 w, vk as double
    uint32_t* top = st;    // where the top entry will be spilled (st + k * L)
    double qd = 0.0;
    int64_t off = 0;
    for (int q = 0; q < n; ++q, qd += 1.0, off += stride) {
        double fq;
        if (!site_cost<NCOMP>(in0, in1, off, w0, w1, fq)) continue;
        const double gq = fq + qd * qd * w_new;
        int b = 0;
        while (k >= 0) {
            // abscissa where parabola q overtakes parabola vk: q serves the samples > s
            const double s = (gq - gk) / (two_w * (qd - vkd));
            b = (int)fmin(fmax(floor(s) + 1.0, 0.0), nd);
            if (b > bk) break;
            --k;             // the top serves no sample any more
            top -= L;
            if (k >= 0) {
                const uint32_t e = *top;
                vk = (int)(e & 0xffffu); bk = (int)(e >> 16);
                double fk;
                site_cost<NCOMP>(in0, in1, (int64_t)vk * stride, w0, w1, fk);
                vkd = (double)vk;
                gk = fk + vkd * vkd * w_new;
            }
        }
        if (k >= 0) { *top = (uint32_t)vk | ((uint32_t)bk << 16); top += L; }   // the old top goes to the stack
        else { b = 0; top = st; }
        ++k;
        vk = q; bk = b; gk = gq; vkd = qd;
    }
    if (k >= 0) *top = (uint32_t)vk | ((uint32_t)bk << 16);
    // evaluation sweep: entries in ascending order
    int16_t* __restrict__ out0 = FINAL ? nullptr : p.out + base;
    float* __restrict__ dout = FINAL ? p.dist_out + base : nullptr;
    const int64_t vol = p.vol;
    if (k < 0) {   // no site anywhere on this line
        off = 0;
        for (int q = 0; q < n; ++q, off += stride) {
            if (FINAL) { const float d = p.sign * INFINITY; dout[off] = p.accumulate ? dout[off] + d : d; }
            else out0[off] = EDT_NONE;
        }
        return;
    }
    const double s_new = p.s_new, s0 = p.s0, s1 = p.s1;
    const float sign = p.sign;
    const bool acc = p.accumulate != 0;
    int j = 0, v = (int)(st[0] & 0xffffu), next_start = n;
    uint32_t e_next = 0;
    const uint32_t* nxt = st + L;
    if (k >= 1) { e_next = *nxt; next_start = (int)(e_next >> 16); }
    int a = 0, bcomp = 0;
    double a2 = 0.0, b2 = 0.0;   // (a*s0)^2 and (b*s1)^2 of the current site (added in scipy's order below)
    bool have = false;
    off = 0;
    for (int q = 0; q < n; ++q, off += stride) {
        while (q >= next_start) {
            ++j;
            v = (int)(e_next & 0xffffu);
            nxt += L;
            if (j < k) { e_next = *nxt; next_start = (int)(e_next >> 16); }
            else next_start = n;
            have = false;
        }
        if (!have) {
            const int64_t soff = (int64_t)v * stride;
            a = in0[soff];
            bcomp = NCOMP > 1 ? in1[soff] : 0;
            if (FINAL) {
                // kept as two products: the sum order below must stay ((t0^2 + t1^2) + t2^2)
                const double t1 = __dmul_rn((double)a, s0), t2 = __dmul_rn((double)bcomp, s1);
                a2 = __dmul_rn(t1, t1); b2 = __dmul_rn(t2, t2);
            }
            have = true;
        }
        const int dnew = v - q;
        if (FINAL) {
            // scipy: dt = (ft - indices) * sampling; sqrt(add.reduce(dt*dt, axis=0)) -- axis order z, y, x
            const double t0 = __dmul_rn((double)dnew, s_new);
            const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(t0, t0), a2), b2);
            const float d = sign * (float)sqrt(d2);
            dout[off] = acc ? dout[off] + d : d;
        } else {
            out0[off] = (int16_t)dnew;
            out0[vol + off] = (int16_t)a;
            if (NCOMP > 1) out0[2 * vol + off] = (int16_t)bcomp;
        }
    }
}

static inline int64_t a256(int64_t x) { return (x + 255) & ~(int64_t)255; }

static int edt_check(int Z, int H, int W, const char* who)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("%s: empty volume", who); return 2; }
    if (Z > 32766 || H > 32766 || W > 32766) { t3d_set_error("%s: extent above 32766", who); return 2; }
    return 0;
}

// x and y passes: dyx_i16 = two (Z,H,W) int16 arrays back to back, [0] = y offset, [1] = x offset of the nearest site
// within the voxel's own z plane (EDT_NONE in [0] if the plane has no site).  These passes never look across planes, so
// a z-slab can run them on its own slices.  workspace: t3d_edt_xy_workspace_bytes.
extern "C" int64_t t3d_edt_xy_workspace_bytes(int Z, int H, int W)
{
    const int64_t vol = (int64_t)Z * H * W;
    return a256(vol * 2) + a256(vol * 4) + 1024;   // x offsets, envelope stacks
}

extern "C" int t3d_edt_xy(const void* occ_bits, int Z, int H, int W, int invert, const double* sampling_host, void* dyx_i16,
                          void* workspace, void* stream)
{
    if (int rc = edt_check(Z, H, W, "t3d_edt_xy")) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t vol = (int64_t)Z * H * W;
    const double sy = sampling_host ? sampling_host[1] : 1.0, sx = sampling_host ? sampling_host[2] : 1.0;
    char* ws = (char*)workspace;
    int16_t* dx = (int16_t*)ws; ws += a256(vol * 2);
    uint32_t* stack = (uint32_t*)ws;
    const int64_t rows = (int64_t)Z * H;
    k_edt_x<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, st>>>((const uint32_t*)occ_bits, rows, W, t3d_wpr(W), invert ? 1 : 0, dx);
    EdtPass p;
    // y pass: lines = (z, x); samples stride W
    p.in = dx; p.in1 = nullptr; p.out = (int16_t*)dyx_i16; p.dist_out = nullptr; p.vol = vol;
    p.n_lines = (int64_t)Z * W; p.inner = W; p.outer_stride = (int64_t)H * W; p.stride = W; p.n = H; p.ncomp_in = 1;
    p.w_new = sy * sy; p.w0 = sx * sx; p.w1 = 0.0; p.s_new = sy; p.s0 = sx; p.s1 = 0.0; p.stack = stack; p.sign = 1.f;
    p.accumulate = 0;
    k_edt_envelope<1, false><<<(unsigned)((p.n_lines + EDT_THREADS - 1) / EDT_THREADS), EDT_THREADS, 0, st>>>(p);
    T3D_CHECK_LAUNCH("t3d_edt_xy");
    t3d_count_launches(2);
    return 0;
}

// z pass + final distance on full z columns: dy_i16 / dx_i16 (Z,H,W) from t3d_edt_xy (for a sharded run: the y-slab this
// rank received in the all-to-all transpose, H = rows of that y-slab).  dist_f32 (Z,H,W) = or += sign * distance.
extern "C" int64_t t3d_edt_z_workspace_bytes(int Z, int H, int W)
{
    const int64_t vol = (int64_t)Z * H * W;
    return a256(vol * 4) + 1024;   // envelope stacks
}

extern "C" int t3d_edt_z(const void* dy_i16, const void* dx_i16, int Z, int H, int W, const double* sampling_host, float sign,
                         int accumulate, void* dist_f32, void* workspace, void* stream)
{
    if (int rc = edt_check(Z, H, W, "t3d_edt_z")) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t vol = (int64_t)Z * H * W;
    const double sz = sampling_host ? sampling_host[0] : 1.0, sy = sampling_host ? sampling_host[1] : 1.0,
                 sx = sampling_host ? sampling_host[2] : 1.0;
    EdtPass p;
    // lines = (y, x); samples stride H*W; input components (dy, dx)
    p.in = (const int16_t*)dy_i16; p.in1 = (const int16_t*)dx_i16; p.out = nullptr; p.dist_out = (float*)dist_f32; p.vol = vol;
    p.n_lines = (int64_t)H * W; p.inner = (int64_t)H * W; p.outer_stride = 0; p.stride = (int64_t)H * W; p.n = Z; p.ncomp_in = 2;
    p.w_new = sz * sz; p.w0 = sy * sy; p.w1 = sx * sx; p.s_new = sz; p.s0 = sy; p.s1 = sx; p.stack = (uint32_t*)workspace; p.sign = sign;
    p.accumulate = accumulate ? 1 : 0;
    k_edt_envelope<2, true><<<(unsigned)((p.n_lines + EDT_THREADS - 1) / EDT_THREADS), EDT_THREADS, 0, st>>>(p);
    T3D_CHECK_LAUNCH("t3d_edt_z");
    t3d_count_launches(1);
    return 0;
}

// dist_f32 (Z,H,W): sign * distance from every foreground voxel (bit set; bit clear if invert) to the nearest voxel of
// the other kind, 0 at the other kind, inf if there is none; accumulate != 0 adds to dist_f32 instead of overwriting.
// sampling_host: {sz, sy, sx}.  Extents up to 32766 per axis.
extern "C" int64_t t3d_edt_workspace_bytes(int Z, int H, int W)
{
    const int64_t vol = (int64_t)Z * H * W;
    const int64_t a = t3d_edt_xy_workspace_bytes(Z, H, W), b = t3d_edt_z_workspace_bytes(Z, H, W);
    return a256(vol * 4) + (a > b ? a : b);     // (dy, dx) + the larger of the two passes' scratch
}

extern "C" int t3d_edt(const void* occ_bits, int Z, int H, int W, int invert, const double* sampling_host, float sign,
                       int accumulate, void* dist_f32, void* workspace, void* stream)
{
    if (int rc = edt_check(Z, H, W, "t3d_edt")) return rc;
    const int64_t vol = (int64_t)Z * H * W;
    int16_t* dyx = (int16_t*)workspace;
    char* scratch = (char*)workspace + a256(vol * 4);
    if (int rc = t3d_edt_xy(occ_bits, Z, H, W, invert, sampling_host, dyx, scratch, stream)) return rc;
    return t3d_edt_z(dyx, dyx + vol, Z, H, W, sampling_host, sign, accumulate, dist_f32, scratch, stream);
}

// ------------------------------------------------------------------------------------------------
// Signed distance in ONE sweep per axis (sdf = edt(occ) - edt(~occ)): every voxel only needs the distance to the nearest
// voxel of the OTHER kind, so each pass stores ONE offset per voxel -- to the nearest opposite-kind voxel found so far --
// with the voxel's own kind in bit 0 of the first component:  enc = (offset << 1) | bit.  A voxel is then
//   * a zero-cost site of the envelope of its own kind (only the two ends of a run of equal voxels can ever serve a
//     voxel of the other kind: interior voxels of a run are skipped), and
//   * a site with cost (stored offsets)^2 of the envelope of the other kind,
// and it is evaluated on exactly one envelope.  Compared with two separate transforms: half the intermediate traffic
// (2 + 4 B/voxel instead of 4 + 8), half the pushes, half the evaluations, one launch per axis, and the final pass writes
// the signed float directly.  Same arithmetic for the result (scipy's sqrt(sum((offset*sampling)^2)), z, y, x order).
//
// Envelope mechanics as above, with three changes that cut the instruction count (the old kernel was issue-bound):
//   * a stack entry (8 bytes) carries the site's offsets, so popping and the evaluation sweep never go back to the input;
//   * the take-over position floor(num/den)+1 comes from a float32 estimate corrected by the exact float64 predicate
//     num < den*p (no float64 division);
//   * persistent threads: a thread walks lines t, t+T, ... and reuses its stack region ([slot][thread] layout), so the
//     stack workspace is bounded by the resident threads, not by the volume.
// Extents up to 16382 per axis (15-bit offsets).
// ------------------------------------------------------------------------------------------------
#define SDF_NONE 0x3fff          // offset sentinel: no opposite-kind voxel along the axes swept so far
#define SDF_THREADS 128

__device__ __forceinline__ int sdf_dec(int enc) { return enc >> 1; }   // arithmetic shift: signed offset

__global__ void __launch_bounds__(256) k_sdf_x(const uint32_t* __restrict__ bits, int64_t n_rows, int W, int nw, int16_t* __restrict__ ex)
{
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n_rows) return;
    const uint32_t l = lane_id();
    const uint32_t* r = bits + row * nw;
    const int nwv = (W + 31) >> 5;
    int16_t* o = ex + row * (int64_t)W;
    const int NEG = -0x40000000, POS = 0x40000000;
    int carry0 = NEG, carry1 = NEG;    // last zero / one before the current chunk
    for (int w0 = 0; w0 < nwv; w0 += 32) {
        const int w = w0 + l;
        uint32_t v = 0, vm = 0;
        if (w < nwv) { v = r[w]; vm = valid_mask(w, W); }
        const uint32_t s1 = v & vm, s0 = ~v & vm;          // ones / zeros of this word
        int pl0 = s0 ? (w << 5) + 31 - __clz(s0) : NEG, pf0 = s0 ? (w << 5) + __ffs(s0) - 1 : POS;
        int pl1 = s1 ? (w << 5) + 31 - __clz(s1) : NEG, pf1 = s1 ? (w << 5) + __ffs(s1) - 1 : POS;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int a0 = __shfl_up_sync(0xffffffffu, pl0, d), b0 = __shfl_down_sync(0xffffffffu, pf0, d);
            const int a1 = __shfl_up_sync(0xffffffffu, pl1, d), b1 = __shfl_down_sync(0xffffffffu, pf1, d);
            if (l >= (uint32_t)d) { pl0 = max(pl0, a0); pl1 = max(pl1, a1); }
            if (l + d < 32) { pf0 = min(pf0, b0); pf1 = min(pf1, b1); }
        }
        int before0 = __shfl_up_sync(0xffffffffu, pl0, 1), before1 = __shfl_up_sync(0xffffffffu, pl1, 1);
        if (l == 0) { before0 = NEG; before1 = NEG; }
        before0 = max(before0, carry0); before1 = max(before1, carry1);
        int after0 = __shfl_down_sync(0xffffffffu, pf0, 1), after1 = __shfl_down_sync(0xffffffffu, pf1, 1);
        if (l == 31) { after0 = POS; after1 = POS; }
        if (w0 + 32 < nwv) {          // rows wider than 1024 voxels: first zero / one beyond this chunk
            int far0 = POS, far1 = POS;
            for (int ww = w0 + 32 + l; ww < nwv; ww += 32) {
                const uint32_t vv = r[ww], vmm = valid_mask(ww, W);
                const uint32_t t1 = vv & vmm, t0 = ~vv & vmm;
                if (t0) far0 = min(far0, (ww << 5) + __ffs(t0) - 1);
                if (t1) far1 = min(far1, (ww << 5) + __ffs(t1) - 1);
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                far0 = min(far0, __shfl_xor_sync(0xffffffffu, far0, d));
                far1 = min(far1, __shfl_xor_sync(0xffffffffu, far1, d));
            }
            after0 = min(after0, far0); after1 = min(after1, far1);
        }
        for (int k = 0; k < 32 && w0 + k < nwv; ++k) {
            const uint32_t vw = __shfl_sync(0xffffffffu, v, k), vmw = __shfl_sync(0xffffffffu, vm, k);
            const int b0 = __shfl_sync(0xffffffffu, before0, k), b1 = __shfl_sync(0xffffffffu, before1, k);
            const int a0 = __shfl_sync(0xffffffffu, after0, k), a1 = __shfl_sync(0xffffffffu, after1, k);
            const int x = ((w0 + k) << 5) + l;
            if (x < W) {
                const uint32_t bit = (vw >> l) & 1u;
                const uint32_t sw = (bit ? ~vw : vw) & vmw;                              // opposite-kind voxels of this word
                const int bw = bit ? b0 : b1, aw = bit ? a0 : a1;
                const uint32_t lo = sw & ((2u << l) - 1u);                               // (2u << 31) wraps to 0: mask = all ones
                const uint32_t hi = sw & ~((1u << l) - 1u);
                const int pl2 = lo ? ((w0 + k) << 5) + 31 - __clz(lo) : bw;
                const int pr2 = hi ? ((w0 + k) << 5) + __ffs(hi) - 1 : aw;
                const int dl = x - pl2, dr = pr2 - x;
                int best;
                if (pl2 < -0x3fffffff && pr2 > 0x3fffffff) best = SDF_NONE;
                else best = (dl <= dr) ? -dl : dr;
                o[x] = (int16_t)((best << 1) | (int)bit);
            }
        }
        carry0 = max(carry0, __shfl_sync(0xffffffffu, pl0, 31));
        carry1 = max(carry1, __shfl_sync(0xffffffffu, pl1, 31));
    }
}

struct SdfPass {
    const int16_t* in0;   // first component, encoded (offset << 1) | kind
    const int16_t* in1;   // second component (plain), NCOMP == 2
    int16_t* out0;        // new component, encoded                       } !FINAL
    int16_t* out1;        // first existing component of the serving site }
    float* sdf;           // FINAL: signed distance
    int64_t n_lines, inner, outer_stride, stride;
    int n;
    int bulk;             // 1: every 128-line tile is one contiguous, 16-byte aligned row segment per sample -> bulk-async tiles
    double w_new, w0, w1, s_new, s0, s1;
    uint2* stack;         // [total threads][n]: a thread's stack is contiguous -- threads are not in lockstep on the slot index, so
                          // thread-major keeps each thread's accesses sequential (4 entries per 32-byte sector)
};

// ---- bulk-async (TMA engine, 1-D form) tile pipeline: raw PTX, sm_90+ ---------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

#define SDF_ROWS 16     // samples per pipeline stage (one bulk copy of 256 bytes per row and component)
#define SDF_STAGES 3    // stages in flight (bulk-async path)

// Per 128-line tile: for K = 0, 1 (the envelope "distance to the nearest K-voxel") a build sweep, then an evaluation sweep
// at the voxels of the other kind -- ONE straight-line code body for both kinds (the kernel is instruction-bound: a version
// that built both envelopes in one sweep paid more in register moves, selects and divergence than it saved in loads; ncu:
// 240-380 instructions per sample, 25 % IMAD moves, 9 % BSSY/BSYNC).  The samples stream through a shared-memory ring of
// [SDF_ROWS][128] int16 tiles: with p.bulk the rows of a tile are contiguous 256-byte segments fetched by cp.async.bulk (one
// lane per row, completion on an mbarrier, SDF_STAGES tiles in flight); else every thread fills its own column with plain
// loads (same layout; a thread only ever reads its own column).
template <int NCOMP, bool FINAL>
__global__ void __launch_bounds__(SDF_THREADS, 8) k_sdf_envelope(SdfPass p)
{
    __shared__ __align__(128) int16_t s_t0[SDF_STAGES][SDF_ROWS][SDF_THREADS];
    __shared__ __align__(128) int16_t s_t1[NCOMP > 1 ? SDF_STAGES : 1][SDF_ROWS][SDF_THREADS];
    __shared__ __align__(8) uint64_t s_full[SDF_STAGES];
    const int tid = threadIdx.x;
    const int64_t t = (int64_t)blockIdx.x * SDF_THREADS + tid;
    const int n = p.n;
    const int64_t stride = p.stride;
    const double w_new = p.w_new, w0 = p.w0, w1 = p.w1, two_w = 2.0 * p.w_new;
    const int n_chunks = (n + SDF_ROWS - 1) / SDF_ROWS;
    const bool bulk = p.bulk != 0;
    if (bulk && tid == 0) {
        for (int s = 0; s < SDF_STAGES; ++s) mbar_init(&s_full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t uses = 0;      // chunks consumed so far by this CTA (stage = uses % STAGES, parity = (uses / STAGES) & 1)
    uint32_t issued = 0;    // chunks issued so far (warp 0)
    uint2* const st = p.stack + t * (int64_t)n;     // this thread's stack: n entries, contiguous (see SdfPass::stack)
    const int64_t n_tiles = (p.n_lines + SDF_THREADS - 1) / SDF_THREADS;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t line0 = tile * SDF_THREADS, line = line0 + tid;
        const bool live = line < p.n_lines;
        const int tile_lines = (int)min((int64_t)SDF_THREADS, p.n_lines - line0);
        const int64_t base0 = (line0 / p.inner) * p.outer_stride + (line0 % p.inner);     // first line of the tile
        const int64_t base = live ? (line / p.inner) * p.outer_stride + (line % p.inner) : 0;
        int k = -1;                                   // index of the top entry of the envelope being built / evaluated
#pragma unroll 1
        for (int pass = 0; pass < 4; ++pass) {
            const int K = pass >> 1;
            const bool build = (pass & 1) == 0;
            const bool need1 = NCOMP > 1 && build;
            // state of a build sweep: the top entry in registers (site, first sample it serves, its offsets, its cost)
            int vk = 0, bk = 0, ak = 0, ck = 0, prev_kind = -1, run_start = 0;
            double gk = 0.0;
            uint2* top = st;
            // state of an evaluation sweep
            int j = 0, v = 0, ea = 0, ec = 0, next_start = n;
            uint2 e_next = make_uint2(0, 0);
            const uint2* nx = st + 1;
            double a2 = 0.0, c2 = 0.0;
            bool fresh = true;
            if (build) k = -1;
            else if (k >= 0) {
                const uint2 e0 = st[0];
                v = (int)(e0.x & 0xffffu); ea = (int)(short)(e0.y & 0xffffu); ec = (int)(short)(e0.y >> 16);
                if (k >= 1) { e_next = *nx; next_start = (int)(e_next.x >> 16); }
            }
            // one site: pop the entries it takes over completely, then push it
            auto push = [&](int q, int a, int c) {
                const double qd = (double)q;
                double gq = (double)(a * a) * w0 + qd * qd * w_new;
                if (NCOMP > 1) gq += (double)(c * c) * w1;
                int b = 0;
                while (k >= 0) {
                    // first sample that site q takes from the top site vk: the smallest integer s with num < den * s
                    const double num = gq - gk, den = two_w * (qd - (double)vk);
                    const float est = fminf(fmaxf(__fdividef((float)num, (float)den), -1.0f), (float)n);   // (also tames +-inf)
                    const float fl = floorf(est);
                    b = max(0, min((int)fl + 1, n));
                    const float fr = est - fl;
                    if (fr < 0.02f || fr > 0.98f) {        // the float32 estimate is too close to an integer to be trusted
                        while (b > 0 && num < den * (double)(b - 1)) --b;
                        while (b < n && !(num < den * (double)b)) ++b;
                    }
                    if (b > bk) break;
                    --k;
                    --top;
                    if (k >= 0) {
                        const uint2 e = *top;
                        vk = (int)(e.x & 0xffffu); bk = (int)(e.x >> 16);
                        ak = (int)(short)(e.y & 0xffffu); ck = (int)(short)(e.y >> 16);
                        const double vd = (double)vk;
                        gk = (double)(ak * ak) * w0 + vd * vd * w_new;
                        if (NCOMP > 1) gk += (double)(ck * ck) * w1;
                    }
                }
                if (k >= 0) { *top = make_uint2((uint32_t)vk | ((uint32_t)bk << 16), ((uint32_t)ak & 0xffffu) | ((uint32_t)ck << 16)); ++top; }
                else { b = 0; top = st; }
                ++k;
                vk = q; bk = b; ak = a; ck = c; gk = gq;
            };
            // chunk loader: rows [c*ROWS, ...) of this tile into stage (issued % STAGES)
            auto issue = [&](int c) {
                const int sg = (int)(issued % SDF_STAGES);
                const int rows = min(SDF_ROWS, n - c * SDF_ROWS);
                if (tid < 32) {
                    const uint32_t row_bytes = (uint32_t)tile_lines * 2u;
                    if (tid == 0) mbar_expect_tx(&s_full[sg], row_bytes * rows * (need1 ? 2u : 1u));
                    __syncwarp();
                    if (tid < rows) {
                        const int64_t off = base0 + (int64_t)(c * SDF_ROWS + tid) * stride;
                        bulk_g2s(&s_t0[sg][tid][0], p.in0 + off, row_bytes, &s_full[sg]);
                        if (need1) bulk_g2s(&s_t1[sg][tid][0], p.in1 + off, row_bytes, &s_full[sg]);
                    }
                }
                ++issued;
            };
            if (bulk) {
                for (int c = 0; c < SDF_STAGES - 1 && c < n_chunks; ++c) issue(c);
            }
            for (int c = 0; c < n_chunks; ++c) {
                const int sg = (int)(uses % SDF_STAGES);
                const int rows = min(SDF_ROWS, n - c * SDF_ROWS);
                if (bulk) {
                    if (c + SDF_STAGES - 1 < n_chunks) issue(c + SDF_STAGES - 1);   // (its stage was released by the barrier below)
                    mbar_wait(&s_full[sg], (uses / SDF_STAGES) & 1u);
                } else if (live) {
                    const int64_t off = base + (int64_t)c * SDF_ROWS * stride;
#pragma unroll 8
                    for (int r = 0; r < rows; ++r) s_t0[sg][r][tid] = p.in0[off + (int64_t)r * stride];
                    if (need1) {
#pragma unroll 8
                        for (int r = 0; r < rows; ++r) s_t1[sg][r][tid] = p.in1[off + (int64_t)r * stride];
                    }
                }
                if (live && build) {
                    // a K-voxel is a zero-cost site, but only the two ends of a run of K-voxels can serve a voxel of the other
                    // kind; a voxel of the other kind is a site with its stored offsets
                    for (int r = 0; r < rows; ++r) {
                        const int q = c * SDF_ROWS + r;
                        const int cur = s_t0[sg][r][tid];
                        const int kind = cur & 1;
                        if (kind == K) {
                            if (prev_kind != K) { push(q, 0, 0); run_start = q; }      // start of a run
                        } else {
                            if (prev_kind == K && q - 1 > run_start) push(q - 1, 0, 0);  // the run that just ended
                            const int a = sdf_dec(cur);
                            if (a != SDF_NONE) push(q, a, NCOMP > 1 ? (int)s_t1[sg][r][tid] : 0);
                        }
                        prev_kind = kind;
                    }
                } else if (live) {
                    int64_t off = base + (int64_t)c * SDF_ROWS * stride;
                    for (int r = 0; r < rows; ++r, off += stride) {
                        const int kind = s_t0[sg][r][tid] & 1;
                        if (kind == K) continue;
                        if (k < 0) {        // no K-voxel reachable from this line
                            if (FINAL) p.sdf[off] = K ? -INFINITY : INFINITY;
                            else { p.out0[off] = (int16_t)((SDF_NONE << 1) | kind); p.out1[off] = 0; }
                            continue;
                        }
                        const int q = c * SDF_ROWS + r;
                        while (q >= next_start) {
                            ++j;
                            v = (int)(e_next.x & 0xffffu); ea = (int)(short)(e_next.y & 0xffffu); ec = (int)(short)(e_next.y >> 16);
                            ++nx;
                            if (j < k) { e_next = *nx; next_start = (int)(e_next.x >> 16); }
                            else next_start = n;
                            fresh = true;
                        }
                        const int dnew = v - q;
                        if (FINAL) {
                            if (fresh) {
                                const double t1 = __dmul_rn((double)ea, p.s0), t2 = __dmul_rn((double)ec, p.s1);
                                a2 = __dmul_rn(t1, t1); c2 = __dmul_rn(t2, t2);
                                fresh = false;
                            }
                            // scipy: dt = (ft - indices) * sampling; sqrt(add.reduce(dt*dt, axis=0)) -- axis order z, y, x
                            const double t0 = __dmul_rn((double)dnew, p.s_new);
                            const float d = (float)sqrt(__dadd_rn(__dadd_rn(__dmul_rn(t0, t0), a2), c2));
                            p.sdf[off] = K ? -d : d;          // distance to the nearest 0 (inside): +, to the nearest 1: -
                        } else {
                            p.out0[off] = (int16_t)((dnew << 1) | kind);
                            p.out1[off] = (int16_t)ea;
                        }
                    }
                }
                ++uses;
                if (bulk) __syncthreads();     // every thread is done with this stage: it may be refilled
            }
            if (live && build) {
                if (prev_kind == K && n - 1 > run_start) push(n - 1, 0, 0);       // end of the last run
                if (k >= 0) *top = make_uint2((uint32_t)vk | ((uint32_t)bk << 16), ((uint32_t)ak & 0xffffu) | ((uint32_t)ck << 16));
            }
        }
    }
}

static int sdf_check(int Z, int H, int W, const char* who)
{
    if (Z <= 0 || H <= 0 || W <= 0) { t3d_set_error("%s: empty volume", who); return 2; }
    if (Z > 16382 || H > 16382 || W > 16382) { t3d_set_error("%s: extent above 16382", who); return 2; }
    return 0;
}

// persistent grid = one resident wave (the stack workspace is sized by it): CTAs per SM from the occupancy calculator,
// queried once per kernel (the smaller of the two instantiations is used for both, so the workspace formula has one input)
static int sdf_ctas_per_sm()
{
    static int v = 0;
    if (!v) {
        int a = 0, b = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, k_sdf_envelope<1, false>, SDF_THREADS, 0);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_sdf_envelope<2, true>, SDF_THREADS, 0);
        v = a < b ? a : b;
        if (v < 1) v = 1;
    }
    return v;
}

static int sdf_grid_blocks(int64_t n_lines)
{
    const int64_t want = (n_lines + SDF_THREADS - 1) / SDF_THREADS, cap = (int64_t)T3D_NUM_SMS * sdf_ctas_per_sm();
    return (int)(want < cap ? want : cap);
}

static int64_t sdf_stack_bytes(int n, int64_t n_lines) { return a256((int64_t)n * sdf_grid_blocks(n_lines) * SDF_THREADS * 8); }

static int sdf_bulk_ok(const void* a, const void* b, int64_t n_lines, int64_t inner, int64_t outer_stride, int64_t stride)
{
    // every 128-line tile must be one contiguous row segment whose start and length are multiples of 16 bytes
    if (((uintptr_t)a & 15) || ((uintptr_t)b & 15) || (stride & 7) || (outer_stride & 7)) return 0;
    if (inner % SDF_THREADS) {                       // tiles may only straddle an `inner` boundary when lines are contiguous anyway
        if (!(outer_stride == 0 || outer_stride == inner)) return 0;
    }
    if ((n_lines % SDF_THREADS) & 7) return 0;       // the last, partial tile
    return 1;
}

// x and y passes of the signed transform on planes that never look across z (a z-slab can run them on its own slices):
// dyx_i16 = two (Z,H,W) int16 arrays, [0] = (y offset << 1) | occupancy bit, [1] = x offset of the nearest opposite-kind
// voxel within the voxel's own plane ([0] offset = 16383 if the plane has none).
extern "C" int64_t t3d_sdf_xy_workspace_bytes(int Z, int H, int W)
{
    return a256((int64_t)Z * H * W * 2) + sdf_stack_bytes(H, (int64_t)Z * W) + 1024;
}

extern "C" int t3d_sdf_xy(const void* occ_bits, int Z, int H, int W, const double* sampling_host, void* dyx_i16, void* workspace,
                          void* stream)
{
    if (int rc = sdf_check(Z, H, W, "t3d_sdf_xy")) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t vol = (int64_t)Z * H * W;
    const double sy = sampling_host ? sampling_host[1] : 1.0, sx = sampling_host ? sampling_host[2] : 1.0;
    char* ws = (char*)workspace;
    int16_t* ex = (int16_t*)ws; ws += a256(vol * 2);
    const int64_t rows = (int64_t)Z * H;
    k_sdf_x<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, st>>>((const uint32_t*)occ_bits, rows, W, t3d_wpr(W), ex);
    SdfPass p;
    p.in0 = ex; p.in1 = nullptr; p.out0 = (int16_t*)dyx_i16; p.out1 = (int16_t*)dyx_i16 + vol; p.sdf = nullptr;
    p.n_lines = (int64_t)Z * W; p.inner = W; p.outer_stride = (int64_t)H * W; p.stride = W; p.n = H;
    p.w_new = sy * sy; p.w0 = sx * sx; p.w1 = 0.0; p.s_new = sy; p.s0 = sx; p.s1 = 0.0;
    p.stack = (uint2*)ws;
    p.bulk = sdf_bulk_ok(p.in0, nullptr, p.n_lines, p.inner, p.outer_stride, p.stride);
    k_sdf_envelope<1, false><<<sdf_grid_blocks(p.n_lines), SDF_THREADS, 0, st>>>(p);
    T3D_CHECK_LAUNCH("t3d_sdf_xy");
    t3d_count_launches(2);
    return 0;
}

// z pass + final signed distance on full z columns (for a sharded run: the y-slab received in the all-to-all transpose)
extern "C" int64_t t3d_sdf_z_workspace_bytes(int Z, int H, int W) { return sdf_stack_bytes(Z, (int64_t)H * W) + 1024; }

extern "C" int t3d_sdf_z(const void* dy_i16, const void* dx_i16, int Z, int H, int W, const double* sampling_host, void* sdf_f32,
                         void* workspace, void* stream)
{
    if (int rc = sdf_check(Z, H, W, "t3d_sdf_z")) return rc;
    const double sz = sampling_host ? sampling_host[0] : 1.0, sy = sampling_host ? sampling_host[1] : 1.0,
                 sx = sampling_host ? sampling_host[2] : 1.0;
    SdfPass p;
    p.in0 = (const int16_t*)dy_i16; p.in1 = (const int16_t*)dx_i16; p.out0 = p.out1 = nullptr; p.sdf = (float*)sdf_f32;
    p.n_lines = (int64_t)H * W; p.inner = (int64_t)H * W; p.outer_stride = 0; p.stride = (int64_t)H * W; p.n = Z;
    p.w_new = sz * sz; p.w0 = sy * sy; p.w1 = sx * sx; p.s_new = sz; p.s0 = sy; p.s1 = sx;
    p.stack = (uint2*)workspace;
    p.bulk = sdf_bulk_ok(p.in0, p.in1, p.n_lines, p.inner, p.outer_stride, p.stride);
    k_sdf_envelope<2, true><<<sdf_grid_blocks(p.n_lines), SDF_THREADS, 0, (cudaStream_t)stream>>>(p);
    T3D_CHECK_LAUNCH("t3d_sdf_z");
    t3d_count_launches(1);
    return 0;
}

// sdf_f32 (Z,H,W) = edt(occ) - edt(~occ): +distance to the nearest unset voxel at set voxels, -distance to the nearest set
// voxel at unset ones, +-inf if the volume holds only one kind.  sampling_host: {sz, sy, sx}.
extern "C" int64_t t3d_sdf_workspace_bytes(int Z, int H, int W)
{
    const int64_t a = t3d_sdf_xy_workspace_bytes(Z, H, W), b = t3d_sdf_z_workspace_bytes(Z, H, W);
    return a256((int64_t)Z * H * W * 4) + (a > b ? a : b);
}

extern "C" int t3d_sdf(const void* occ_bits, int Z, int H, int W, const double* sampling_host, void* sdf_f32, void* workspace,
                       void* stream)
{
    if (int rc = sdf_check(Z, H, W, "t3d_sdf")) return rc;
    const int64_t vol = (int64_t)Z * H * W;
    int16_t* dyx = (int16_t*)workspace;
    char* scratch = (char*)workspace + a256(vol * 4);
    if (int rc = t3d_sdf_xy(occ_bits, Z, H, W, sampling_host, dyx, scratch, stream)) return rc;
    return t3d_sdf_z(dyx, dyx + vol, Z, H, W, sampling_host, sdf_f32, scratch, stream);
}

// ------------------------------------------------------------------------------------------------
// area-weighted vertex normals (additive: the reference discards skimage's normals, surface_extractor.py:55 vs :72)
// ------------------------------------------------------------------------------------------------
template <typename IdxT>
__global__ void __launch_bounds__(256) k_normals_accumulate(const float* __restrict__ verts, const IdxT* __restrict__ faces,
                                                            int64_t F, float* __restrict__ acc)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    const int64_t ia = faces[3 * i], ib = faces[3 * i + 1], ic = faces[3 * i + 2];
    const float* a = verts + 3 * ia; const float* b = verts + 3 * ib; const float* c = verts + 3 * ic;
    const float ux = b[0] - a[0], uy = b[1] - a[1], uz = b[2] - a[2], vx = c[0] - a[0], vy = c[1] - a[1], vz = c[2] - a[2];
    const float nx = uy * vz - uz * vy, ny = uz * vx - ux * vz, nz = ux * vy - uy * vx;
    const int64_t ids[3] = {ia, ib, ic};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        atomicAdd(acc + 3 * ids[k], nx); atomicAdd(acc + 3 * ids[k] + 1, ny); atomicAdd(acc + 3 * ids[k] + 2, nz);
    }
}

__global__ void __launch_bounds__(256) k_normals_normalize(float* __restrict__ n, int64_t V)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const float x = n[3 * i], y = n[3 * i + 1], z = n[3 * i + 2];
    const float len = sqrtf(x * x + y * y + z * z);
    if (len > 0.f) { n[3 * i] = x / len; n[3 * i + 1] = y / len; n[3 * i + 2] = z / len; }
}

extern "C" int t3d_vertex_normals(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64,
                                  void* normals_f32, void* stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (V <= 0) return 0;
    T3D_CUDA(cudaMemsetAsync(normals_f32, 0, sizeof(float) * 3 * V, st));
    if (F > 0) {
        if (faces_are_i64)
            k_normals_accumulate<long long><<<(unsigned)((F + 255) / 256), 256, 0, st>>>((const float*)verts_f32, (const long long*)faces, F, (float*)normals_f32);
        else
            k_normals_accumulate<int32_t><<<(unsigned)((F + 255) / 256), 256, 0, st>>>((const float*)verts_f32, (const int32_t*)faces, F, (float*)normals_f32);
    }
    k_normals_normalize<<<(unsigned)((V + 255) / 256), 256, 0, st>>>((float*)normals_f32, V);
    T3D_CHECK_LAUNCH("t3d_vertex_normals");
    t3d_count_launches(F > 0 ? 2 : 1);
    return 0;
}
