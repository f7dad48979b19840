/*
 * t3d.h -- C ABI of libt3d.so: the B200 (sm_100a) reconstruction hot path of
 * victorramirez952/tomography_3d_reconstructor.
 *
 * Boundary.  The reference is pure Python; its hot path is three classes (voxel_processor.py:27,
 * surface_extractor.py:28, volume_calculator.py:10) whose arithmetic is delegated to numpy / scipy.ndimage /
 * scikit-image.  This library replaces exactly those delegated calls.  The Python classes of the same names
 * in tomography_3d_reconstructor_b200/ bind it through ctypes (see INTEGRATION.md); every entry point below
 * cites the reference line(s) it replaces.
 *
 * Conventions
 *   - plain C, no torch types; `stream` is a cudaStream_t passed as void* (0 = default stream);
 *   - pointers are DEVICE pointers unless the parameter name ends in `_host`;
 *   - volumes are C-contiguous (Z, H, W); occupancy is bit-packed along x, LSB first, row stride
 *     t3d_words_per_row(W) = ceil(W/32) uint32 words, bits at x >= W are zero;
 *   - every function returns 0 on success; otherwise t3d_last_error() describes the failure
 *     (1 = CUDA error, 2 = invalid argument).  Nothing here falls back to the CPU.
 *   - variable-size outputs use count -> caller allocates -> emit.
 */
#ifndef T3D_H
#define T3D_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* t3d_last_error(void);
int t3d_version(void);
int64_t t3d_words_per_row(int W);
/* number of kernels of this library launched so far by this process (bench.py gpu_launches) */
int64_t t3d_launch_count(void);
void t3d_count_launches(int n);

/* ---- VoxelProcessor.create_voxel_data  (voxel_processor.py:36-54) -------------------------------------- */

/* image_loader.py:108 `img >= threshold` + np.stack (voxel_processor.py:46).  masks: uint8 (Z,H,W); numpy bool
 * masks use threshold = 1.  bits: (Z,H,wpr) uint32. */
int t3d_pack_masks(const void* masks_u8, int Z, int H, int W, int threshold, void* bits, void* stream);

/* The same threshold + stack fused with the z loop of _close_volume_ends (voxel_processor.py:72-75: out[z] = v[z] | (v[z-1] & v[z+1])
 * for 1 <= z <= Z-2) and with np.sum per slice / the np.where extrema of volume_calculator.py:62-79, in one pass over the
 * masks (the kernel of the single-enqueue path that streams the uint8 stack).  The end planes are written raw: the caller
 * hole-fills them and rewrites planes 0, 1, Z-2, Z-1 (what t3d_reconstruct does).  Requires Z >= 3, W % 128 == 0, a 16-byte
 * aligned stack and 1 <= threshold <= 255 (returns 2 otherwise).  counts_u64: Z per-slice counts or NULL; bbox_u32x6:
 * {INT_MAX - zmin, zmax + 1, INT_MAX - ymin, ymax + 1, INT_MAX - xmin, xmax + 1} or NULL.  Both are accumulated into with
 * atomics (add / max): the CALLER zeroes them beforehand (the call itself is this one kernel and nothing else). */
int t3d_pack_gap(const void* masks_u8, int Z, int H, int W, int threshold, void* bits, void* counts_u64, void* bbox_u32x6,
                 void* stream);

/* inverse: numpy-bool view of a packed volume (the ndarray the reference API returns). out: uint8 (Z,H,W) 0/1 */
int t3d_unpack_bits(const void* bits, int Z, int H, int W, void* out_u8, void* stream);

/* scipy.ndimage.binary_fill_holes on 2-D planes, in place (voxel_processor.py:60-70).  Planes are
 * plane_stride_words apart; scratch: t3d_fill_holes_scratch_bytes(n_planes, H, W) bytes. */
int64_t t3d_fill_holes_scratch_bytes(int n_planes, int H, int W);
int t3d_fill_holes_2d(void* bits, int n_planes, int64_t plane_stride_words, int H, int W, void* scratch, void* stream);

/* z loop of _close_volume_ends (voxel_processor.py:72-75): out[z] = in[z] | (in[z-1] & in[z+1]), end planes
 * copied.  lo_plane / hi_plane (may be NULL): neighbour planes of a z-slab (multi-GPU).  slice_counts_u64
 * (may be NULL): Z per-slice popcounts of the result (np.sum, voxel_processor.py:51). */
int t3d_gap_fill(const void* in_bits, void* out_bits, const void* lo_plane, const void* hi_plane, int Z, int H, int W,
                 void* slice_counts_u64, void* stream);

/* ---- VoxelProcessor.smooth_voxel_data  (voxel_processor.py:79-97) -------------------------------------- */

/* n_stages 6-connected erosions (bit s of erode_mask = 1; outside = True) / dilations (0; outside = False), one
 * launch per stage: skimage.morphology.binary_opening = stages {E,D}, binary_closing = {D,E}; opening then closing
 * = {E,D,D,E} = n_stages 4, erode_mask 0b1001.  Out of place; scratch: t3d_morph_scratch_bytes(...) bytes. */
int64_t t3d_morph_scratch_bytes(int Z, int H, int W, int n_stages);
int t3d_morph(const void* in_bits, void* out_bits, int Z, int H, int W, int n_stages, unsigned erode_mask,
              void* slice_counts_u64, void* scratch, void* stream);

/* ---- VolumeCalculator  (volume_calculator.py:16-94) ----------------------------------------------------- */

/* per-slice np.sum (volume_calculator.py:31-33) and np.where min/max (:39-44, :62-79).
 * slice_counts_u64: Z uint64; bbox_i32x6: zmin,zmax,ymin,ymax,xmin,xmax (INT_MAX/-1 if empty). Either may be NULL. */
int t3d_volume_stats(const void* bits, int Z, int H, int W, void* slice_counts_u64, void* bbox_i32x6, void* stream);

/* ---- VoxelProcessor.generate_point_cloud  (voxel_processor.py:99-127) ----------------------------------- */
int t3d_row_popcounts(const void* bits, int Z, int H, int W, void* row_counts_u32, void* stream);
int t3d_point_cloud_emit(const void* bits, int Z, int H, int W, const void* row_base_u64, int subsample,
                         const void* z_centre_mm_f64, double mm_per_pixel_y, double mm_per_pixel_x, void* out_f64,
                         void* stream);

/* generic exclusive scan of n_arrays uint32 arrays of n_cap elements, `stride` elements apart (array k at in + k*stride),
 * into uint32 (out_is_u64 = 0) or uint64 (1) arrays of the same layout; popcount_input = 1 scans popcount(in[i]).
 * totals_u64: n_arrays uint64.  n_dev_u64: the true length in device memory (at most n_cap); NULL = the capacity is the size. */
int64_t t3d_scan_workspace_bytes(int64_t n, int n_arrays);
int t3d_exclusive_scan_u32_dev(const void* in, void* out, int64_t n_cap, int64_t stride, int n_arrays, int out_is_u64,
                               int popcount_input, const void* n_dev_u64, void* totals_u64, void* workspace, void* stream);

/* ---- SurfaceExtractor.extract_manifold_surface  (surface_extractor.py:34-75) ---------------------------- */

/* Sign of (float32(gaussian_filter(float64(pad(occ)), 0.5)) - 0.5) packed in padded coordinates
 * (Z+2p, H+2p, wpr(W+2p)); surface_extractor.py:43-53 + the `> 0` test of marching cubes.  weights3_host: the three
 * scipy kernel weights {centre, +-1, +-2} (NULL = the sigma 0.5 constants). */
int t3d_field_sign(const void* occ_bits, int Z, int H, int W, int pad, const double* weights3_host, void* sign_bits,
                   void* n_exact_u64, void* stream);

/* Same sign volume through a leaner kernel: the (rare) words that need the exact evaluation are recorded in
 * exc_list_u64 (exc_cap entries) and patched by a second small kernel.  exc_count_u64 (device) = recorded words; if it
 * exceeds exc_cap the result is incomplete and t3d_field_sign must be run instead. */
int t3d_field_sign_lean(const void* occ_bits, int Z, int H, int W, int pad, const double* weights3_host, void* sign_bits,
                        void* n_exact_u64, void* exc_list_u64, uint32_t exc_cap, void* exc_count_u64, void* stream);

/* Two-pass marching cubes on a sign volume (Zs,Hs,Ws) = skimage.measure.marching_cubes(volume, 0.5), sparse after the
 * first dense pass (see csrc/t3d_mc.cu).  The data-dependent sizes stay in device memory, in the block
 * sizes_u64 = {n_active, n_x, n_y, n_z, n_t} that the two scans write their totals into; arrays are capacity-sized
 * (cap_active, cap_verts, cap_faces) and nothing is written beyond a capacity, so the whole sequence needs no host round
 * trip and can be graph-captured.  A caller that has read the sizes back passes capacities equal to them.
 *   t3d_mc_flags        -> ballots_u32[t3d_mc_num_chunks]: bit l of word c set iff sign word 32c+l owns a cut edge or an
 *                          active cube origin
 *   (caller) t3d_exclusive_scan_u32_dev of popcount(ballots) -> chunkbase_u32, total n_active -> sizes_u64[0]
 *   t3d_mc_words_dev    -> aw_idx_u32[n_active] (flat word index) and aw_cnt_u32[4][cap_active] (owned x/y/z cut edges,
 *                          triangles); n_ambiguous_u64: cubes tiled through Lewiner's face / interior tests (mc_field)
 *   (caller) t3d_exclusive_scan_u32_dev of aw_cnt -> aw_base_u32, totals n_x, n_y, n_z, n_t -> sizes_u64[1..4]
 *   t3d_mc_emit_dev     -> vkeys_u64[n_x+n_y+n_z] (edge key per vertex) and faces_i32 (n_t,3): reference cube order,
 *                          reversed winding (gradient_direction='descent')
 *   t3d_mc_vertices_dev -> verts_f32 (V,3) [z,y,x]: skimage's interpolation on the exact float64 field, then un-pad,
 *                          variable-depth z map and mm scaling (surface_extractor.py:57-65, 82-113).
 * z_begin/z_end: owned planes of the sign volume ([0, Zs) on one device; -1 = Zs).  With z-slab sharding a rank owns
 * [z_begin, z_end) and additionally emits the x/y-edge vertices of ghost plane z_end; z_offset is the global padded
 * plane index of local padded plane 0. */
/* The marched field as the ambiguity tests of t3d_mc_words_dev / t3d_mc_emit_dev see it.  Cubes whose index has an ambiguous
 * face (Lewiner's cases 3, 6, 7, 10, 12, 13) or is case 4 are tiled by the row that Lewiner's face test (asymptotic decider) and
 * interior test select (csrc/mc33_tables.h; oracle/mc_ref.c restates the same decisions); both need the corner VALUES:
 *   field_f32 != NULL: dense float32 field of the sign volume's own shape (Z,H,W), marched at `level`;
 *   else occ_bits != NULL: Gaussian(0.5) (gaussian = 1) of the occupancy (Z,H,W) padded by `pad`, as for t3d_mc_vertices_dev;
 *   NULL struct: only the signs are known (values level +- 0.5: every face test is a tie -> positive corners joined). */
typedef struct t3d_mc_field {
    const void* occ_bits;
    int Z, H, W, pad, gaussian;
    const double* weights3_host;
    const void* field_f32;
    double level;
} t3d_mc_field;

int64_t t3d_mc_num_chunks(int Zs, int Hs, int Ws);
int t3d_mc_flags(const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end, void* ballots_u32, void* stream);
int t3d_mc_words_dev(const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end, const void* ballots_u32,
                     const void* chunkbase_u32, uint32_t cap_active, const void* sizes_u64, void* aw_idx_u32, void* aw_cnt_u32,
                     void* n_ambiguous_u64, const t3d_mc_field* mc_field, void* stream);
/* parts 1: vertex keys; 2: faces (the words without an ambiguous cube, then the others: two launches); 3: both in one launch */
int t3d_mc_emit_dev(const void* sign_bits, int Zs, int Hs, int Ws, int z_begin, int z_end, const void* ballots_u32,
                    const void* chunkbase_u32, const void* aw_idx_u32, const void* aw_base_u32, uint32_t cap_active,
                    const void* sizes_u64, uint32_t cap_verts, uint32_t cap_faces, void* vkeys_u64, void* faces_i32,
                    int parts, const t3d_mc_field* mc_field, void* stream);
/* Field: occ_bits as t3d_field_sign had it (pad / gaussian; gaussian = 0: the sign volume IS the occupancy and pad must be 0,
 * level 0.5), or field_f32 != NULL: the dense (Z,H,W) field the sign volume was taken from (t3d_sign_from_f32), at `level`.
 * cum/adj: device float64 arrays of the variable-slice-depth z map (n_cum = 0 disables it). */
int t3d_mc_vertices_dev(const void* occ_bits, int Z, int H, int W, int pad, int gaussian, const double* weights3_host,
                        const void* field_f32, double level, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts,
                        int unpad_shift, int z_offset, const void* cum_f64, const void* adj_f64, int n_cum, double mm_per_pixel_y,
                        double mm_per_pixel_x, int scale_in_f64, int which_blocks /* 1: x-edge, 2: y-edge, 4: z-edge vertices */,
                        void* verts_f32, void* stream);

/* test aids: the float32 field itself and the uint8 cube-case volume */
int t3d_field_dense(const void* occ_bits, int Z, int H, int W, int pad, int gaussian, const double* weights3_host,
                    void* out_f32, void* stream);
int t3d_cube_cases(const void* sign_bits, int Zs, int Hs, int Ws, void* out_u8, void* stream);

/* _ensure_manifold_mesh (surface_extractor.py:115-126): np.unique rows + degenerate-face drop.
 * counts_u64[0] = V', [1] = F'. */
int64_t t3d_canonicalize_workspace_bytes(int64_t V, int64_t F);
int t3d_mesh_canonicalize(const void* verts_in, int64_t V, const void* faces_in, int64_t F, void* verts_out,
                          void* faces_out_i64, void* faces_out_i32, void* counts_u64, void* workspace, void* stream);

/* Same outputs for meshes in t3d_mc_emit_dev's vertex order ([x|y|z]-edge blocks, raster order inside each): ONE stable
 * 64-bit (z,y)-key sort; counts_u64 has 3 entries, [2] != 0 = ordering not verified, call t3d_mesh_canonicalize.
 * V_dev_u64 / F_dev_u64: the true vertex / face counts in device memory (at most the capacities); NULL = the capacity is
 * the size. */
int64_t t3d_canonicalize_fast_workspace_bytes(int64_t V, int64_t F);
int t3d_mesh_canonicalize_fast_dev(const void* verts_in, int64_t V_cap, const void* V_dev_u64, const void* faces_in, int64_t F_cap,
                                   const void* F_dev_u64, void* verts_out, void* faces_out_i64, void* faces_out_i32,
                                   void* counts_u64, void* workspace, void* stream);
/* Structured canonical order (same outputs as t3d_mesh_canonicalize_fast_dev, a third of the sorting work): uses the
 * vertex keys of t3d_mc_emit_dev.  x-edge vertices are already in order, y-edge vertices are ranked inside their (plane, row
 * gap) segment, z-edge vertices get one stable radix sort by (layer, z) over cap_z entries, final positions come from
 * the per-row prefix counts of the emit pass (chunkbase_u32 / aw_base_u32 with array stride aw_stride, as passed to
 * t3d_mc_emit_dev; Zs,Hs,Ws = the marched sign volume).  The vertices the z map clamps onto z = 0 (surface_extractor.py:100-103;
 * non-empty only when the object touches slice 0) are ordered by a generic (y,x) sort over cap_g0 entries (0 = not
 * provisioned).  sizes_u64 = {n_active, n_x, n_y, n_z, n_t}; Zs / z_offset / unpad_shift / n_cum as for t3d_mc_vertices_dev.
 * counts_u64[2] != 0: order not verified (level model broken by rounding, cap_z or cap_g0 too small) -> fall back.
 * zkey_bits (0 = 32): the z keys are sorted as (layer, key(z) - key(z of the layer's lower plane)) truncated to that many
 * bits -- the caller bounds the span of one layer from the z map (fewer radix passes); a wrong bound only fails the
 * verification.  phases: 1 = only the z-edge sort (needs only the z-edge vertices; can run on another stream while the
 * other vertices are still being computed), 2 = everything after it, 3 = both. */
int64_t t3d_canonicalize_structured_workspace_bytes(int64_t V, int64_t F, uint32_t cap_z, uint32_t cap_g0, int Zs);
int t3d_mesh_canonicalize_structured_dev(const void* verts_in, const void* vkeys_u64, int64_t V_cap, const void* sizes_u64,
                                         const void* V_dev_u64, int Zs, int Hs, int Ws, const void* chunkbase_u32,
                                         const void* aw_base_u32, uint32_t aw_stride, int z_offset, int unpad_shift,
                                         const void* cum_f64, const void* adj_f64, int n_cum, int zkey_bits, uint32_t cap_z,
                                         uint32_t cap_g0, const void* faces_in, int64_t F_cap, const void* F_dev_u64,
                                         void* verts_out, void* faces_out_i64, void* faces_out_i32, void* counts_u64,
                                         void* n_g0_u64, void* workspace, int phases, void* stream);

/* calculate_mesh_volume / calculate_surface_area (surface_extractor.py:128-148): out_f64 = {signed volume, area}.  F_dev_u64:
 * the true face count in device memory (at most F_cap); NULL = the capacity is the size. */
int64_t t3d_mesh_measure_workspace_bytes(void);
int t3d_mesh_measure_dev(const void* verts_f32, const void* faces, int64_t F_cap, const void* F_dev_u64, int faces_are_i64,
                         void* out_f64, void* workspace, void* stream);

/* The whole hot path in the order tomography_3d_reconstruction.py runs it (create_voxel_data :88-100, smooth + extract +
 * mesh volume :120-140, surface area :207-223, analyze :225-229) as ONE enqueue on `stream` (plus an internal side stream,
 * forked/joined with events): uint8 masks (Z,H,W) -> verts_out_f32 (cap_verts,3) / faces_out_i64 (cap_faces,3) in canonical
 * order + the result block results_u64[t3d_reconstruct_results_len(Z)]:
 *   [0] n_active [1] n_x [2] n_y [3] n_z [4] n_t (raw faces) [5] V' [6] F' [7] fast ordering unverified [8] overflow bits
 *   (1: active words, 2: vertices, 4: faces exceeded their capacity -> retry larger) [9] ambiguous cubes [10] exact field
 *   evaluations [11] signed mesh volume (f64) [12] area (f64) [13..15] bbox int32 x 6 [16] raw vertices [17] recorded
 *   exact-evaluation words (overflow bit 8 if above the internal list capacity).  On overflow nothing is emitted: slots
 *   [0..4] and [16] read 0 and the sizes that did not fit are kept in [20..24].  [25] size of the z-clamp group of the
 *   canonical ordering (t3d_mesh_canonicalize_structured_dev): [7] != 0 with [25] > cap_g0 -> retry with a larger cap_g0.
 * cap_zverts: capacity for the z-edge vertices ([3]); cap_zverts = 0 selects the generic 64-bit sort
 * (t3d_mesh_canonicalize_fast_dev) instead of the structured ordering; zkey_bits as for
 * t3d_mesh_canonicalize_structured_dev (0 = no bound known).
 *   [32 .. 32+Z) per-slice voxel counts after close_ends, [32+Z .. 32+2Z) after smoothing.
 * n_stages/erode_mask as t3d_morph (0 stages = no smoothing).  cum/adj: device float64 z-map arrays. */
int64_t t3d_reconstruct_workspace_bytes(int Z, int H, int W, int add_padding, int n_stages, uint32_t cap_active,
                                        uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0);
int64_t t3d_reconstruct_results_len(int Z);
int t3d_reconstruct(const void* masks_u8, int Z, int H, int W, int threshold, int close_ends, int n_stages, unsigned erode_mask,
                    int add_padding, const double* weights3_host, const void* cum_f64, const void* adj_f64, int n_cum,
                    double mm_per_pixel_y, double mm_per_pixel_x, int scale_in_f64, uint32_t cap_active, uint32_t cap_verts,
                    uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0, int zkey_bits, void* verts_out_f32,
                    void* faces_out_i64, void* results_u64, void* workspace, void* stream);

/* z-slab variant of t3d_reconstruct for one rank of a sharded run (SURVEY.md 8e; host side: sharded.py).  ext_bits holds
 * halo_lo + n_own + halo_hi bit-planes: the rank's own packed slices (global end slices already hole-filled) between the
 * planes received from its z-neighbours.  Gap fill and morphology are recomputed on the halo; the surface is marched on
 * min(3, halo) planes either side with z_begin/z_end (owned planes of the local padded sign volume, as t3d_mc_flags) and
 * z_offset (global plane index of local surface plane 0, as t3d_mc_vertices_dev).  The result block is t3d_reconstruct's with
 * Zx = halo_lo + n_own + halo_hi per-plane counts twice from slot 32 (bbox is over the own planes, local z), plus
 *   [18] ghost tail: canonical vertices with z == z_ghost (the next rank's first plane), if want_ghost
 *   [19] lead: canonical vertices with z == z_lead (this rank's first plane), if want_lead.
 * t3d_slab_pack packs the own slices (uint8, n_own x H x W) into ext_bits and fills the holes of the global end slices
 * (fill_first / fill_last; fill_scratch = t3d_fill_holes_scratch_bytes(2, H, W)) on an internal side stream, which
 * t3d_reconstruct_slab joins when join_fill != 0 -- the halo exchange in between does not wait for it.
 * Pre-filled mode (pre_grid_bits and pre_stats_u64 non-NULL in BOTH calls; allowed when t3d_slab_pack_gap_ok returns 1: at
 * least 16 own slices, W % 128 == 0, 16-byte aligned masks, 1 <= threshold <= 255): the own planes [4, n_own - 4) depend on
 * no neighbour, so t3d_slab_pack sends them through the one-pass kernel of t3d_pack_gap straight into pre_grid_bits (a
 * halo_lo + n_own + halo_hi plane bit volume) with their counts / extrema in pre_stats_u64 (that many + 3 uint64), and packs
 * only the 8 own planes at either end raw into ext_bits (what the halo exchange sends); t3d_reconstruct_slab then gap-fills
 * just the two ends into pre_grid_bits.  Same results as the plain mode; the uint8 stack is read once. */
int t3d_slab_pack_gap_ok(const void* masks_u8, int n_own, int H, int W, int threshold);
int t3d_slab_pack(const void* masks_u8, int n_own, int H, int W, int threshold, int halo_lo, int halo_hi, int fill_first,
                  int fill_last, void* ext_bits, void* fill_scratch, void* pre_grid_bits, void* pre_stats_u64, void* stream);
int64_t t3d_reconstruct_slab_workspace_bytes(int halo_lo, int n_own, int halo_hi, int H, int W, int add_padding, int n_stages,
                                             uint32_t cap_active, uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts,
                                             uint32_t cap_g0);
int t3d_reconstruct_slab(const void* ext_bits, int halo_lo, int n_own, int halo_hi, int H, int W, int n_stages,
                         unsigned erode_mask, int add_padding, int z_begin, int z_end, int z_offset, int want_ghost, float z_ghost,
                         int want_lead, float z_lead, int join_fill, const double* weights3_host, const void* cum_f64, const void* adj_f64,
                         int n_cum, double mm_per_pixel_y, double mm_per_pixel_x, int scale_in_f64, uint32_t cap_active,
                         uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0, int zkey_bits,
                         void* verts_out_f32, void* faces_out_i64, void* results_u64, void* workspace, void* pre_grid_bits,
                         const void* pre_stats_u64, void* stream);
/* faces_i64[0 .. 3*F'[rank]) += sum over lower ranks of (V' - ghost tail), read from the all-gathered result blocks
 * (world x stride_u64 uint64 on the device): local vertex ids -> ids in the stitched mesh. */
int t3d_slab_stitch_faces(void* faces_i64, int64_t cap_faces, const void* gathered_results_u64, int64_t stride_u64, int rank,
                          void* stream);

/* ---- additive stages (no reference counterpart; SURVEY.md 8a-16, 8b) ------------------------------------- */

/* Exact Euclidean distance transform (oracle: scipy.ndimage.distance_transform_edt(occ, sampling)): dist_f32 (Z,H,W) =
 * sign * distance between voxel centres from every foreground voxel (bit set; bit clear if invert) to the nearest
 * voxel of the other kind, 0 there, inf if there is none; accumulate != 0 adds into dist_f32.  sampling_host = {sz, sy,
 * sx} (NULL = 1,1,1).  sdf = t3d_edt(invert 0, sign +1) then t3d_edt(invert 1, sign -1, accumulate 1). */
int64_t t3d_edt_workspace_bytes(int Z, int H, int W);
/* The two halves of t3d_edt, for z-slab sharding (SURVEY.md 8e): the x and y passes never look across planes, so every
 * rank runs t3d_edt_xy on its own slices (dyx_i16 = two (Z,H,W) int16 arrays back to back: y offset, then x offset of
 * the nearest site in the plane); after the all-to-all transpose z-slabs -> y-slabs, t3d_edt_z runs the z pass and the
 * final distance on full z columns (Z = all slices, H = rows of the rank's y-slab). */
int64_t t3d_edt_xy_workspace_bytes(int Z, int H, int W);
int t3d_edt_xy(const void* occ_bits, int Z, int H, int W, int invert, const double* sampling_host, void* dyx_i16, void* workspace,
               void* stream);
int64_t t3d_edt_z_workspace_bytes(int Z, int H, int W);
int t3d_edt_z(const void* dy_i16, const void* dx_i16, int Z, int H, int W, const double* sampling_host, float sign, int accumulate,
              void* dist_f32, void* workspace, void* stream);
int t3d_edt(const void* occ_bits, int Z, int H, int W, int invert, const double* sampling_host, float sign, int accumulate,
            void* dist_f32, void* workspace, void* stream);

/* Half-ellipsoid end-cap slices (ellipsoid_slice_generator.py:61-77): out_u8 (n,H,W), slice k = cv2.warpAffine(base, M_k,
 * INTER_LINEAR, constant border 0) in OpenCV's own fixed-point arithmetic (bit-identical; csrc/t3d_generator.cu);
 * inv_matrices_f64 = 6 float64 per slice (device), already inverted the way cv::warpAffine inverts its argument; an all-zero
 * matrix gives an all-zero slice. */
int t3d_endcap_slices(const void* base_u8, int H, int W, const void* inv_matrices_f64, int n, void* out_u8, void* stream);

/* Signed distance in one sweep per axis (csrc/t3d_edt.cu): sdf_f32 (Z,H,W) = edt(occ) - edt(~occ) -- +distance to the nearest
 * unset voxel at set voxels, -distance to the nearest set voxel at unset ones (scipy's arithmetic, bit-equal at unit sampling),
 * +-inf if only one kind exists.  t3d_sdf_xy / t3d_sdf_z are its two halves for z-slab sharding: dyx_i16 = two (Z,H,W) int16
 * arrays, [0] = (y offset << 1) | occupancy bit, [1] = x offset of the nearest opposite-kind voxel in the voxel's own plane;
 * the z pass runs on full columns (after the all-to-all transpose).  Extents up to 16382 per axis. */
int64_t t3d_sdf_xy_workspace_bytes(int Z, int H, int W);
int t3d_sdf_xy(const void* occ_bits, int Z, int H, int W, const double* sampling_host, void* dyx_i16, void* workspace, void* stream);
int64_t t3d_sdf_z_workspace_bytes(int Z, int H, int W);
int t3d_sdf_z(const void* dy_i16, const void* dx_i16, int Z, int H, int W, const double* sampling_host, void* sdf_f32, void* workspace,
              void* stream);
int64_t t3d_sdf_workspace_bytes(int Z, int H, int W);
int t3d_sdf(const void* occ_bits, int Z, int H, int W, const double* sampling_host, void* sdf_f32, void* workspace, void* stream);

/* Marching a dense float32 field directly (e.g. the SDF): sign bits = (field > level) packed like an occupancy volume, then
 * the marching-cubes entry points above on them with the field passed as field_f32 (mc_field, t3d_mc_vertices_dev). */
int t3d_sign_from_f32(const void* field_f32, int Z, int H, int W, double level, void* sign_bits, void* stream);

/* area-weighted unit vertex normals (the reference discards skimage's normals, surface_extractor.py:55 vs :72) */
int t3d_vertex_normals(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64, void* normals_f32,
                       void* stream);

/* Field-gradient vertex normals (DESIGN.md §2): n = -(Gz/dz, Gy/mm_y, Gx/mm_x) / |.|, float32 (V', 3) [z, y, x], G = the
 * np.gradient of the marched field at the two end nodes of the vertex's grid edge blended with the vertex kernel's weight t,
 * dz = slope of the variable-depth z map at the vertex (1 without one).  Outward: from field > level to field < level.
 * Field source as t3d_mc_vertices_dev (occ_bits, pad, gaussian; level 0.5) or, if field_f32 != NULL, that dense (Z,H,W) field
 * at `level`.  vkeys / sizes_u64 / unpad_shift / z_offset / adj (n_cum = the z map's cum length, 0 = none) as for the vertex
 * kernel; nothing runs when the raw vertex count n_x + n_y + n_z exceeds cap_verts.  newid_u32 (NULL: raw order) scatters row i
 * to its canonical slot; perm_u32 (NULL: no vertices were merged) is the canonicalisation's sorted order and selects the tie
 * rule: a slot that several raw vertices merged into takes the normal of the one with the smallest edge key (z, y, x, axis).
 * dup_u64 (optional): the unique pass's "equal pair seen" flag -- the tie pass returns at once while it reads 0.  winner_u32:
 * scratch of V' entries (tie pass).  The map, the order, the flag and a dead scratch range of each canonicalisation's
 * workspace are found with t3d_canonical_map_offsets. */
int t3d_mc_normals_dev(const void* occ_bits, int Z, int H, int W, int pad, int gaussian, const double* weights3_host,
                       const void* field_f32, double level, const void* vkeys_u64, const void* sizes_u64, uint32_t cap_verts,
                       int unpad_shift, int z_offset, const void* adj_f64, int n_cum, double mm_per_pixel_y, double mm_per_pixel_x,
                       const void* newid_u32, const void* perm_u32, const void* dup_u64, void* winner_u32, void* normals_f32,
                       void* stream);
/* byte offsets in a canonicalisation's workspace, out4 = {newid (raw -> slot, u32), perm (sorted position -> raw id, u32),
 * a u32 scratch of >= V entries dead after the call, "equal pair seen" flag (u64; -1 = none)}; valid once the call finished.
 * kind 0: t3d_mesh_canonicalize (V, F); 1: t3d_mesh_canonicalize_fast_dev (V, F); 2: the structured variant with the same
 * (V, F, cap_z, cap_g0, Zs) it was sized with. */
int t3d_canonical_map_offsets(int kind, int64_t V, int64_t F, uint32_t cap_z, uint32_t cap_g0, int Zs, int64_t* out4);
/* Post-step of t3d_reconstruct (same stream, same geometry, capacities and workspace, enqueued after it): field-gradient
 * normals of the step's canonical mesh into normals_out_f32 (cap_verts, 3), rows [0, V') valid.  Writes nothing else. */
int t3d_reconstruct_normals(int Z, int H, int W, int n_stages, unsigned erode_mask, int add_padding, const double* weights3_host,
                            const void* adj_f64, int n_cum, double mm_per_pixel_y, double mm_per_pixel_x, uint32_t cap_active,
                            uint32_t cap_verts, uint32_t cap_faces, uint32_t cap_zverts, uint32_t cap_g0, const void* results_u64,
                            void* workspace, void* normals_out_f32, void* stream);

/* ---- connected components (additive) --------------------------------------------------------------------- */

/* Connected components of an occupancy volume, labelled over x-runs (maximal stretches of set bits in one row;
 * csrc/t3d_label.cu).  connectivity 6 = scipy.ndimage.generate_binary_structure(3, 1), 26 = np.ones((3, 3, 3)).
 *   t3d_cc_count   -> row_base_u32[Z*H + 1]: index of each row's first run, [Z*H] = R; n_runs_u64 (device) = R.
 *   (caller reads R and allocates)
 *   t3d_cc_label   -> runs_i32 = three int32 arrays of R back to back: x_begin | x_end (inclusive) | row (z*H + y), raster
 *                     order; run_label_i32[R] = the label of each run, n_components_u64 (device) = K.  Labels are those of
 *                     scipy.ndimage.label(occ, structure): components numbered 1..K in raster (z, y, x) order of their first
 *                     voxel, independent of the order the device merges in.  R must fit int32 (returns 2 naming R
 *                     otherwise, nothing is truncated); K <= R.
 *   t3d_cc_stats   -> counts_i64[K] = np.bincount(labels.ravel())[1:]; bbox_i32 (K, 6) = {zmin, zmax, ymin, ymax, xmin, xmax}
 *                     inclusive = scipy.ndimage.find_objects with stop - 1.
 *   t3d_cc_volumes -> volumes_f64[K]: volume_calculator.py:23-35 applied to each component alone (labels == c):
 *                     sum over z ascending, z < n_slices, of count[c, z] * slice_volumes_f64[z] in float64 without FMA
 *                     contraction; slice_volumes_f64[z] = mm_x * mm_y * slice_depths[z] as the reference forms it (caller);
 *                     bbox_i32 as t3d_cc_stats left it.  Workspace: t3d_cc_volumes_workspace_bytes(R, K).
 *   t3d_cc_expand  -> labels_i32 (Z, H, W) dense: the scipy.ndimage.label array itself.
 *   t3d_cc_select  -> out_bits (Z, H, wpr) packed: the voxels whose component has keep_u8[label] != 0 (keep_u8: K + 1 bytes,
 *                     [0] ignored), padding words written zero. */
int64_t t3d_cc_count_workspace_bytes(int Z, int H);
int t3d_cc_count(const void* bits, int Z, int H, int W, void* row_base_u32, void* n_runs_u64, void* workspace, void* stream);
int64_t t3d_cc_label_workspace_bytes(int64_t n_runs);
int t3d_cc_label(const void* bits, int Z, int H, int W, int connectivity, const void* row_base_u32, int64_t n_runs, void* runs_i32,
                 void* run_label_i32, void* n_components_u64, void* workspace, void* stream);
int t3d_cc_stats(const void* runs_i32, const void* run_label_i32, int64_t n_runs, int H, int64_t n_components, void* counts_i64,
                 void* bbox_i32, void* stream);
int64_t t3d_cc_volumes_workspace_bytes(int64_t n_runs, int64_t n_components);
int t3d_cc_volumes(const void* runs_i32, const void* run_label_i32, int64_t n_runs, int H, int64_t n_components, const void* bbox_i32,
                   const void* slice_volumes_f64, int n_slices, void* volumes_f64, void* workspace, void* stream);
int t3d_cc_expand(const void* bits, int Z, int H, int W, const void* row_base_u32, const void* run_label_i32, void* labels_i32,
                  void* stream);
int t3d_cc_select(const void* bits, int Z, int H, int W, const void* row_base_u32, const void* run_label_i32, const void* keep_u8,
                  void* out_bits, void* stream);

/* ---- mesh bodies (additive) ------------------------------------------------------------------------------ */

/* Connected bodies of a triangle mesh: verts_f32 (V, 3), faces (F, 3) int32 or int64 (faces_are_i64).  A body is a connected
 * component of the graph with the edges f0-f1 and f0-f2 of every face (csrc/t3d_label.cu).  V and the body count B must fit
 * int32 and F must be at most 2^31 - 1 (status 2 naming the size otherwise, before any memory is touched).
 *   t3d_mesh_bodies_workspace_bytes(V, F, B): enough for any of the calls below; before B is known pass B = 0 (labelling).
 *   t3d_mesh_bodies_label     -> vertex_body_i32[V] = scipy.sparse.csgraph.connected_components(G, directed=False)[1]: bodies
 *                                numbered 0..B-1 by their smallest vertex, independent of the order the device merges in; a
 *                                vertex used by no face is a body of its own.  n_bodies_u64: two device uint64, [0] = B,
 *                                [1] = faces with an index outside [0, V) (skipped; the other calls need it to be 0).
 *   (caller reads B and allocates)
 *   t3d_mesh_bodies_stats     -> per body: vertex_counts_i64, face_counts_i64 (faces whose f0 is in the body),
 *                                first_vertex_i64 (its smallest vertex), bbox_f32 (B, 6) {zmin, zmax, ymin, ymax, xmin, xmax} of
 *                                its vertex columns (a zero bound is +0.0), and volumes_f64 / areas_f64: the sum over its faces of
 *                                the terms of t3d_mesh_measure_dev (float64, left to right, no FMA contraction), each rounded
 *                                half-to-even to a multiple of 2^-64 and added exactly in 128-bit fixed point, the sum rounded
 *                                once to float64.  Bit-identical in any launch order.  Reads one word back at its end: if a
 *                                |term| >= 2^62 or F * max|term| >= 2^63 (the sums could leave 128 bits) it returns 2 naming the
 *                                bound, and the sums are not valid.
 *   t3d_mesh_bodies_face_body -> face_body_i32[F] = vertex_body[faces[f, 0]].
 *   t3d_mesh_bodies_select    -> the vertices (and normal rows, if normals_f32 is not NULL) of the bodies with keep_u8[b] != 0
 *                                and their faces, each in input order; faces (input dtype) renumbered to the kept vertices.
 *                                The caller sizes the outputs from the counts of t3d_mesh_bodies_stats. */
int64_t t3d_mesh_bodies_workspace_bytes(int64_t V, int64_t F, int64_t B);
int t3d_mesh_bodies_label(const void* faces, int64_t F, int faces_are_i64, int64_t V, void* vertex_body_i32, void* n_bodies_u64,
                          void* workspace, void* stream);
int t3d_mesh_bodies_stats(const void* verts_f32, const void* faces, int64_t F, int faces_are_i64, int64_t V, const void* vertex_body_i32,
                          int64_t B, void* vertex_counts_i64, void* face_counts_i64, void* first_vertex_i64, void* bbox_f32,
                          void* volumes_f64, void* areas_f64, void* workspace, void* stream);
int t3d_mesh_bodies_face_body(const void* faces, int64_t F, int faces_are_i64, const void* vertex_body_i32, void* face_body_i32,
                              void* stream);
int t3d_mesh_bodies_select(const void* verts_f32, const void* normals_f32, const void* faces, int64_t F, int faces_are_i64, int64_t V,
                           const void* vertex_body_i32, int64_t B, const void* keep_u8, void* verts_out_f32, void* normals_out_f32,
                           void* faces_out, void* workspace, void* stream);

/* ---- mesh smoothing (additive) --------------------------------------------------------------------------- */

/* Vertex adjacency and Taubin smoothing of a triangle mesh: verts_f32 (V, 3), faces (F, 3) int32 or int64 (faces_are_i64)
 * (csrc/t3d_smooth.cu).  V must fit int32 (the neighbour ids) and F must be at most (2^32 - 1) / 6 = 715 827 882 (the raw
 * entries, up to 6 per face, are counted in 32 bits); otherwise status 2 naming the size, before any memory is touched.
 *   t3d_mesh_adjacency_workspace_bytes(V, F): the workspace of both adjacency calls; emit reads what count left in it.
 *   t3d_mesh_adjacency_count -> offsets_i64[V + 1]: CSR row offsets of the neighbours, [V] = N; n_u64: two device uint64,
 *                               [0] = N, [1] = faces with an index outside [0, V) (skipped; the result needs it to be 0).
 *                               The neighbours of i are the distinct j != i that share a face edge with i (each face
 *                               (a, b, c) gives the edges {a,b}, {b,c}, {c,a}), in ascending order.
 *   (caller reads N and allocates)
 *   t3d_mesh_adjacency_emit  -> neighbours_i32[N].
 *   t3d_mesh_taubin          -> verts_out_f32 (V, 3): `iterations` steps of trimesh.smoothing.filter_taubin with equal
 *                               weights, from the float32 input in float64: s = +0.0, s = s + w * x[j] over the neighbours
 *                               in ascending order (w = 1.0 / degree), dd = s - x[i], x[i] + lamb * dd on even steps and
 *                               x[i] - nu * dd on odd ones, every vertex from the previous iterate, no FMA contraction; a
 *                               vertex without neighbours keeps its position; rounded once to float32 at the end.
 *                               iterations >= 0 and finite lamb / nu (status 2 otherwise).  verts_out must not overlap verts.
 *                               Workspace: t3d_mesh_taubin_workspace_bytes(V). */
int64_t t3d_mesh_adjacency_workspace_bytes(int64_t V, int64_t F);
int t3d_mesh_adjacency_count(const void* faces, int64_t F, int faces_are_i64, int64_t V, void* offsets_i64, void* n_u64,
                             void* workspace, void* stream);
int t3d_mesh_adjacency_emit(int64_t V, int64_t F, const void* offsets_i64, void* neighbours_i32, void* workspace, void* stream);
int64_t t3d_mesh_taubin_workspace_bytes(int64_t V);
int t3d_mesh_taubin(const void* verts_f32, int64_t V, const void* offsets_i64, const void* neighbours_i32, int iterations, double lamb,
                    double nu, void* verts_out_f32, void* workspace, void* stream);

/* ---- device-side mesh consumers: the step right after the path (SURVEY.md 8f-3) ----------------------------- */

/* glb_exporter.py:52-91 create_layer_colors: rgba_u8 (V,4) = grey (200,200,200,255); red where first_start <= z <=
 * first_end (if has_first); blue where last_start <= z <= last_end (if has_last; blue wins), z = vertex column 0 compared
 * in float64 as numpy does. */
int t3d_layer_colors(const void* verts_f32, int64_t V, int has_first, double first_start, double first_end, int has_last,
                     double last_start, double last_end, void* rgba_u8, void* stream);

/* obj_exporter.py:25-31 as text formatting on the device, two-phase: t3d_obj_measure computes every line's length and
 * their scan into `workspace` and the total (device uint64); the caller allocates total + 1 bytes; t3d_obj_emit writes
 * "v %.6f %.6f %.6f\n" per vertex, one blank line, "f a b c\n" (1-based) per face -- byte-identical to the reference's
 * loop (the two comment lines and the blank line in front of the body stay with the host). */
int64_t t3d_obj_workspace_bytes(int64_t V, int64_t F);
/* glb_exporter.py:26-50 (trimesh's GLB export of Trimesh(vertices, faces, vertex_colors) after fix_normals()): the binary
 * chunk of a glTF 2.0 file assembled on the device: [uint32 indices (3F) | float32 positions (3V) | uint8 RGBA (4V, only
 * if rgba_u8)]; flip_winding reverses every face (fix_normals() of a closed mesh whose signed volume is negative);
 * minmax_f32x6 = per-column minima then maxima of the positions (required on the POSITION accessor). */
int64_t t3d_glb_payload_bytes(int64_t V, int64_t F, int with_colors);
int t3d_glb_pack(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64, const void* rgba_u8,
                 int flip_winding, void* bin_out, void* minmax_f32x6, void* stream);
int t3d_obj_measure(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64, void* total_len_u64,
                    void* workspace, void* stream);
int t3d_obj_emit(const void* verts_f32, int64_t V, const void* faces, int64_t F, int faces_are_i64, const void* total_len_u64,
                 const void* workspace, void* out_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* T3D_H */
