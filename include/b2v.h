/* b2v.h — C ABI of libb2v.so, the Blackwell-native (sm_100a) replacement for the
 * per-voxel hot path of InVesalius 3.
 *
 * Conventions (all entry points):
 *   - every pointer is a DEVICE pointer unless the parameter name ends in `_host`;
 *   - volumes are dense C-order [dz][dy][dx] (x fastest); strided / file-backed host
 *     views are packed by b2v_copy3d_* before the call;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - return value is a B2V_* status; b2v_last_error() gives the message of the
 *     last failure on the calling thread;
 *   - nothing is retained after return; scratch memory is supplied by the caller
 *     (query the size with the matching *_workspace_bytes function);
 *   - no entry point synchronises the stream unless documented.
 *
 * Each function cites the reference interface it replaces (paths relative to the
 * invesalius3 checkout).
 */
#ifndef B2V_H
#define B2V_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2V_OK 0
#define B2V_ERR_ARG 1      /* bad argument (shape, dtype code, axis, alignment) */
#define B2V_ERR_CUDA 2     /* CUDA runtime failure */
#define B2V_ERR_RANGE 3    /* value not representable (mirrors a Rust NumCast panic) */
#define B2V_ERR_NOCONV 4   /* iterative kernel hit its round cap */

/* element type codes (reference: invesalius_rs/src/types.rs:5-70) */
#define B2V_I16 0
#define B2V_U8 1
#define B2V_F64 2

/* projection kinds for b2v_mip */
#define B2V_MIP_MAX 0
#define B2V_MIP_MIN 1
#define B2V_MIP_MEAN 2

const char* b2v_last_error(void);
int b2v_version(void);
/* number of kernels launched by this library on the calling thread since the last reset */
int64_t b2v_launch_count(void);
void b2v_launch_count_reset(void);

/* ---- host<->device packing of strided views --------------------------------
 * Replaces the implicit stride handling of rust-numpy `as_array()` for callers that
 * pass `mask.matrix[1:,1:,1:]` (invesalius/data/styles.py:2493,2917,3157).
 * Copies a [dz][dy][dx] box of `elem` byte elements between a host view with byte
 * pitches (row_pitch, plane_pitch; x contiguous) and a dense device buffer. */
int b2v_copy3d_h2d(void* dst_dev, const void* src_host, int64_t dz, int64_t dy, int64_t dx, int64_t elem,
                   int64_t src_row_pitch, int64_t src_plane_pitch, void* stream);
int b2v_copy3d_d2h(void* dst_host, const void* src_dev, int64_t dz, int64_t dy, int64_t dx, int64_t elem,
                   int64_t dst_row_pitch, int64_t dst_plane_pitch, void* stream);

/* ---- threshold ---------------------------------------------------------------
 * Slice.SetMaskThreshold (whole-volume branch) invesalius/data/slice_.py:1238-1246:
 *     mask[v] = 255 if lo <= img[v] <= hi else 0               (preserve_markers = 0)
 * Slice.do_threshold_to_a_slice / do_threshold_to_all_slices slice_.py:1722-1769:
 *     same, except voxels whose OLD mask value is 1, 2, 253 or 254 keep it
 *                                                              (preserve_markers = 1)
 * img: int16 [n]; mask: uint8 [n] (read only when preserve_markers). Elementwise over
 * n voxels of a dense buffer. Algorithmic bytes: 3 B/voxel (4 with preservation). */
int b2v_threshold_i16(const int16_t* img, int64_t n, int32_t lo, int32_t hi, uint8_t* mask,
                      int preserve_markers, void* stream);
/* same on the padded Mask layout of invesalius/data/mask.py:422-431: mask has shape
 * [dz+1][dy+1][dx+1], voxel (z,y,x) at [z+1][y+1][x+1]; also sets the axial flag
 * mask[z+1][0][0] = 1 (slice_.py:1246,1767). When only_dirty != 0, slices whose flag is
 * already non-zero are skipped (slice_.py:1762-1763). */
int b2v_threshold_i16_masklayout(const int16_t* img, int64_t dz, int64_t dy, int64_t dx, int32_t lo, int32_t hi,
                                 uint8_t* mask_padded, int preserve_markers, int only_dirty, void* stream);

/* ---- intensity projections ---------------------------------------------------
 * NumPy reductions in Slice.get_image_slice, invesalius/data/slice_.py:881-886 /
 * 970-975 / 1057-1062: tmp_array.max(axis) / .min(axis) / .mean(axis).
 * img dense [dz][dy][dx] of dtype code `dtype` (int16 or uint8); axis 0/1/2.
 * out: same dtype for MAX/MIN, float64 for MEAN; shape [dy][dx] / [dz][dx] / [dz][dy].
 * workspace: b2v_mip_workspace_bytes() bytes (may be 0). 2 B/voxel for int16. */
int64_t b2v_mip_workspace_bytes(int dtype, int64_t dz, int64_t dy, int64_t dx, int axis, int kind);
int b2v_mip(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, int axis, int kind, void* out,
            void* workspace, void* stream);

/* global min/max of a dense buffer as float32 (first step of MIDA,
 * invesalius_rs/src/mips.rs:113-122). minmax_out: float[2] on the device. */
int64_t b2v_minmax_workspace_bytes(int64_t n);
int b2v_minmax_f32(const void* img, int dtype, int64_t n, float* minmax_out, void* workspace, void* stream);

/* ---- seeded flood fill / region grow -------------------------------------------
 * invesalius_rs.floodfill_threshold(data, seeds, t0, t1, fill, strct, out)
 *   invesalius_rs/__init__.py:21-40 -> src/floodfill_py.rs:137-185 -> src/floodfill.rs:96-166
 * data: dense [dz][dy][dx] of dtype code `dtype`; out: uint8, same shape, read-write.
 * seeds_host: HOST array of nseeds (x, y, z) triples (int64). A seed is used only if
 * t0 <= data[seed] <= t1. Voxels of `out` already equal to `fill` are walls. Result: every
 * voxel reachable from the valid seeds gets out = fill; everything else is untouched.
 * strct_host: HOST uint8 [odz][ody][odx], each dim <= 3; offset of entry (kk,jj,ii) is
 * (kk - odz/2, jj - ody/2, ii - odx/2) as in floodfill.rs:110-112.
 * A seed outside the volume returns B2V_ERR_RANGE (the reference panics).
 * SYNCHRONISES the stream (round control reads one flag per batch of rounds).
 * rounds_out (optional, host): number of flood rounds launched.
 * Algorithmic bytes: 4 B/voxel (int16 data 2 + out read 1 + out write 1). */
int64_t b2v_floodfill_workspace_bytes(int64_t dz, int64_t dy, int64_t dx, int64_t nseeds);
/* Convergence engine of the flood-fill family: 1 (default) = every round inside ONE
 * persistent cooperative launch (rotating bitmaps of active tiles, grid-wide barrier per
 * round), 0 = one launch per round driven from the host. Same result either way.
 * Environment knobs read once per process (tuning only, results identical): B2V_FF_TILE=8
 * (small tiles), B2V_FF_TRIPS=n (sweep sets per tile visit), B2V_FF_GRID=n (blocks of the
 * persistent grid), B2V_FF_DEFER=n (surplus tiles a round may pass on). */
void b2v_floodfill_set_engine(int persistent);
int b2v_floodfill_threshold(const void* data, int dtype, int64_t dz, int64_t dy, int64_t dx,
                            const int64_t* seeds_host, int64_t nseeds, double t0, double t1, uint8_t fill,
                            const uint8_t* strct_host, int64_t odz, int64_t ody, int64_t odx, uint8_t* out,
                            void* workspace, void* stream, int* rounds_out);
/* invesalius_rs.floodfill_threshold_inplace(data, seeds, t0, t1, fill, strct)
 *   __init__.py:43-54 -> floodfill_py.rs:187-231 -> floodfill.rs:168-237
 * Same walk, but `data` is both the tested and the written array (visited <=> data == fill). */
int b2v_floodfill_threshold_inplace(void* data, int dtype, int64_t dz, int64_t dy, int64_t dx,
                                    const int64_t* seeds_host, int64_t nseeds, double t0, double t1, double fill,
                                    const uint8_t* strct_host, int64_t odz, int64_t ody, int64_t odx,
                                    void* workspace, void* stream, int* rounds_out);
/* invesalius_rs.floodfill(data, i, j, k, v, fill, out): floodfill_py.rs:87-135 -> floodfill.rs:5-49.
 * 6-connected walk over data == v starting at (x=i, y=j, z=k); the seed is marked
 * unconditionally. */
int b2v_floodfill_equal(const void* data, int dtype, int64_t dz, int64_t dy, int64_t dx, int64_t i, int64_t j,
                        int64_t k, double v, uint8_t fill, uint8_t* out, void* workspace, void* stream,
                        int* rounds_out);
/* invesalius_rs.fill_holes_automatically(mask, labels, nlabels, max_size) -> bool
 *   floodfill_py.rs:233-249 -> floodfill.rs:51-94. mask uint8 [n] rw, labels uint32 [n].
 * modified_out (host) receives the bool. SYNCHRONISES the stream. 6 B/voxel. */
int64_t b2v_fill_holes_workspace_bytes(uint32_t nlabels);
/* In two stages for Z-sharded masks (labels of the WHOLE mask, mask.py:526-530): 1 = histogram
 * of this shard's labels into the workspace (uint32 [nlabels + 1] at byte offset 256; the shards
 * sum them with one all_reduce), 2 = qualify + apply + report. stages = 3 is b2v_fill_holes. */
int b2v_fill_holes_staged(int stages, uint8_t* mask, const uint32_t* labels, int64_t n, uint32_t nlabels,
                          uint32_t max_size, void* workspace, void* stream, int* modified_out);
int b2v_fill_holes(uint8_t* mask, const uint32_t* labels, int64_t n, uint32_t nlabels, uint32_t max_size,
                   void* workspace, void* stream, int* modified_out);

/* ---- ray-sequential projections -----------------------------------------------------
 * workspace for the three functions below: b2v_proj_workspace_bytes(dz*dy*dx) bytes.
 * All three SYNCHRONISE the stream (they report B2V_ERR_RANGE where the reference's
 * NumCast panics: NaN / out-of-range MIDA result, contour intensity overflowing T).
 * out shape: axis 0 -> [dy][dx], axis 1 -> [dz][dx], axis 2 -> [dz][dy].
 *
 * invesalius_rs.mida(image, axis, wl, ww, out): __init__.py:91-95 -> mips_py.rs:161-202 ->
 * mips.rs:102-168. dtype pairs (int16,int16), (uint8,uint8), (float64,uint8); anything else
 * is B2V_ERR_ARG ("Invalid image or output type"). wl / ww are taken AS THE IMAGE TYPE
 * (mips_py.rs:174-175). 4 B/voxel for int16 (min/max pass + ray pass). */
int64_t b2v_proj_workspace_bytes(int64_t n);
/* rays along x of int16 volumes: 1 = rows staged by the TMA engine (cp.async.bulk + mbarrier, two
 * stages), 0 = 32-bit lane loads through a padded shared-memory tile (default: measured faster,
 * profiles/README.md). Process-wide, like b2v_floodfill_set_engine. */
void b2v_proj_set_tma(int on);
int b2v_mida(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, int axis, double wl, double ww,
             void* out, int out_dtype, void* workspace, void* stream);
/* same, with the (min, max) pair of mips.rs:113-122 supplied by the caller as float[2] on
 * the device: a Z shard passes the all-reduced global pair (invesalius3_b200/dist.py). */
int b2v_mida_minmax(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, int axis, double wl, double ww,
                    const float* minmax_dev, void* out, int out_dtype, void* workspace, void* stream);
/* lmip(image, axis, tmin, tmax, out): mips.rs:7-86 (called as mips.lmip by slice_.py:892,
 * 980,1063 although the crate forgets to export it). out has the image dtype. */
int b2v_lmip(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, int axis, double tmin, double tmax,
             void* out, void* workspace, void* stream);
/* invesalius_rs.fast_countour_mip(image, n, axis, wl, ww, tmip, out): __init__.py:98-101 ->
 * mips_py.rs:204-253 -> mips.rs:215-279. int16, uint8 or float64, out of the same dtype. tmip 0:
 * max, 1: lmip(700, 3033) (uint8: B2V_ERR_RANGE, the reference panics), 2: mida (float64:
 * B2V_ERR_ARG, not built). As in the reference the contour volume tmp[z, y, x] =
 * T(calc_fcm_intensity) (mips.rs:197-242) is materialised — b2v_fcm_volume, one stencil pass,
 * sizeof(T) read + sizeof(T) written per voxel — and then projected by the same kernels as the
 * plain projections. workspace: b2v_fcm_workspace_bytes (holds the contour volume).
 * b2v_fcm_volume alone (workspace: b2v_proj_workspace_bytes) serves the Z-sharded projections:
 * computed on an extended slab, its own planes are exact. */
int64_t b2v_fcm_workspace_bytes(int dtype, int64_t dz, int64_t dy, int64_t dx, int axis, int tmip);
int b2v_fcm_volume(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, float n, int axis, void* tmp,
                   void* workspace, void* stream);
int b2v_fast_countour_mip(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, float n, int axis,
                          double wl, double ww, int tmip, void* out, void* workspace, void* stream);

/* ---- context-aware mesh smoothing (SURVEY 8f-2) ------------------------------------------------
 * invesalius_rs.context_aware_smoothing(vertices, faces, normals, T, tmax, bmin, n_iters)
 * (mesh_py.rs -> mesh.rs:27-395; Mesh.ca_smoothing, invesalius_rs/__init__.py:220-249; caller
 * invesalius/data/surface_process.py:312-320). vertices float32 [V][3], smoothed in place; faces4
 * int64 [M][4] with the leading 3; normals float32 [M][3] (per face). order: int64 [4 M], the STABLE
 * ascending argsort of the 4 M face entries (any stable sort; the host wrapper uses torch.sort).
 * The reference's quirks are kept (every column of a face row counts as a vertex id in the
 * vertex->face map; the staircase test flags every vertex that has a face). workspace:
 * b2v_ca_smoothing_workspace_bytes. SYNCHRONISES. */
int64_t b2v_ca_smoothing_workspace_bytes(int64_t nverts, int64_t nfaces);
int b2v_ca_smoothing(float* vertices, int64_t nverts, const int64_t* faces4, int64_t nfaces, const float* normals,
                     const int64_t* order, double t, double tmax, double bmin, uint32_t n_iters, void* workspace,
                     void* stream);

/* ---- pre-filters and mask algebra (SURVEY 8f-4) -------------------------------------------------
 * b2v_boolean_op: Slice.do_boolean_op (invesalius/data/slice_.py:1906-1916) on two mask bodies:
 *   op 0 union, 1 difference, 2 intersection, 3 xor; selected <=> value > 2; out = 0 / 255.
 * b2v_convolve_non_zero: invesalius_rs.convolve_non_zero (transforms_py.rs:52-93; Slice.calc_mask_area,
 *   slice_.py:2299-2322): float64 volume and kernel (device), out[p] = sum over the kernel window
 *   (cval outside the volume) where volume[p] != 0, else 0; summed in the reference's loop order.
 * b2v_median_filter_i16: scipy.ndimage.median_filter(matrix, size) with size 3, 4 or 5, mode 'reflect'
 *   (filters.py:9-12). in != out.
 * b2v_uniform_filter_i16: scipy.ndimage.uniform_filter(matrix, size) on int16 (filters.py:15-18):
 *   three separable passes, each storing trunc(window sum / size) in int16 as SciPy does when the
 *   output array is int16. tmp: a third int16 volume. All bit-exact against SciPy. */
int b2v_boolean_op(const uint8_t* m1, const uint8_t* m2, int64_t n, int op, uint8_t* out, void* stream);
int b2v_convolve_non_zero(const double* volume, int64_t sz, int64_t sy, int64_t sx, const double* kernel_dev, int64_t skz,
                          int64_t sky, int64_t skx, double cval, double* out, void* stream);
int b2v_median_filter_i16(const int16_t* in, int64_t nz, int64_t ny, int64_t nx, int size, int16_t* out, void* stream);
int b2v_uniform_filter_i16(const int16_t* in, int64_t nz, int64_t ny, int64_t nx, int size, int16_t* out, int16_t* tmp,
                           void* stream);
/* The Gaussian-based filters of filters.py (gaussian_blur :5-6, sharpening :21-29, despeckle :32-36,
 * border detection :39-66) are built from scipy.ndimage.correlate1d evaluated exactly as SciPy's
 * NI_Correlate1D does for symmetric (symmetry = +1) and antisymmetric (-1) odd kernels: tmp = x[c] w[0];
 * for jj = -radius .. -1: tmp += (x[c + jj] +/- x[c - jj]) w[jj]; float64; 'reflect'; an int16 output
 * takes the C cast. weights_dev: 2 radius + 1 centred float64 weights on the device (for a Gaussian:
 * scipy.ndimage._filters._gaussian_kernel1d, reversed). dtype pairs (int16,int16), (int16,float64),
 * (float64,float64). b2v_sharpen_i16, b2v_sobel_magnitude, b2v_rescale_cast_i16: the elementwise
 * float64 statements around them, in NumPy's order. Bit-exact against SciPy. */
int b2v_correlate1d(const void* in, int in_dtype, int64_t nz, int64_t ny, int64_t nx, int axis, const double* weights_dev,
                    int radius, int symmetry, void* out, int out_dtype, void* stream);
int b2v_sharpen_i16(const int16_t* img, const double* blurred, int64_t n, double value, double lo, double hi, int16_t* out,
                    void* stream);
int b2v_sobel_magnitude(double* sx_inout, const double* sy, const double* sz, int64_t n, void* stream);
int b2v_rescale_cast_i16(const double* m, int64_t n, int rescale, double mag_min, double mag_range, double span,
                         double min_val, int16_t* out, void* stream);

/* ---- connected components (SURVEY 8f-3) ------------------------------------------------------
 * b2v_label: scipy.ndimage.label(input, structure, output=uint32) as InVesalius calls it
 * (invesalius/data/mask.py:526-530, 549-552; imagedata_utils.py:717-721): input uint8, non-zero =
 * feature; strct_host uint8, 1 or 3 wide per axis, centrosymmetric (else B2V_ERR_ARG, SciPy raises
 * too); labels uint32, numbered in raster order of each component's first voxel like SciPy.
 * *nlabels_host receives the count. SYNCHRONISES. workspace: b2v_label_workspace_bytes(n voxels).
 * b2v_count_regions: invesalius_rs.count_regions (count_regions.rs:5-18): out[p] = number of voxels
 * holding image[p]'s value; values outside [0, number_regions] are B2V_ERR_RANGE (the reference
 * panics). workspace: 256 + 4 * (number_regions + 1) bytes. */
int64_t b2v_label_workspace_bytes(int64_t n);
int b2v_label(const uint8_t* input, int64_t nz, int64_t ny, int64_t nx, const uint8_t* strct_host, int64_t odz, int64_t ody,
              int64_t odx, uint32_t* labels, void* workspace, void* stream, int64_t* nlabels_host);
int b2v_count_regions(const void* image, int dtype, int64_t n, uint32_t number_regions, uint32_t* out, void* workspace,
                      void* stream);

/* ---- view-matrix resampling (SURVEY 8f-1) --------------------------------------------
 * invesalius_rs.apply_view_matrix_transform(volume, spacing, M, n, orientation, minterpol, cval,
 * out): __init__.py:84 -> transforms_py.rs:96-148 -> transforms.rs:9-55 -> interpolation.rs.
 * out[cz, cy, cx] samples `volume` at M * (z sz, y sy, x sx, 1) with (z, y, x) = the output
 * index shifted by n along the slab axis (orientation 0 AXIAL: z, 1 CORONAL: y, 2 SAGITAL: x,
 * anything else: no shift); minterpol 0 nearest, 1 trilinear, 2 tricubic, else Lanczos-4; outside
 * [0, d - 1) on any axis: cval. float64 arithmetic in the reference's order. spacing_host =
 * (sx, sy, sz), m_host = 16 doubles row-major, both on the HOST. volume / out: dense device
 * arrays of the same dtype (int16, uint8, float64). workspace: >= 256 bytes. SYNCHRONISES (a value
 * that does not fit the output type is B2V_ERR_RANGE: the reference panics). */
int b2v_apply_view_matrix_transform(const void* volume, int dtype, int64_t dz, int64_t dy, int64_t dx,
                                    const double* spacing_host, const double* m_host, int64_t n, int orientation,
                                    int minterpol, double cval, void* out, int64_t odz, int64_t ody, int64_t odx,
                                    void* workspace, void* stream);

/* ---- 3-D mask editor (invesalius/data/mask3d_editor_state.py) --------------------------------
 * float64 in the reference's operation order throughout (no FMA, IEEE division and sqrt).
 *
 * b2v_mask_cut: invesalius_rs.mask_cut (mask_cut.rs:7-62). out: dense device uint8 [dz][dy][dx],
 * edited in place. Each voxel > 127 at (z, y, x) maps p = (x sx, y sy, z sz, 1) through M and MV;
 * when (M p)[3] > 0 and |MV p / (MV p)[3]| <= max_depth it becomes 0 if its screen position
 * (px, py) = ((q0 / 2 + 0.5)(w - 1), (q1 / 2 + 0.5)(h - 1)) lies on the filter and
 * filter[trunc py][trunc px] != 0, or if it lies off the filter and edit_mode == 0.
 * filter: dense device uint8 [h][w] (may be NULL when h * w == 0). spacing_host = (sx, sy, sz),
 * m_host / mv_host = 16 doubles row-major, all on the HOST. Does not synchronise. */
int b2v_mask_cut(uint8_t* out, int64_t dz, int64_t dy, int64_t dx, const double* spacing_host, double max_depth,
                 const uint8_t* filter, int64_t h, int64_t w, const double* m_host, const double* mv_host, int edit_mode,
                 void* stream);
/* The voxel box brush_mask.rs:24-31 visits for a sphere of `radius` at center_host = (cx, cy, cz)
 * (millimetres) in a [dz][dy][dx] volume with spacing_host = (sx, sy, sz): box_host receives
 * (z0, y0, x0, nz, ny, nx), all zero when the box is empty. Host only: no device work. */
int b2v_brush_bbox(int64_t dz, int64_t dy, int64_t dx, const double* spacing_host, const double* center_host,
                   double radius, int64_t* box_host);
/* b2v_brush_mask: invesalius_rs.brush_mask_rs (brush_mask.rs:5-71) applied to the part of a
 * [dz][dy][dx] volume held on the device as the box [oz, oz + bz) x [oy, oy + by) x [ox, ox + bx):
 * out (and orig, when not NULL) are dense device uint8 [bz][by][bx] copies of that box. Voxels in
 * both the box and b2v_brush_bbox's box with (dx^2 + dy^2) + dz^2 <= radius^2: edit_mode 1 sets
 * those > 0 to 0; edit_mode 0 sets them to orig when orig > 0, or to 255 without orig; any other
 * mode does nothing. Does not synchronise. */
int b2v_brush_mask(uint8_t* out, const uint8_t* orig, int64_t bz, int64_t by, int64_t bx, int64_t oz, int64_t oy,
                   int64_t ox, int64_t dz, int64_t dy, int64_t dx, const double* spacing_host, const double* center_host,
                   double radius, int edit_mode, void* stream);
/* b2v_polygons_raster: invesalius_rs.polygon2mask_rs (polygon_mask.rs:4-79) for k >= 1 polygons at
 * once on a (w, h) screen. points: device float64 [total][2] (x, y); offsets: device int64 [k + 1],
 * polygon p is points[offsets[p] .. offsets[p + 1]). Pixel (r < w, c < h) is the even-odd
 * inside(px = r, py = c) OR-ed over the polygons (each inside its own bounding box), XOR negate.
 * transpose == 0 writes out[r][c] (uint8 [w][h], polygon2mask_rs's layout); transpose != 0 writes
 * out[c][r] (uint8 [h][w], the filter of b2v_mask_cut). workspace: b2v_polygons_workspace_bytes(k)
 * device bytes. Does not synchronise. */
int64_t b2v_polygons_workspace_bytes(int64_t k);
int b2v_polygons_raster(const double* points, const int64_t* offsets, int64_t k, int64_t w, int64_t h, int transpose,
                        int negate, uint8_t* out, void* workspace, void* stream);

/* ---- marching cubes ---------------------------------------------------------------
 * Replaces the contour step of create_surface_piece, invesalius/data/surface_process.py:
 * 156-186 (vtkImageFlip about the origin + vtkContourFilter at iso 127 on the uint8 mask,
 * or at tmin / tmax on the int16 image); geometry as converters.to_vtk, converters.py:34-101.
 * vol: dense [nz][ny][nx] uint8 or int16. inside(p) <=> vol[p] >= iso.
 * Two calls sharing one caller-owned workspace:
 *   b2v_mc_count  classifies, scans and returns the vertex / triangle counts (host);
 *                 SYNCHRONISES the stream.
 *   b2v_mc_emit   writes verts float32 [V][3] and tris int32 [T][3] (shared vertices).
 * Vertex (i + ox [+t], j + oy [+t], k + oz [+t]) * (sx, sy, sz), y negated when flip_y
 * (and the winding reversed, so normals keep pointing from inside to outside);
 * t = (iso - s0) / (s1 - s0) in float32. Canonical ordering: see DESIGN.md.
 * Algorithmic bytes: 1 B/voxel (uint8) or 2 B/voxel (int16) + 12 B per vertex + 12 B per
 * triangle. */
int64_t b2v_mc_workspace_bytes(int64_t nz, int64_t ny, int64_t nx);
int b2v_mc_count(const void* vol, int dtype, int64_t nz, int64_t ny, int64_t nx, double iso, void* workspace,
                 void* stream, int64_t* nverts_host, int64_t* ntris_host);
int b2v_mc_emit(const void* vol, int dtype, int64_t nz, int64_t ny, int64_t nx, double iso, const void* workspace,
                float sx, float sy, float sz, int32_t ox, int32_t oy, int32_t oz, int flip_y, float* verts,
                int32_t* tris, void* stream);

/* ---- watershed -------------------------------------------------------------------------
 * do_watershed, invesalius/data/watershed_process.py:19-60.
 * b2v_ws_lut_i16: get_LUT_value(image, ww, wl).astype('uint16'), invesalius/data/
 *   imagedata_utils.py:555-564 (float64 piecewise, truncated into int16, reinterpreted).
 * b2v_ws_shift_i16: (image - image.min()).astype('uint16') (watershed_process.py:50,55);
 *   workspace: b2v_ws_workspace_bytes.
 * b2v_ws_morph_gradient_u16: scipy.ndimage.morphological_gradient(pre, size=(sz,sy,sx)),
 *   mode 'reflect' (watershed_process.py:36,49). Bit-exact against SciPy.
 * b2v_ws_flood: mode 0 = scipy.ndimage.watershed_ift cost model (max |dI| along the path),
 *   mode 1 = skimage.segmentation.watershed cost model (max I along the path). markers
 *   int16 (0 = unlabeled); labels int16 out. Exact minimax costs; labels follow cost-optimal
 *   edges, ties resolved by hop count then smaller label (the reference's ties follow its
 *   queue order: see DESIGN.md section 6). ambiguous (uint8, optional, may be NULL): 1 where two
 *   different labels can reach the voxel along cost-optimal edges, i.e. where the reference's
 *   answer is an artefact of its queue order; everywhere else (0) the labelling IS the
 *   reference's, whatever its order. SYNCHRONISES the stream. strct_host: uint8, dims
 *   1 or 3. 14 B/voxel for the whole do_watershed as the reference defines it. */
int b2v_ws_lut_i16(const int16_t* img, int64_t n, double window, double level, uint16_t* out, void* stream);
int b2v_ws_shift_i16(const int16_t* img, int64_t n, uint16_t* out, void* workspace, void* stream);
int b2v_ws_morph_gradient_u16(const uint16_t* in, int64_t nz, int64_t ny, int64_t nx, int sz, int sy, int sx,
                              uint16_t* out, void* stream);
int64_t b2v_ws_workspace_bytes(int64_t nz, int64_t ny, int64_t nx);
int b2v_ws_flood(const uint16_t* img, const int16_t* markers, int64_t nz, int64_t ny, int64_t nx,
                 const uint8_t* strct_host, int64_t odz, int64_t ody, int64_t odx, int mode, int16_t* labels,
                 uint8_t* ambiguous, void* workspace, void* stream, int* rounds_out);

/* The flood in stages, for Z-sharded volumes (6-connected only; dist.watershed drives it). The slab
 * passed in is an extended slab: with frozen_lo / frozen_hi its first / last plane is a halo plane
 * that is never relaxed locally; b2v_ws_plane reads a plane (merge = 0) or merges a neighbour's
 * values into one (merge = 1: minimum of the costs / of the keys, join of the label sets; tiles
 * next to a voxel that changed are queued for the next *_CONVERGE; *changed_host = 1 if any did).
 * what = 0: uint32 costs (phase 1); what = 1: uint64 keys followed by uint16 label sets (phase 2);
 * plane buffers are device memory of b2v_ws_plane_bytes(ny, nx, what) bytes.
 * stages (bit mask, executed in this order): 1 INIT, 2 COST_CONVERGE, 4 LABEL_BEGIN (admissible
 * predecessors from the final costs), 8 LABEL_CONVERGE, 16 FINISH (labels + ambiguous mask out).
 * *rounds_io accumulates the rounds. Every *_CONVERGE synchronises the stream.
 * b2v_ws_shift_i16_with: (image - min).astype('uint16') with the minimum supplied on the device
 * (minmax_dev[0], float32: the global minimum of a sharded volume after its all_reduce). */
int b2v_ws_flood_staged(int stages, const uint16_t* img, const int16_t* markers, int64_t nz, int64_t ny, int64_t nx,
                        int mode, int frozen_lo, int frozen_hi, int16_t* labels, uint8_t* ambiguous, void* workspace,
                        void* stream, int* rounds_io);
int64_t b2v_ws_plane_bytes(int64_t ny, int64_t nx, int what);
int b2v_ws_plane(int merge, int what, int64_t nz, int64_t ny, int64_t nx, int mode, int frozen_lo, int frozen_hi,
                 int64_t z, void* plane, void* workspace, void* stream, int* changed_host);
int b2v_ws_shift_i16_with(const int16_t* img, int64_t n, const float* minmax_dev, uint16_t* out, void* stream);
/* diagnostics of the persistent engine: [0..2] phase-1 tile visits / sweep sets / visits that
 * changed something, [4..6] the same for phase 2; reset != 0 clears them */
int b2v_ws_stats(int* out8, int reset);

/* ---- Z-sharded volumes (one shard per GPU; invesalius3_b200/dist.py drives these) ---------
 * The reference's only decomposition is the Z-piece split of the surface step
 * (invesalius/data/surface.py:1360-1381: pieces of 20 slices + 1 overlap, stitched by
 * vtkAppendPolyData + vtkCleanPolyData, surface_process.py:229-268). Here every shard holds
 * a slab plus one halo plane per inner side.
 *
 * Flood fill in stages (bit 0 BEGIN: build + seeds, bit 1 CONVERGE: rounds from *round_io,
 * bit 2 FINISH: write). Between CONVERGE calls the caller exchanges the reached bits of the
 * shared planes with its neighbours (byte offsets from b2v_floodfill_layout: [0] passable
 * bits, [1] reached bits, [2] round flags (int32 each), [3] bytes per z-plane, [4] tiles,
 * [5] round capacity) and ORs them in with b2v_floodfill_merge_plane, which re-activates
 * the touched tiles for round `round` and raises flags[round]. */
int b2v_floodfill_threshold_staged(int stages, const void* data, int dtype, int64_t dz, int64_t dy, int64_t dx,
                                   const int64_t* seeds_host, int64_t nseeds, double t0, double t1, uint8_t fill,
                                   const uint8_t* strct_host, int64_t odz, int64_t ody, int64_t odx, uint8_t* out,
                                   void* workspace, void* stream, int* round_io);
int b2v_floodfill_layout(int64_t dz, int64_t dy, int64_t dx, int64_t nseeds, int64_t* layout_out);
int b2v_floodfill_merge_plane(int64_t dz, int64_t dy, int64_t dx, int64_t nseeds, void* workspace, int64_t z,
                              const uint32_t* plane_bits, int round, void* stream);
/* Marching cubes on a slab whose last plane is shared with the next shard: that plane's
 * vertices are owned (numbered, emitted) by the next shard. b2v_mc_layout (layout_out[4]): [0]
 * byte offset of the dense plane-0 records {cx, cy, cz, vertex offset} in the workspace (filled
 * by b2v_mc_count_shard), [1] their size in bytes, [2] byte offset of the uint64 totals (V, T).
 * The emitting shard receives the next shard's plane-0 records and global
 * vertex base; concatenating the shards' outputs in rank order reproduces the single-GPU
 * output bit for bit (the boundary stitch). */
int b2v_mc_count_shard(const void* vol, int dtype, int64_t nz, int64_t ny, int64_t nx, double iso,
                       int skip_last_plane, void* workspace, void* stream, int64_t* nverts_host,
                       int64_t* ntris_host);
int b2v_mc_emit_shard(const void* vol, int dtype, int64_t nz, int64_t ny, int64_t nx, double iso,
                      const void* workspace, float sx, float sy, float sz, int32_t ox, int32_t oy, int32_t oz,
                      int flip_y, int skip_last_plane, int32_t vertex_base, const void* next_shard_plane0_records,
                      int32_t next_shard_vertex_base, float* verts, int32_t* tris, void* stream);
int b2v_mc_layout(int64_t nz, int64_t ny, int64_t nx, int64_t* layout_out);

/* ---- peer mailboxes: the NVLink exchange layer of the Z-sharded ops ------------------------------
 * Replaces the temp-file exchange between the reference's worker processes
 * (invesalius/data/surface.py:1360-1430 pieces -> surface_process.py:229-268 stitch;
 * invesalius/data/styles.py:2083-2108 watershed child). One process per GPU; every rank owns one
 * MAILBOX in its HBM (b2v_peer_alloc: cudaMalloc + cudaIpc export), maps every other rank's
 * (b2v_peer_open) and hands the array of the `world` base pointers (its own included, index =
 * rank) to the *_peer entry points. Ranks only WRITE into peers (stores over NVLink + a release
 * store of a signal word) and poll their own mailbox, with a time-out (B2V_ERR_NOCONV), so a
 * mismatched call sequence cannot hang a GPU. `epoch` is a job-wide counter >= 1 that every rank
 * advances identically: b2v_floodfill_threshold_peer reports how many epochs it consumed, the
 * other calls consume one. Layout and protocol: invesalius3_b200/csrc/peer.cuh.
 * b2v_peer_mailbox_bytes(dy, dx): size for shards whose planes are dy x dx voxels; the
 * `mailbox_plane_bytes` argument of the calls below is dy * ceil(dx / 32) * 4 of that link. */
int64_t b2v_peer_mailbox_bytes(int64_t dy, int64_t dx);
int b2v_peer_alloc(int64_t bytes, void** dev_ptr_out, uint8_t* handle_out /* [64] */);
int b2v_peer_open(const uint8_t* handle /* [64] */, void** dev_ptr_out);
int b2v_peer_close(void* mapped_ptr);
int b2v_peer_free(void* dev_ptr);
/* all ranks meet (consumes one epoch); the self-check of a new link. Synchronises the stream. */
int b2v_peer_barrier(int rank, int world, const void* const* mailboxes_host, int64_t mailbox_plane_bytes,
                     uint32_t epoch, void* stream);
/* invesalius_rs.floodfill_threshold over one Z shard with the boundary exchange FUSED into the
 * persistent flood kernel: data / out are the extended slab (own planes + one halo plane per
 * inner side, halo planes of data valid), seeds are local to it (a shard without seeds passes
 * nseeds = 0 and still takes part). After local convergence the kernel pushes the reached bits
 * of the two planes around each inner boundary into the neighbours' mailboxes, merges what they
 * pushed, all ranks agree whether anyone gained a bit, and the rounds resume — ONE launch per
 * GPU for the whole sharded flood, no host round trip. Synchronises the stream (verdict). */
int b2v_floodfill_threshold_peer(const void* data, int dtype, int64_t dz, int64_t dy, int64_t dx,
                                 const int64_t* seeds_host, int64_t nseeds, double t0, double t1, uint8_t fill,
                                 const uint8_t* strct_host, int64_t odz, int64_t ody, int64_t odx, uint8_t* out,
                                 void* workspace, void* stream, int rank, int world,
                                 const void* const* mailboxes_host, int64_t mailbox_plane_bytes, uint32_t epoch,
                                 int* rounds_out, int* epochs_used_out);
/* b2v_mc_count_shard + the exchange the stitch needs, in one stream-ordered sequence: every
 * rank's (V, T) lands in counts_host [world][2], and the upper neighbour's plane-0 records land
 * in this rank's mailbox at byte offset b2v_peer_mc_inbox_offset(plane_bytes, epoch) — pass that
 * device address as next_shard_plane0_records to b2v_mc_emit_shard. Synchronises the stream. */
int b2v_mc_count_shard_peer(const void* vol, int dtype, int64_t nz, int64_t ny, int64_t nx, double iso,
                            int skip_last_plane, void* workspace, void* stream, int rank, int world,
                            const void* const* mailboxes_host, int64_t mailbox_plane_bytes, uint32_t epoch,
                            int64_t* counts_host);
int64_t b2v_peer_mc_inbox_offset(int64_t mailbox_plane_bytes, uint32_t epoch);
/* MIDA (mips.rs:102-168) / LMIP (mips.rs:7-86) with rays along z over ONE Z shard: the rays
 * cross the shards, so each shard continues from the per-ray state its predecessor left and
 * hands its own on (the per-ray operation order is that of the whole-volume walk: bit-exact).
 * state: device uint32 [3][dy][dx] — MIDA: (fmax, alpha, colour) as float bits; LMIP: running
 * maximum (two words), then bit 0 "inside [tmin, tmax] seen", bit 1 "ray finished".
 * first != 0: this slab starts the rays (state is written, not read); last != 0: it ends
 * them and writes out [dy][dx] (otherwise out may be NULL). minmax_dev: device float[2], the
 * GLOBAL (min, max) of the volume. b2v_mida_z_partial synchronises the stream (range check). */
int b2v_mida_z_partial(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, double wl, double ww,
                       const float* minmax_dev, uint32_t* state, int first, int last, void* out, int out_dtype,
                       void* workspace, void* stream);
int b2v_lmip_z_partial(const void* img, int dtype, int64_t dz, int64_t dy, int64_t dx, double tmin, double tmax,
                       uint32_t* state, int first, int last, void* out, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2V_H */
