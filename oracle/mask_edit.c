/* CPU checker — TEST INFRASTRUCTURE ONLY (never linked into the product).
 *
 * The three native functions of the 3-D mask editor (invesalius/data/mask3d_editor_state.py:14),
 * restated in C from their semantics: mask_cut (mask_cut.rs:7-62), brush_mask_rs (brush_mask.rs:5-71)
 * and polygon2mask_rs (polygon_mask.rs:4-79). One thread, plain loops over every voxel / pixel,
 * float64 in the reference's operation order (-ffp-contract=off), Rust's saturating float -> integer
 * casts and the release crate's wrapping integer arithmetic. The reference holds no test for these
 * functions: PARITY UNPINNED (restated, not pinned). Arrays are addressed through element strides. */
#include <math.h>
#include <stdint.h>

static uint64_t as_usize(double v) {
  if (v != v || v <= 0.0) return 0;
  if (v >= 18446744073709551616.0) return UINT64_MAX;
  return (uint64_t)v;
}

static int64_t as_isize(double v) {
  if (v != v) return 0;
  if (v >= 9223372036854775808.0) return INT64_MAX;
  if (v <= -9223372036854775808.0) return INT64_MIN;
  return (int64_t)v;
}

/* f64::max / f64::min: a NaN operand yields the other one */
static double rmax(double a, double b) { return a != a ? b : (b != b ? a : (a > b ? a : b)); }
static double rmin(double a, double b) { return a != a ? b : (b != b ? a : (a < b ? a : b)); }

static void mat_vec(const double* m, const double p[4], double r[4]) {
  for (int i = 0; i < 4; ++i) r[i] = ((m[4 * i] * p[0] + m[4 * i + 1] * p[1]) + m[4 * i + 2] * p[2]) + m[4 * i + 3] * p[3];
}

void orc_mask_cut(uint8_t* out, const int64_t* os, int64_t dz, int64_t dy, int64_t dx, double sx, double sy, double sz,
                  double max_depth, const uint8_t* mask, const int64_t* ms, int64_t h, int64_t w, const double* m,
                  const double* mv, int edit_mode) {
  const double wm1 = (double)(uint64_t)(w - 1), hm1 = (double)(uint64_t)(h - 1);
  for (int64_t z = 0; z < dz; ++z)
    for (int64_t y = 0; y < dy; ++y)
      for (int64_t x = 0; x < dx; ++x) {
        uint8_t* v = out + z * os[0] + y * os[1] + x * os[2];
        if (!(*v > 127)) continue;
        const double p[4] = {(double)x * sx, (double)y * sy, (double)z * sz, 1.0};
        double q_[4], c_[4], q[4], c[4];
        mat_vec(m, p, q_);
        if (!(q_[3] > 0.0)) continue;
        mat_vec(mv, p, c_);
        for (int i = 0; i < 4; ++i) { q[i] = q_[i] / q_[3]; c[i] = c_[i] / c_[3]; }
        const double dist = sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
        if (!(dist <= max_depth)) continue;
        const double px = (q[0] / 2.0 + 0.5) * wm1, py = (q[1] / 2.0 + 0.5) * hm1;
        if (px >= 0.0 && px < (double)w && py >= 0.0 && py < (double)h) {
          if (mask[(int64_t)as_usize(py) * ms[0] + (int64_t)as_usize(px) * ms[1]]) *v = 0;
        } else if (edit_mode == 0) {
          *v = 0;
        }
      }
}

/* Returns 0, or 1 where the reference panics (orig indexed outside its shape). */
int orc_brush_mask(uint8_t* out, const int64_t* os, int64_t d, int64_t h, int64_t w, const uint8_t* orig,
                   const int64_t* gs, int64_t gd, int64_t gh, int64_t gw, const double* spacing, const double* center,
                   double radius, int edit_mode) {
  if (d == 0 || h == 0 || w == 0) return 0;
  const double sx = spacing[0], sy = spacing[1], sz = spacing[2];
  const double cx = center[0], cy = center[1], cz = center[2];
  const uint64_t min_x = as_usize(rmax(floor((cx - radius) / sx), 0.0));
  const uint64_t max_x = as_usize(rmin(rmax(ceil((cx + radius) / sx), 0.0), (double)(uint64_t)(w - 1)));
  const uint64_t min_y = as_usize(rmax(floor((cy - radius) / sy), 0.0));
  const uint64_t max_y = as_usize(rmin(rmax(ceil((cy + radius) / sy), 0.0), (double)(uint64_t)(h - 1)));
  const uint64_t min_z = as_usize(rmax(floor((cz - radius) / sz), 0.0));
  const uint64_t max_z = as_usize(rmin(rmax(ceil((cz + radius) / sz), 0.0), (double)(uint64_t)(d - 1)));
  const double radius_sq = radius * radius;
  for (uint64_t z = 0; z < (uint64_t)d; ++z)
    for (uint64_t y = 0; y < (uint64_t)h; ++y)
      for (uint64_t x = 0; x < (uint64_t)w; ++x) {
        if (!(z >= min_z && z <= max_z && y >= min_y && y <= max_y && x >= min_x && x <= max_x)) continue;
        uint8_t* v = out + (int64_t)z * os[0] + (int64_t)y * os[1] + (int64_t)x * os[2];
        const double ddx = (double)x * sx - cx, ddy = (double)y * sy - cy, ddz = (double)z * sz - cz;
        const double dist_sq = ddx * ddx + ddy * ddy + ddz * ddz;
        if (edit_mode == 1) {
          if (*v > 0 && dist_sq <= radius_sq) *v = 0;
        } else if (edit_mode == 0 && dist_sq <= radius_sq) {
          if (orig) {
            if ((int64_t)z >= gd || (int64_t)y >= gh || (int64_t)x >= gw) return 1;
            const uint8_t o = orig[(int64_t)z * gs[0] + (int64_t)y * gs[1] + (int64_t)x * gs[2]];
            if (o > 0) *v = o;
          } else {
            *v = 255;
          }
        }
      }
  return 0;
}

/* out: dense [w][h] bytes, out[r * h + c] = inside(px = r, py = c); pts through element strides. */
void orc_polygon2mask(int64_t w, int64_t h, const double* pts, const int64_t* ps, int64_t n, uint8_t* out) {
  for (int64_t i = 0; i < w * h; ++i) out[i] = 0;
  if (n == 0 || w == 0 || h == 0) return;
  double min_px = 1.7976931348623157e308, max_px = -1.7976931348623157e308, min_py = min_px, max_py = max_px;
  for (int64_t i = 0; i < n; ++i) {
    const double x = pts[i * ps[0]], y = pts[i * ps[0] + ps[1]];
    if (x < min_px) min_px = x;
    if (x > max_px) max_px = x;
    if (y < min_py) min_py = y;
    if (y > max_py) max_py = y;
  }
  int64_t lo_r = (int64_t)((uint64_t)as_isize(floor(min_px)) - 1u), hi_r = (int64_t)((uint64_t)as_isize(ceil(max_px)) + 1u);
  int64_t lo_c = (int64_t)((uint64_t)as_isize(floor(min_py)) - 1u), hi_c = (int64_t)((uint64_t)as_isize(ceil(max_py)) + 1u);
  lo_r = lo_r < 0 ? 0 : lo_r; hi_r = hi_r < 0 ? 0 : hi_r; lo_c = lo_c < 0 ? 0 : lo_c; hi_c = hi_c < 0 ? 0 : hi_c;
  lo_r = lo_r > w ? w : lo_r; hi_r = hi_r > w ? w : hi_r; lo_c = lo_c > h ? h : lo_c; hi_c = hi_c > h ? h : hi_c;
  for (int64_t r = 0; r < w; ++r) {
    if (!(r >= lo_r && r <= hi_r)) continue;
    const double px = (double)r;
    for (int64_t c = 0; c < h; ++c) {
      if (!(c >= lo_c && c <= hi_c)) continue;
      const double py = (double)c;
      int inside = 0;
      int64_t j = n - 1;
      for (int64_t i = 0; i < n; ++i) {
        const double xi = pts[i * ps[0]], yi = pts[i * ps[0] + ps[1]];
        const double xj = pts[j * ps[0]], yj = pts[j * ps[0] + ps[1]];
        if (((yi > py) != (yj > py)) && (px < (xj - xi) * (py - yi) / (yj - yi) + xi)) inside = !inside;
        j = i;
      }
      out[r * h + c] = (uint8_t)inside;
    }
  }
}
