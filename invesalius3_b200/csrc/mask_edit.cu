// The 3-D mask editor (invesalius/data/mask3d_editor_state.py): mask_cut (mask_cut.rs:7-62), the sphere
// brush (brush_mask.rs:5-71) and the even-odd screen-polygon rasteriser (polygon_mask.rs:4-79).
// Every decision is taken in the reference's float64 operation order: nalgebra's row sums left to
// right, true IEEE divisions and sqrt, no FMA (-fmad=false), Rust's saturating float -> integer casts
// and its wrapping integer arithmetic where the release crate wraps.
//
// mask_cut: 16 voxels per thread from one 128-bit load; chunks without a byte > 127 leave at once,
// FP64 runs for candidates only and only changed chunks are written back. Bound by FP64 issue (two
// 4x4 transforms, five divisions and a sqrt per candidate), not by the 1 B / voxel it reads.
// brush: one thread per voxel of the sphere's bounding box; launch / transfer bound.
// rasteriser: one thread per pixel, polygon vertices staged through shared memory in chunks.
#include <math.h>

#include "b2v_common.cuh"

namespace {

struct Mat4 { double m[16]; };

struct CutParams {
  Mat4 M, MV;
  double sx, sy, sz, max_depth;
  double wm1, hm1;        // (w - 1) as f64, (h - 1) as f64 with usize wrap-around
  long long dz, dy, dx, h, w;
  int edit_mode;
};

// true when the voxel (x, y, z) is to be set to 0 (it is known to be > 127)
__device__ __forceinline__ bool cut_voxel(const CutParams& P, const uint8_t* __restrict__ filter, long long x,
                                          long long y, long long z) {
  const double p0 = (double)x * P.sx, p1 = (double)y * P.sy, p2 = (double)z * P.sz;
  const double* M = P.M.m;
  const double q3 = ((M[12] * p0 + M[13] * p1) + M[14] * p2) + M[15] * 1.0;
  if (!(q3 > 0.0)) return false;
  const double q0 = (((M[0] * p0 + M[1] * p1) + M[2] * p2) + M[3] * 1.0) / q3;
  const double q1 = (((M[4] * p0 + M[5] * p1) + M[6] * p2) + M[7] * 1.0) / q3;
  const double* V = P.MV.m;
  const double c3 = ((V[12] * p0 + V[13] * p1) + V[14] * p2) + V[15] * 1.0;
  const double c0 = (((V[0] * p0 + V[1] * p1) + V[2] * p2) + V[3] * 1.0) / c3;
  const double c1 = (((V[4] * p0 + V[5] * p1) + V[6] * p2) + V[7] * 1.0) / c3;
  const double c2 = (((V[8] * p0 + V[9] * p1) + V[10] * p2) + V[11] * 1.0) / c3;
  const double dist = sqrt((c0 * c0 + c1 * c1) + c2 * c2);
  if (!(dist <= P.max_depth)) return false;
  const double px = (q0 / 2.0 + 0.5) * P.wm1;
  const double py = (q1 / 2.0 + 0.5) * P.hm1;
  if (px >= 0.0 && px < (double)P.w && py >= 0.0 && py < (double)P.h)
    return filter[(long long)py * P.w + (long long)px] != 0;
  return P.edit_mode == 0;
}

// 0x80-per-byte flags of a 16-byte chunk -> 16 bits (byte k -> bit k)
__device__ __forceinline__ uint32_t chunk_flags(const uint4& v) {
  return flags_to_nibble(v.x & 0x80808080u) | flags_to_nibble(v.y & 0x80808080u) << 4 |
         flags_to_nibble(v.z & 0x80808080u) << 8 | flags_to_nibble(v.w & 0x80808080u) << 12;
}
// 4 bits -> 0xff in every byte whose bit is set
__device__ __forceinline__ uint32_t nibble_to_bytes(uint32_t nib) { return ((nib * 0x00204081u) & 0x01010101u) * 0xffu; }

__global__ void __launch_bounds__(256) k_mask_cut(uint8_t* __restrict__ out, long long n, CutParams P,
                                                  const uint8_t* __restrict__ filter, int vec) {
  const long long nchunks = (n + 15) / 16;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < nchunks; c += stride) {
    const long long base = c * 16;
    const long long x0 = base % P.dx, r0 = base / P.dx, y0 = r0 % P.dy, z0 = r0 / P.dy;
    const bool full = vec && base + 16 <= n;     // else: unaligned buffer or the ragged tail
    uint4 v = make_uint4(0, 0, 0, 0);
    if (full) {
      v = *reinterpret_cast<const uint4*>(out + base);
    } else {
      uint32_t wd[4] = {0, 0, 0, 0};
#pragma unroll
      for (int k = 0; k < 16; ++k)
        if (base + k < n) wd[k / 4] |= (uint32_t)out[base + k] << (8 * (k % 4));
      v = make_uint4(wd[0], wd[1], wd[2], wd[3]);
    }
    uint32_t cand = chunk_flags(v), clr = 0;
    while (cand) {
      const int k = __ffs(cand) - 1;
      cand &= cand - 1;
      long long x = x0 + k, y = y0, z = z0;
      while (x >= P.dx) { x -= P.dx; if (++y == P.dy) { y = 0; ++z; } }
      if (cut_voxel(P, filter, x, y, z)) clr |= 1u << k;
    }
    if (!clr) continue;
    if (full) {
      v.x &= ~nibble_to_bytes(clr & 0xfu);
      v.y &= ~nibble_to_bytes((clr >> 4) & 0xfu);
      v.z &= ~nibble_to_bytes((clr >> 8) & 0xfu);
      v.w &= ~nibble_to_bytes((clr >> 12) & 0xfu);
      *reinterpret_cast<uint4*>(out + base) = v;
    } else {
      for (int k = 0; k < 16; ++k)
        if (clr >> k & 1u) out[base + k] = 0;
    }
  }
}

// ---- brush ------------------------------------------------------------------------------------
// Rust's `f as usize`: NaN and negatives -> 0, saturating at the top.
uint64_t sat_usize(double v) {
  if (!(v > 0.0)) return 0;
  if (v >= 18446744073709551616.0) return UINT64_MAX;
  return (uint64_t)v;
}

// [lo, hi] on one axis as brush_mask.rs:24-31 computes it (fmax / fmin ignore NaN like f64::max / min)
void brush_axis(double c, double r, double s, int64_t d, uint64_t* lo, uint64_t* hi) {
  *lo = sat_usize(fmax(floor((c - r) / s), 0.0));
  *hi = sat_usize(fmin(fmax(ceil((c + r) / s), 0.0), (double)(uint64_t)(d - 1)));
}

struct BrushParams {
  double sx, sy, sz, cx, cy, cz, r2;
  long long by, bx;                 // box row / plane extents of the dense buffers
  long long rz, ry, rx;             // where the launched region starts inside the box
  long long nz, ny, nx;             // launched region
  long long oz, oy, ox;             // the box's origin in the volume
  int edit_mode;
};

__global__ void __launch_bounds__(256) k_brush(uint8_t* __restrict__ out, const uint8_t* __restrict__ orig, BrushParams P) {
  const long long total = P.nz * P.ny * P.nx;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const long long lx = i % P.nx, r = i / P.nx, ly = r % P.ny, lz = r / P.ny;
    const long long bz = P.rz + lz, by = P.ry + ly, bx = P.rx + lx;
    const long long at = (bz * P.by + by) * P.bx + bx;
    const uint8_t val = out[at];
    if (P.edit_mode == 1 && val == 0) continue;
    const double dx = (double)(P.ox + bx) * P.sx - P.cx;
    const double dy = (double)(P.oy + by) * P.sy - P.cy;
    const double dz = (double)(P.oz + bz) * P.sz - P.cz;
    if (!((dx * dx + dy * dy) + dz * dz <= P.r2)) continue;
    if (P.edit_mode == 1) {
      out[at] = 0;
    } else if (orig) {
      const uint8_t o = orig[at];
      if (o > 0) out[at] = o;
    } else {
      out[at] = 255;
    }
  }
}

// ---- rasteriser -------------------------------------------------------------------------------
// Rust's `f as isize`: NaN -> 0, saturating at both ends.
__device__ __forceinline__ int64_t sat_isize(double v) {
  if (v != v) return 0;
  if (v >= 9223372036854775808.0) return INT64_MAX;
  if (v <= -9223372036854775808.0) return INT64_MIN;
  return (int64_t)v;
}
// polygon_mask.rs:26-34: (f as isize -/+ 1) wraps in the release crate, then .max(0) as usize, .min(n)
__device__ __forceinline__ int64_t idx_clamp(int64_t v, int64_t n) { return v < 0 ? 0 : (v > n ? n : v); }

constexpr int kPolyThreads = 256;
constexpr int kChunk = 1024;        // vertices staged per pass (16 KB of shared memory)

// one block per polygon: box[k] = (row_lo, row_hi, col_lo, col_hi), inclusive; empty when lo > hi
__global__ void __launch_bounds__(kPolyThreads) k_poly_bbox(const double* __restrict__ pts, const int64_t* __restrict__ offs,
                                                            int64_t w, int64_t h, int64_t* __restrict__ box) {
  __shared__ double s[4][kPolyThreads];
  const int64_t a = offs[blockIdx.x], b = offs[blockIdx.x + 1];
  // the min over the non-NaN values (or the start value) does not depend on the order
  double mnx = 1.7976931348623157e308, mxx = -1.7976931348623157e308, mny = mnx, mxy = mxx;
  for (int64_t i = a + threadIdx.x; i < b; i += blockDim.x) {
    const double px = pts[2 * i], py = pts[2 * i + 1];
    if (px < mnx) mnx = px;
    if (px > mxx) mxx = px;
    if (py < mny) mny = py;
    if (py > mxy) mxy = py;
  }
  s[0][threadIdx.x] = mnx; s[1][threadIdx.x] = mxx; s[2][threadIdx.x] = mny; s[3][threadIdx.x] = mxy;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const int t = threadIdx.x + o;
      if (s[0][t] < s[0][threadIdx.x]) s[0][threadIdx.x] = s[0][t];
      if (s[1][t] > s[1][threadIdx.x]) s[1][threadIdx.x] = s[1][t];
      if (s[2][t] < s[2][threadIdx.x]) s[2][threadIdx.x] = s[2][t];
      if (s[3][t] > s[3][threadIdx.x]) s[3][threadIdx.x] = s[3][t];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    int64_t* o = box + 4 * blockIdx.x;
    if (a == b) { o[0] = 1; o[1] = 0; o[2] = 1; o[3] = 0; return; }      // no points: all false
    o[0] = idx_clamp((int64_t)((uint64_t)sat_isize(floor(s[0][0])) - 1u), w);
    o[1] = idx_clamp((int64_t)((uint64_t)sat_isize(ceil(s[1][0])) + 1u), w);
    o[2] = idx_clamp((int64_t)((uint64_t)sat_isize(floor(s[2][0])) - 1u), h);
    o[3] = idx_clamp((int64_t)((uint64_t)sat_isize(ceil(s[3][0])) + 1u), h);
  }
}

// Pixel (r, c), r < w, c < h, is inside(px = r, py = c) OR-ed over the k polygons, negated on request.
// transpose == 0: out[r][c] (the (w, h) array of polygon2mask_rs); transpose != 0: out[c][r].
// threadIdx.x runs along the output's rows so the stores coalesce.
__global__ void __launch_bounds__(kPolyThreads) k_poly_raster(const double* __restrict__ pts, const int64_t* __restrict__ offs,
                                                              int64_t k, const int64_t* __restrict__ box, int64_t w, int64_t h,
                                                              int transpose, int negate, uint8_t* __restrict__ out) {
  __shared__ double2 sp[kChunk + 1];
  const int64_t fast = (int64_t)blockIdx.x * 32 + threadIdx.x % 32;
  const int64_t slow = (int64_t)blockIdx.y * (kPolyThreads / 32) + threadIdx.x / 32;
  const int64_t r = transpose ? fast : slow, c = transpose ? slow : fast;
  const bool live = r < w && c < h;
  const double px = (double)r, py = (double)c;
  bool any = false;
  for (int64_t p = 0; p < k; ++p) {
    const int64_t a = offs[p], n = offs[p + 1] - a;
    const bool in_box = live && r >= box[4 * p] && r <= box[4 * p + 1] && c >= box[4 * p + 2] && c <= box[4 * p + 3];
    if (!__syncthreads_or(in_box)) continue;
    bool inside = false;
    for (int64_t s0 = 0; s0 < n; s0 += kChunk) {
      const int m = n - s0 < kChunk ? (int)(n - s0) : kChunk;
      __syncthreads();
      for (int t = threadIdx.x; t <= m; t += blockDim.x) {
        const int64_t i = t == 0 ? (s0 == 0 ? n - 1 : s0 - 1) : s0 + t - 1;       // sp[0] = vertex j of edge s0
        sp[t] = make_double2(pts[2 * (a + i)], pts[2 * (a + i) + 1]);
      }
      __syncthreads();
      if (in_box) {
        for (int t = 1; t <= m; ++t) {
          const double xi = sp[t].x, yi = sp[t].y, xj = sp[t - 1].x, yj = sp[t - 1].y;
          if (((yi > py) != (yj > py)) && (px < (xj - xi) * (py - yi) / (yj - yi) + xi)) inside = !inside;
        }
      }
    }
    any = any || inside;
  }
  if (live) {
    const uint8_t v = (uint8_t)(any != (negate != 0));
    out[transpose ? c * w + r : r * h + c] = v;
  }
}

int launch_blocks(long long work) {
  long long blocks = ceil_div64(work, 256);
  const long long cap = (long long)b2v_sm_count() * 32;
  if (blocks > cap) blocks = cap;
  return blocks < 1 ? 1 : (int)blocks;
}

}  // namespace

extern "C" int b2v_mask_cut(uint8_t* out, int64_t dz, int64_t dy, int64_t dx, const double* spacing_host, double max_depth,
                            const uint8_t* filter, int64_t h, int64_t w, const double* m_host, const double* mv_host,
                            int edit_mode, void* stream) {
  B2V_REQUIRE(spacing_host && m_host && mv_host, B2V_ERR_ARG, "mask_cut: null host pointer");
  B2V_REQUIRE(dz >= 0 && dy >= 0 && dx >= 0 && h >= 0 && w >= 0, B2V_ERR_ARG, "mask_cut: bad shape");
  const long long n = dz * dy * dx;
  if (n == 0) return B2V_OK;
  B2V_REQUIRE(out && (filter || h * w == 0), B2V_ERR_ARG, "mask_cut: null device pointer");
  CutParams P;
  for (int k = 0; k < 16; ++k) { P.M.m[k] = m_host[k]; P.MV.m[k] = mv_host[k]; }
  P.sx = spacing_host[0]; P.sy = spacing_host[1]; P.sz = spacing_host[2];
  P.max_depth = max_depth;
  P.wm1 = (double)(uint64_t)(w - 1);
  P.hm1 = (double)(uint64_t)(h - 1);
  P.dz = dz; P.dy = dy; P.dx = dx; P.h = h; P.w = w;
  P.edit_mode = edit_mode;
  k_mask_cut<<<launch_blocks(ceil_div64(n, 16)), 256, 0, (cudaStream_t)stream>>>(out, n, P, filter, b2v_aligned16(out) ? 1 : 0);
  return b2v_check_launch("k_mask_cut");
}

extern "C" int b2v_brush_bbox(int64_t dz, int64_t dy, int64_t dx, const double* spacing_host, const double* center_host,
                              double radius, int64_t* box_host) {
  B2V_REQUIRE(spacing_host && center_host && box_host, B2V_ERR_ARG, "brush_bbox: null pointer");
  B2V_REQUIRE(dz >= 0 && dy >= 0 && dx >= 0, B2V_ERR_ARG, "brush_bbox: bad shape");
  const int64_t dims[3] = {dz, dy, dx};
  const double c[3] = {center_host[2], center_host[1], center_host[0]}, s[3] = {spacing_host[2], spacing_host[1], spacing_host[0]};
  bool empty = dz == 0 || dy == 0 || dx == 0;
  uint64_t lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
  for (int a = 0; a < 3 && !empty; ++a) {
    brush_axis(c[a], radius, s[a], dims[a], &lo[a], &hi[a]);
    empty = lo[a] > hi[a];
  }
  for (int a = 0; a < 3; ++a) {
    box_host[a] = empty ? 0 : (int64_t)lo[a];
    box_host[3 + a] = empty ? 0 : (int64_t)(hi[a] - lo[a] + 1);
  }
  return B2V_OK;
}

extern "C" int b2v_brush_mask(uint8_t* out, const uint8_t* orig, int64_t bz, int64_t by, int64_t bx, int64_t oz, int64_t oy,
                              int64_t ox, int64_t dz, int64_t dy, int64_t dx, const double* spacing_host,
                              const double* center_host, double radius, int edit_mode, void* stream) {
  B2V_REQUIRE(bz >= 0 && by >= 0 && bx >= 0 && oz >= 0 && oy >= 0 && ox >= 0 && oz + bz <= dz && oy + by <= dy &&
                  ox + bx <= dx,
              B2V_ERR_ARG, "brush_mask: the box does not lie inside the volume");
  int64_t bb[6];
  const int rc = b2v_brush_bbox(dz, dy, dx, spacing_host, center_host, radius, bb);
  if (rc) return rc;
  if (edit_mode != 0 && edit_mode != 1) return B2V_OK;
  BrushParams P;
  const int64_t o[3] = {oz, oy, ox}, b[3] = {bz, by, bx};
  int64_t rs[3], ns[3];
  for (int a = 0; a < 3; ++a) {                  // the sphere's box intersected with the box held
    const int64_t lo = bb[a] > o[a] ? bb[a] : o[a];
    const int64_t hi = bb[a] + bb[3 + a] < o[a] + b[a] ? bb[a] + bb[3 + a] : o[a] + b[a];
    rs[a] = lo - o[a];
    ns[a] = hi > lo ? hi - lo : 0;
  }
  const long long total = (long long)ns[0] * ns[1] * ns[2];
  if (total == 0) return B2V_OK;
  B2V_REQUIRE(out, B2V_ERR_ARG, "brush_mask: null device pointer");
  P.sx = spacing_host[0]; P.sy = spacing_host[1]; P.sz = spacing_host[2];
  P.cx = center_host[0]; P.cy = center_host[1]; P.cz = center_host[2];
  P.r2 = radius * radius;
  P.by = by; P.bx = bx;
  P.rz = rs[0]; P.ry = rs[1]; P.rx = rs[2];
  P.nz = ns[0]; P.ny = ns[1]; P.nx = ns[2];
  P.oz = oz; P.oy = oy; P.ox = ox;
  P.edit_mode = edit_mode;
  k_brush<<<launch_blocks(total), 256, 0, (cudaStream_t)stream>>>(out, orig, P);
  return b2v_check_launch("k_brush");
}

extern "C" int64_t b2v_polygons_workspace_bytes(int64_t k) { return k > 0 ? 4 * k * (int64_t)sizeof(int64_t) : 0; }

extern "C" int b2v_polygons_raster(const double* points, const int64_t* offsets, int64_t k, int64_t w, int64_t h,
                                   int transpose, int negate, uint8_t* out, void* workspace, void* stream) {
  B2V_REQUIRE(k >= 1 && k <= 65535, B2V_ERR_ARG, "polygons_raster: between 1 and 65535 polygons");
  B2V_REQUIRE(w >= 0 && h >= 0, B2V_ERR_ARG, "polygons_raster: bad shape");
  if (w == 0 || h == 0) return B2V_OK;
  B2V_REQUIRE(offsets && out && workspace, B2V_ERR_ARG, "polygons_raster: null device pointer");
  const int64_t fast = transpose ? w : h, slow = transpose ? h : w;
  const int64_t gx = ceil_div64(fast, 32), gy = ceil_div64(slow, kPolyThreads / 32);
  B2V_REQUIRE(gx < (1ll << 31) && gy < 65536, B2V_ERR_ARG, "polygons_raster: screen too large");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t* box = (int64_t*)workspace;
  k_poly_bbox<<<(unsigned)k, kPolyThreads, 0, s>>>(points, offsets, w, h, box);
  int rc = b2v_check_launch("k_poly_bbox");
  if (rc) return rc;
  k_poly_raster<<<dim3((unsigned)gx, (unsigned)gy), kPolyThreads, 0, s>>>(points, offsets, k, box, w, h, transpose, negate, out);
  return b2v_check_launch("k_poly_raster");
}
