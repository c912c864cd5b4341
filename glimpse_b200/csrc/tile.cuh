// Per-(point, observer) tile pipeline, executed by one CTA out of shared memory:
//   raw window -> histogram -> CDF-matching look-up table -> 5x5 median high-pass -> SSD surface
//   -> bicubic not-a-knot spline in Hermite form.
// Reference: Tracker.extract_tile (track/tracker.py:494-534), helpers.normalize / compute_cdf /
// match_cdf (helpers.py:324-344, 433-493), scipy.ndimage.median_filter(size=5x5, mode='reflect'),
// cv2.matchTemplate(TM_SQDIFF) / (w h) (tracker.py:609-614), RectBivariateSpline(kx=ky=3, s=0)
// (track/observer.py:178-214).
//
// Two identities keep the work integer-valued until the last moment (frames are uint8 band sums):
//  * CDF matching only depends on pixel ranks, so the matched tile is LUT[raw] with one LUT entry
//    per grey level: LUT[g] = interp(count(raw <= g) / size, template_quantiles, template_values).
//  * LUT is non-decreasing and the median of 25 values is one of them, so
//    median5x5(LUT[raw]) == LUT[median5x5(raw)]; the median runs on integers, two vertically
//    adjacent pixels at a time in the halves of one 32-bit word (VIMNMX.U16x2).
#pragma once
#include "common.cuh"
#include "median25.cuh"

namespace gb {

// Thomas-algorithm factors of the not-a-knot slope system (rows [1 2], [1 4 1]..., [2 1]); they
// depend only on the row index, not on the system size.  Filled once per device by the host.
#define GB_MAX_SURFACE 1024 /* cells per axis of an SSE surface (the factors below converge after ~30 rows) */
__constant__ double c_spline_cp[GB_MAX_SURFACE];
__constant__ double c_spline_inv[GB_MAX_SURFACE];

struct TileWork {
  float4* herm;      // [Mv][Mp] (F, dF/du, dF/dv, d2F/dudv); Mp odd keeps row solves off the same banks
  uint32_t* packed;  // [Sv + 4][Su + 4] reflect-padded window, row r in the low and r + 1 in the high half; aliases herm
  double* lut;       // [nbins]
  double* tq;        // [nvals] template quantiles
  double* tv;        // [nvals] template values
  float* hp;         // [Sv][Sp] high-passed search tile, Sp = Su rounded up to 4
  uint16_t* raw;     // [Sv][Su] raw window; aliases hp (dead before hp is written)
  float2* tmpl;      // [th][tw] high-passed template, negated and duplicated (-t, -t): the packed FP32 SSD adds it to two pixels
  float* tcol = nullptr;  // templates above GB_SMEM_TEMPLATE pixels instead: [tw][th] negated, column by column, in the window's
                          // global region (tmpl unused; tq / tv point at the template's global tables)
  uint32_t* hist;    // [nbins]
  int Su, Sv, Mu, Mv, Mp, Sp, Tp, nbins, nvals, tw, th;
  int dtype = 0;               // GB_PIX_* of the frame: other than uint8, the window goes through `vals` and becomes ranks
  double* vals = nullptr;      // [Sv][Su] grey values of the window (global work area behind the tile's data), frames other than uint8
  const void* tmap = nullptr;  // CUtensorMap of the frame (global memory), or null: the window is read with ordinary loads
  uint64_t* bar = nullptr;     // mbarrier of the CTA for the TMA loads (phase 0)
  int mh = 5, mw = 5;  // rows x columns of the median high-pass (Tracker.highpass['size'])
  int hp_mode = 0, hp_org_r = 0, hp_org_c = 0;  // its border mode (GB_HP_*) and origin (Tracker.highpass['mode'], ['origin'])
  double hp_cval = 0.0;                          // ... and the constant beyond the border for GB_HP_CONSTANT
  const uint32_t* hp_fp = nullptr;               // ... and the footprint (one word per window row), or null: the full window
  bool cub_u = true, cub_v = true;  // cubic (default) or piecewise-linear interpolation along the columns / rows (Tracker.interpolation)
  int ku = 3, kv = 3;               // the degrees themselves; other than 1 / 3: B-spline coefficients instead of Hermite data
  double* band = nullptr;           // ... and the work area of their collocation solves (global memory)
};

__host__ __device__ inline int64_t align16(int64_t b) { return (b + 15) / 16 * 16; }

// Bytes of the template copy and its CDF tables next to the window: none for templates above GB_SMEM_TEMPLATE pixels, which
// the SSD reads from global memory (a 128 x 128 template alone would take 128 KB of the window's shared memory).
__host__ __device__ inline int64_t tile_template_bytes(int tw, int th, int nvals) {
  if ((int64_t)tw * th > GB_SMEM_TEMPLATE) return 0;
  return align16((int64_t)nvals * 8) * 2 + align16((int64_t)th * tw * 8);
}

__host__ __device__ inline int64_t tile_bytes_needed(int Su, int Sv, int tw, int th, int nbins, int nvals) {
  const int64_t Mu = Su - tw + 1, Mv = Sv - th + 1, Mp = Mu | 1, Sp = (Su + 3) / 4 * 4;
  const int64_t herm = Mv * Mp * 16, packed = (int64_t)(Sv + 4) * (Su + 4) * 4;
  int64_t b = align16(herm > packed ? herm : packed);
  b += align16((int64_t)nbins * 8) + tile_template_bytes(tw, th, nvals);
  b += align16((int64_t)Sv * Sp * 4);
  b += align16((int64_t)nbins * 4);
  return b;
}

__device__ inline void tile_carve(char* base, TileWork& w) {
  w.Mp = w.Mu | 1;
  w.Sp = (w.Su + 3) / 4 * 4;
  w.Tp = (w.tw + 3) / 4 * 4;
  char* p = base;
  const int64_t herm = (int64_t)w.Mv * w.Mp * 16, packed = (int64_t)(w.Sv + 4) * (w.Su + 4) * 4;
  w.herm = reinterpret_cast<float4*>(p);
  w.packed = reinterpret_cast<uint32_t*>(p);
  p += align16(herm > packed ? herm : packed);
  w.lut = reinterpret_cast<double*>(p);
  p += align16((int64_t)w.nbins * 8);
  if (!w.tcol) {
    w.tq = reinterpret_cast<double*>(p);
    p += align16((int64_t)w.nvals * 8);
    w.tv = reinterpret_cast<double*>(p);
    p += align16((int64_t)w.nvals * 8);
  }
  w.hp = reinterpret_cast<float*>(p);
  w.raw = reinterpret_cast<uint16_t*>(p);
  p += align16((int64_t)w.Sv * w.Sp * 4);
  if (!w.tcol) {
    w.tmpl = reinterpret_cast<float2*>(p);
    p += align16((int64_t)w.th * w.tw * 8);
  }
  w.hist = reinterpret_cast<uint32_t*>(p);
}

// Large templates: the negated high-passed template, column by column, into the window's global region (tile_prepare, all
// threads; the SSD reads it after the CTA's next barrier).
__device__ __forceinline__ void tile_template_global(const TileWork& w, const double* __restrict__ g_tmpl) {
  const int ta = w.tw * w.th;
  for (int k = threadIdx.x; k < ta; k += blockDim.x) {
    const int c = k / w.th, r = k - c * w.th;
    w.tcol[k] = -(float)g_tmpl[r * w.tw + c];
  }
}

// np.interp(q, xp, fp) for one abscissa (numpy compiled_base.c arr_interp): clamped at the ends,
// exact hit returns fp[j], otherwise slope * (q - xp[j]) + fp[j] unfused.
__device__ inline double interp_clamped(double q, const double* xp, const double* fp, int n) {
  if (q > xp[n - 1]) return fp[n - 1];
  if (q < xp[0]) return fp[0];
  int lo = 0, hi = n;  // largest j with xp[j] <= q
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (xp[mid] <= q) lo = mid; else hi = mid;
  }
  const int j = lo;
  if (j == n - 1 || xp[j] == q) return fp[j];
  const double slope = quo(sub(fp[j + 1], fp[j]), sub(xp[j + 1], xp[j]));
  return add(mul(slope, sub(q, xp[j])), fp[j]);
}

__device__ __forceinline__ int reflect_index(int i, int n) {
  // scipy.ndimage 'reflect': d c b a | a b c d | d c b a
  if (i < 0) i = -i - 1;
  if (i >= n) i = 2 * n - i - 1;
  return min(max(i, 0), n - 1);
}

// Median of the 5x5 neighbourhood of (r, c) in an integer tile with reflected borders (scalar
// version, used by the template kernel).
__device__ __forceinline__ int median5x5(const uint16_t* raw, int Su, int Sv, int r, int c) {
  int v[25];
  int cols[5];
#pragma unroll
  for (int j = 0; j < 5; ++j) cols[j] = reflect_index(c + j - 2, Su);
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const uint16_t* row = raw + reflect_index(r + i - 2, Sv) * Su;
#pragma unroll
    for (int j = 0; j < 5; ++j) v[i * 5 + j] = row[cols[j]];
  }
  return gb_median25(v);
}

// scipy.ndimage 'reflect' for an offset of any length (the pattern has period 2 n).
__device__ __forceinline__ int reflect_index_any(int i, int n) {
  while (i < 0 || i >= n) i = i < 0 ? -i - 1 : 2 * n - i - 1;
  return i;
}

// Median of an mh x mw neighbourhood with reflected borders, any size: scipy.ndimage.median_filter(size=(mh, mw))
// places the window at offsets -(m / 2) .. m - 1 - m / 2 along each axis and returns the element of rank
// (mh * mw) / 2.  Grey levels are integers below 1024 (band sums of uint8), so the element is found bit by bit:
// it is >= L exactly when at most `rank` neighbours are < L.  (The 5x5 default never comes here.)
// `nlevels` = number of grey levels (sets the first bit tried).
__device__ __forceinline__ int top_bit_below(int n) {
  int top = 1;
  while (2 * top < n) top *= 2;
  return top;
}
__device__ inline int median_window(const uint16_t* raw, int Su, int Sv, int r, int c, int mh, int mw, int nlevels = 1024) {
  const int rank = (mh * mw) >> 1, r0 = r - (mh >> 1), c0 = c - (mw >> 1);
  const bool inside = r0 >= 0 && r0 + mh <= Sv && c0 >= 0 && c0 + mw <= Su;
  int level = 0;
  for (int bit = top_bit_below(nlevels); bit; bit >>= 1) {
    const int cand = level | bit;
    int below = 0;
    if (inside) {
      for (int a = 0; a < mh; ++a) {
        const uint16_t* row = raw + (r0 + a) * Su + c0;
        for (int b = 0; b < mw; ++b) below += (int)row[b] < cand;
      }
    } else {
      for (int a = 0; a < mh; ++a) {
        const uint16_t* row = raw + reflect_index_any(r0 + a, Sv) * Su;
        for (int b = 0; b < mw; ++b) below += (int)row[reflect_index_any(c0 + b, Su)] < cand;
      }
    }
    if (below <= rank) level = cand;
  }
  return level;
}

// Border handling of scipy.ndimage filters for an index beyond [0, n): the index it maps to, or -1 for 'constant'.
__device__ __forceinline__ int border_index(int i, int n, int mode) {
  if (i >= 0 && i < n) return i;
  switch (mode) {
    case GB_HP_CONSTANT: return -1;
    case GB_HP_NEAREST: return i < 0 ? 0 : n - 1;
    case GB_HP_MIRROR: {  // d c b | a b c d | c b a: period 2 n - 2
      if (n == 1) return 0;
      const int period = 2 * n - 2;
      i = i % period;
      if (i < 0) i += period;
      return i < n ? i : period - i;
    }
    case GB_HP_WRAP: {
      i = i % n;
      return i < 0 ? i + n : i;
    }
    default: return reflect_index_any(i, n);
  }
}

// The general median high-pass (Tracker.highpass with `mode`, `cval`, `origin`): rank (mh mw) / 2 of the window that starts at
// (r - mh / 2 - origin_r, c - mw / 2 - origin_c), borders by `mode`.  Works on CODES: a pixel of grey level g has code 2 g + 1,
// the constant beyond the border has the even code `cval_code` = 2 x (number of grey levels whose filtered-tile value is below
// cval) — the codes are ordered like the values, so the rank element is found on integers (bit by bit, as median_window does).
// Returns the code of the median: odd = grey level (code - 1) / 2, even = the border constant.
// `fp` = the footprint, one word per window row (bit b = column b takes part), or null for the full window.
__device__ inline int median_window_codes(const uint16_t* raw, int Su, int Sv, int r, int c, int mh, int mw, int mode, int org_r, int org_c,
                                          int cval_code, const uint32_t* fp = nullptr, int nlevels = 1024) {
  int count = mh * mw;
  if (fp) {
    count = 0;
    for (int a = 0; a < mh; ++a) count += __popc(fp[a]);
  }
  const int rank = count >> 1, r0 = r - (mh >> 1) - org_r, c0 = c - (mw >> 1) - org_c;
  int level = 0;
  for (int bit = top_bit_below(2 * nlevels + 2); bit; bit >>= 1) {
    const int cand = level | bit;
    int below = 0;
    for (int a = 0; a < mh; ++a) {
      const int rr = border_index(r0 + a, Sv, mode);
      for (int b = 0; b < mw; ++b) {
        if (fp && !(fp[a] >> b & 1u)) continue;
        const int cc = border_index(c0 + b, Su, mode);
        const int code = (rr < 0 || cc < 0) ? cval_code : 2 * (int)raw[rr * Su + cc] + 1;
        below += code < cand;
      }
    }
    if (below <= rank) level = cand;
  }
  return level;
}

// Solve the not-a-knot slope system along one line of the Hermite array (stride in floats).
// `in` holds the samples, `out` receives the slopes; the forward-sweep values pass through `out`
// as floats.  The loop-carried chain is one DFMA per element in each direction.
// `cubic` = false (degree-1 interpolation along this axis, Tracker.interpolation): the slopes are never used by the
// evaluation; zeros keep the unused Hermite terms finite (the line may then be shorter than the four samples a cubic needs).
__device__ __forceinline__ void spline_slopes_line(const float* __restrict__ in, float* __restrict__ out, int stride, int m, bool cubic = true) {
  if (!cubic) {
    for (int i = 0; i < m; ++i) out[i * stride] = 0.0f;
    return;
  }
  const double f0 = in[0], f1 = in[stride], f2 = in[2 * stride];
  double d = 0.5 * (5.0 * (f1 - f0) + (f2 - f1));
  out[0] = (float)d;
  double prev = f0, cur = f1;
  int i = 1;
  for (; i + 3 < m - 1; i += 4) {  // four elements per trip: loads and rhs products are off the chain
    const double n0 = in[(i + 1) * stride], n1 = in[(i + 2) * stride], n2 = in[(i + 3) * stride], n3 = in[(i + 4) * stride];
    const double v0 = c_spline_inv[i], v1 = c_spline_inv[i + 1], v2 = c_spline_inv[i + 2], v3 = c_spline_inv[i + 3];
    const double a0 = 3.0 * (n0 - prev) * v0, a1 = 3.0 * (n1 - cur) * v1, a2 = 3.0 * (n2 - n0) * v2, a3 = 3.0 * (n3 - n1) * v3;
    const double d0 = fma(-v0, d, a0);
    const double d1 = fma(-v1, d0, a1);
    const double d2 = fma(-v2, d1, a2);
    d = fma(-v3, d2, a3);
    out[i * stride] = (float)d0;
    out[(i + 1) * stride] = (float)d1;
    out[(i + 2) * stride] = (float)d2;
    out[(i + 3) * stride] = (float)d;
    prev = n2;
    cur = n3;
  }
  for (; i < m - 1; ++i) {
    const double next = in[(i + 1) * stride];
    const double v = c_spline_inv[i];
    d = fma(-v, d, 3.0 * (next - prev) * v);
    out[i * stride] = (float)d;
    prev = cur;
    cur = next;
  }
  {
    const double fa = in[(m - 3) * stride], fb = in[(m - 2) * stride], fc = in[(m - 1) * stride];
    const double rhs = 0.5 * (5.0 * (fc - fb) + (fb - fa));
    d = (rhs - 2.0 * d) / (1.0 - 2.0 * c_spline_cp[m - 2]);
  }
  double s = d;
  out[(m - 1) * stride] = (float)s;
  i = m - 2;
  for (; i - 3 >= 0; i -= 4) {
    const double e0 = out[i * stride], e1 = out[(i - 1) * stride], e2 = out[(i - 2) * stride], e3 = out[(i - 3) * stride];
    const double s0 = fma(-c_spline_cp[i], s, e0);
    const double s1 = fma(-c_spline_cp[i - 1], s0, e1);
    const double s2 = fma(-c_spline_cp[i - 2], s1, e2);
    s = fma(-c_spline_cp[i - 3], s2, e3);
    out[i * stride] = (float)s0;
    out[(i - 1) * stride] = (float)s1;
    out[(i - 2) * stride] = (float)s2;
    out[(i - 3) * stride] = (float)s;
  }
  for (; i >= 0; --i) {
    s = fma(-c_spline_cp[i], s, (double)out[i * stride]);
    out[i * stride] = (float)s;
  }
}

// Bicubic Hermite evaluation at (x, y) measured from the first cell centre, in cell units.  The cell
// index and the in-cell offset are taken in double; the 16-term patch is evaluated in float (the
// data are float32: the SSE surface is cv2.matchTemplate's float32 output in the reference).
// `lin_u` / `lin_v`: degree-1 interpolation along that axis (Tracker.interpolation ky / kx = 1): the value weights become
// (1 - t, t) and the slope weights vanish — FITPACK's interpolating linear spline has a knot at every data site.
__device__ __forceinline__ float hermite_eval(const float4* __restrict__ herm, int Mp, int Mu, int Mv, double x, double y, bool lin_u = false,
                                              bool lin_v = false) {
  int j = min((int)x, Mu - 2), i = min((int)y, Mv - 2);  // x, y >= 0
  j = max(j, 0);
  i = max(i, 0);
  const float tx = (float)(x - (double)j), ty = (float)(y - (double)i);
  const float tx2 = tx * tx, tx3 = tx2 * tx, ty2 = ty * ty, ty3 = ty2 * ty;
  const float a2 = lin_u ? tx : 3.0f * tx2 - 2.0f * tx3, a0 = 1.0f - a2, a3 = lin_u ? 0.0f : tx3 - tx2, a1 = lin_u ? 0.0f : a3 - tx2 + tx;
  const float b2 = lin_v ? ty : 3.0f * ty2 - 2.0f * ty3, b0 = 1.0f - b2, b3 = lin_v ? 0.0f : ty3 - ty2, b1 = lin_v ? 0.0f : b3 - ty2 + ty;
  const float4* row0 = herm + i * Mp + j;
  const float4 h00 = row0[0], h01 = row0[1], h10 = row0[Mp], h11 = row0[Mp + 1];
  // rows of the patch: value and u-slope interpolated along u, for f and for df/dv
  const float top_f = a0 * h00.x + a2 * h01.x + a1 * h00.y + a3 * h01.y;
  const float bot_f = a0 * h10.x + a2 * h11.x + a1 * h10.y + a3 * h11.y;
  const float top_v = a0 * h00.z + a2 * h01.z + a1 * h00.w + a3 * h01.w;
  const float bot_v = a0 * h10.z + a2 * h11.z + a1 * h10.w + a3 * h11.w;
  return b0 * top_f + b2 * bot_f + b1 * top_v + b3 * bot_v;
}

// ---------------------------------------------------------------------------------------------
// Interpolating splines of degree 2, 4 and 5 (Tracker.interpolation; RectBivariateSpline(kx, ky, s = 0) = FITPACK regrid).
// The data sites are the cell centres 0 .. m - 1 (unit spacing), so FITPACK's knots (fpregr.f, interpolation case) are known
// in closed form: k + 1 copies of 0 and of m - 1 at the ends and m - k - 1 interior knots — the sites (k + 1) / 2 ..
// m - 1 - (k + 1) / 2 for an odd degree, the midpoints k / 2 + 1 / 2 .. m - 1 - k / 2 - 1 / 2 for an even one.  The surface
// is kept as tensor-product B-spline coefficients (one float per cell, in the x component of the Hermite array): they solve
// the two banded collocation systems, and a sample is a (kx + 1) x (ky + 1) sum over de Boor's basis values (fpbspl.f).
// Any degree 1 .. 5 per axis can take this path; degrees 1 and 3 on both axes keep the cheaper Hermite form.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double bspline_knot(int i, int m, int k) {
  if (i <= k) return 0.0;
  if (i >= m) return (double)(m - 1);
  const int q = i - k - 1;
  return (k & 1) ? (double)((k + 1) / 2 + q) : (double)(k / 2 + q) + 0.5;
}
// knot interval l (k <= l <= m - 1) with t[l] <= x < t[l + 1] for x in [0, m - 1] (the last interval is closed, fpbisp.f)
__device__ __forceinline__ int bspline_span(double x, int m, int k) {
  const double first = (k & 1) ? (double)((k + 1) / 2) : (double)(k / 2) + 0.5;
  const int cnt = (int)floor(x - first) + 1;  // interior knots <= x
  return k + max(0, min(cnt, m - k - 1));
}
// the k + 1 B-splines that do not vanish on interval l, at x (fpbspl.f)
__device__ __forceinline__ void bspline_basis(double x, int l, int m, int k, double (&h)[6]) {
  double hh[5];
  h[0] = 1.0;
  for (int j = 1; j <= k; ++j) {
    for (int i = 0; i < j; ++i) hh[i] = h[i];
    h[0] = 0.0;
    for (int i = 0; i < j; ++i) {
      const int li = l + 1 + i, lj = li - j;
      const double tli = bspline_knot(li, m, k), tlj = bspline_knot(lj, m, k);
      const double f = hh[i] / (tli - tlj);
      h[i] += f * (tli - x);
      h[i + 1] = f * (x - tlj);
    }
  }
}
// LU factors (no pivoting: B-spline collocation matrices are totally positive) of the m x m collocation matrix
// A[i][j] = B_j(site i) in band storage ab[i][j - i + k], |j - i| <= k.  One thread.
__device__ inline void bspline_factor(double* ab, int m, int k) {
  const int W = 2 * k + 1;
  for (int i = 0; i < m * W; ++i) ab[i] = 0.0;
  for (int i = 0; i < m; ++i) {
    const int l = bspline_span((double)i, m, k);
    double h[6];
    bspline_basis((double)i, l, m, k, h);
    for (int a = 0; a <= k; ++a) {
      const int j = l - k + a;
      if (j - i >= -k && j - i <= k) ab[i * W + (j - i + k)] = h[a];
    }
  }
  for (int c = 0; c < m; ++c) {
    const double piv = ab[c * W + k];
    const int last = min(m - 1, c + k);
    for (int r = c + 1; r <= last; ++r) {
      const double f = ab[r * W + (c - r + k)] / piv;
      ab[r * W + (c - r + k)] = f;
      for (int j = c + 1; j <= last; ++j) ab[r * W + (j - r + k)] -= f * ab[c * W + (j - c + k)];
    }
  }
}
// Solve A x = b in place along one line of floats (stride in floats) with the factors above.
__device__ inline void bspline_solve_line(const double* __restrict__ ab, int m, int k, float* line, int stride) {
  const int W = 2 * k + 1;
  for (int r = 0; r < m; ++r) {  // L y = b (unit diagonal)
    double y = (double)line[r * stride];
    for (int c = max(0, r - k); c < r; ++c) y -= ab[r * W + (c - r + k)] * (double)line[c * stride];
    line[r * stride] = (float)y;
  }
  for (int r = m - 1; r >= 0; --r) {  // U x = y
    double x = (double)line[r * stride];
    const int last = min(m - 1, r + k);
    for (int c = r + 1; c <= last; ++c) x -= ab[r * W + (c - r + k)] * (double)line[c * stride];
    line[r * stride] = (float)(x / ab[r * W + k]);
  }
}
// Sample of the coefficient surface at (x, y) from the first cell centre in cell units (fpbisp.f): arguments clamped to the
// data sites.  ku / kv = degree along the columns / rows.
__device__ __noinline__ float bspline_eval(const float4* __restrict__ coef, int Mp, int Mu, int Mv, double x, double y, int ku, int kv) {
  x = fmin(fmax(x, 0.0), (double)(Mu - 1));
  y = fmin(fmax(y, 0.0), (double)(Mv - 1));
  const int lu = bspline_span(x, Mu, ku), lv = bspline_span(y, Mv, kv);
  double hu[6], hv[6];
  bspline_basis(x, lu, Mu, ku, hu);
  bspline_basis(y, lv, Mv, kv, hv);
  double acc = 0.0;
  for (int a = 0; a <= kv; ++a) {
    const float4* row = coef + (lv - kv + a) * Mp + (lu - ku);
    double r = 0.0;
    for (int b = 0; b <= ku; ++b) r = fma(hu[b], (double)row[b].x, r);
    acc = fma(hv[a], r, acc);
  }
  return (float)acc;
}
__host__ __device__ inline bool spline_is_hermite(int ku, int kv) { return (ku == 1 || ku == 3) && (kv == 1 || kv == 3); }
__host__ __device__ inline int64_t bspline_band_bytes(int Mu, int Mv, int ku, int kv) {
  return ((int64_t)Mu * (2 * ku + 1) + (int64_t)Mv * (2 * kv + 1)) * 8;
}

// Phases 1-5 of the surface of one search window: raw window -> high-passed, CDF-matched float tile `w.hp`
// (plus the template in `w.tmpl`).  All threads of the CTA participate.  `box` = (left, top, right, bottom);
// template data in global memory.  The caller has verified the capacity and carved `w`.
// Grey value of pixel (row, col) of a frame of any supported type, as the reference sees it after to_gray (tracker.py:522-524):
// the pixel itself for one band, else tile.mean(axis=2) — NumPy sums the few bands in order, in float64 for integer types and in
// float32 for float32 frames, and divides by their number.
__device__ __forceinline__ double pixel_gray(const uint8_t* pixels, int64_t pitch, int nchan, int dtype, int row, int col) {
  const uint8_t* base = pixels + (int64_t)row * pitch;
  switch (dtype) {
    case GB_PIX_U16: {
      const uint16_t* q = reinterpret_cast<const uint16_t*>(base) + (int64_t)col * nchan;
      double sum = (double)q[0];
      for (int ch = 1; ch < nchan; ++ch) sum += (double)q[ch];
      return nchan > 1 ? quo(sum, (double)nchan) : sum;
    }
    case GB_PIX_F32: {
      const float* q = reinterpret_cast<const float*>(base) + (int64_t)col * nchan;
      float sum = q[0];
      for (int ch = 1; ch < nchan; ++ch) sum = __fadd_rn(sum, q[ch]);
      return nchan > 1 ? (double)__fdiv_rn(sum, (float)nchan) : (double)sum;
    }
    case GB_PIX_F64: {
      const double* q = reinterpret_cast<const double*>(base) + (int64_t)col * nchan;
      double sum = q[0];
      for (int ch = 1; ch < nchan; ++ch) sum = add(sum, q[ch]);
      return nchan > 1 ? quo(sum, (double)nchan) : sum;
    }
    default: {
      const uint8_t* q = base + (int64_t)col * nchan;
      double sum = (double)q[0];
      for (int ch = 1; ch < nchan; ++ch) sum += (double)q[ch];
      return nchan > 1 ? quo(sum, (double)nchan) : sum;
    }
  }
}

// Frames are read through the TMA engine when the frame has a tensor map (`w.tmap`, built by the host for frames whose
// pitch and base are 16-byte aligned): the window arrives as boxes of GB_TMA_BOXW bytes x GB_TMA_BOXH rows, staged where the
// padded window copy (`w.packed`) is built afterwards.
#define GB_TMA_BOXW 32
#define GB_TMA_BOXH 8
__device__ __forceinline__ bool tile_window_by_tma(const TileWork& w, int nchan) {
  if (!w.tmap || !w.bar) return false;
  const int nbx = (w.Su * nchan + GB_TMA_BOXW - 1) / GB_TMA_BOXW, nby = (w.Sv + GB_TMA_BOXH - 1) / GB_TMA_BOXH;
  return (int64_t)nbx * nby * (GB_TMA_BOXW * GB_TMA_BOXH) <= (int64_t)(w.Sv + 4) * (w.Su + 4) * 4 && (smem_u32(w.packed) & 127u) == 0u &&
         __isShared(w.packed);
}

__device__ inline void tile_prepare(const uint8_t* __restrict__ pixels, int pitch, int nchan, const int* box, const double* __restrict__ g_tmpl,
                                    const double* __restrict__ g_tq, const double* __restrict__ g_tv, TileWork& w,
                                    float* dump_search, int64_t dump_cap, long long* clk) {
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int Su = w.Su, Sv = w.Sv, Sp = w.Sp;
  const int area = Su * Sv;
  const bool by_tma = w.dtype == GB_PIX_U8 && tile_window_by_tma(w, nchan);
  const bool ranked = w.dtype != GB_PIX_U8;
  if (ranked) {
    // 1. (frames other than uint8) grey values of the window, then every pixel becomes the number of window pixels below it:
    //    equal values get equal levels and the order is kept, which is all CDF matching and the median need (nbins = Su Sv)
    const int ta = w.tw * w.th;
    for (int e = tid; e < area; e += nthr) {
      const int r = e / Su, c = e - r * Su;
      w.vals[e] = pixel_gray(pixels, pitch, nchan, w.dtype, box[1] + r, box[0] + c);
    }
    for (int i = tid; i < w.nbins; i += nthr) w.hist[i] = 0u;
    if (w.tcol) {
      tile_template_global(w, g_tmpl);
    } else {
      for (int i = tid; i < ta; i += nthr) {
        const float tv = -(float)g_tmpl[i];
        w.tmpl[i] = make_float2(tv, tv);
      }
      for (int i = tid; i < w.nvals; i += nthr) {
        w.tq[i] = g_tq[i];
        w.tv[i] = g_tv[i];
      }
    }
    __syncthreads();
    for (int e = tid; e < area; e += nthr) {
      const double v = w.vals[e];
      int below = 0;
      for (int j = 0; j < area; ++j) below += w.vals[j] < v;
      w.raw[e] = (uint16_t)below;
      atomicAdd(&w.hist[below], 1u);
    }
  } else if (by_tma) {
    // 1. (TMA) one thread asks for every box of the window; everybody fills the tables meanwhile, then turns the staged
    //    bytes into band sums and counts them (the histogram pass of phase 2 is folded into this one)
    const int nbx = (Su * nchan + GB_TMA_BOXW - 1) / GB_TMA_BOXW, nby = (Sv + GB_TMA_BOXH - 1) / GB_TMA_BOXH;
    uint8_t* stage = reinterpret_cast<uint8_t*>(w.packed);
    if (tid == 0) {
      mbar_expect_tx(w.bar, (uint32_t)(nbx * nby * GB_TMA_BOXW * GB_TMA_BOXH));
      for (int by = 0; by < nby; ++by)
        for (int bx = 0; bx < nbx; ++bx)
          tma_load_2d(stage + (by * nbx + bx) * (GB_TMA_BOXW * GB_TMA_BOXH), w.tmap, box[0] * nchan + bx * GB_TMA_BOXW,
                      box[1] + by * GB_TMA_BOXH, w.bar);
    }
    const int ta = w.tw * w.th;
    for (int i = tid; i < w.nbins; i += nthr) w.hist[i] = 0u;
    if (w.tcol) {
      tile_template_global(w, g_tmpl);
    } else {
      for (int i = tid; i < ta; i += nthr) {
        const float tv = -(float)g_tmpl[i];
        w.tmpl[i] = make_float2(tv, tv);
      }
      for (int i = tid; i < w.nvals; i += nthr) {
        w.tq[i] = g_tq[i];
        w.tv[i] = g_tv[i];
      }
    }
    __syncthreads();
    mbar_wait(w.bar, 0);
    const int lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
    for (int r = warp; r < Sv; r += nwarp) {
      const uint8_t* rowb = stage + (r >> 3) * nbx * (GB_TMA_BOXW * GB_TMA_BOXH) + (r & 7) * GB_TMA_BOXW;
      for (int c = lane; c < Su; c += 32) {
        unsigned v = 0;
        for (int ch = 0; ch < nchan; ++ch) {
          const int x = c * nchan + ch;
          v += rowb[(x >> 5) * (GB_TMA_BOXW * GB_TMA_BOXH) + (x & 31)];
        }
        w.raw[r * Su + c] = (uint16_t)v;
        atomicAdd(&w.hist[v], 1u);
      }
    }
  } else
  // 1. raw window, template and its CDF; clear the histogram.  Every global load a thread needs first is issued
  //    before anything waits on one (the template words, then four window pixels per trip): the phase costs about
  //    one memory round trip instead of one per loop.
  {
    const int ta = w.tw * w.th;
    const double t_first = tid < ta ? g_tmpl[tid] : 0.0;
    const double q_first = tid < w.nvals ? g_tq[tid] : 0.0;
    const double v_first = tid < w.nvals ? g_tv[tid] : 0.0;
    const uint8_t* px = pixels + (int64_t)box[1] * pitch + (int64_t)box[0] * nchan;
    for (int e0 = tid; e0 < area; e0 += 4 * nthr) {
      unsigned v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int e = e0 + k * nthr;
        v[k] = 0;
        if (e < area) {
          const int r = e / Su, c = e - r * Su;
          const uint8_t* q = px + (int64_t)r * pitch + c * nchan;
          v[k] = q[0];
          for (int ch = 1; ch < nchan; ++ch) v[k] += q[ch];
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int e = e0 + k * nthr;
        if (e < area) w.raw[e] = (uint16_t)v[k];
      }
    }
    for (int i = tid; i < w.nbins; i += nthr) w.hist[i] = 0u;
    if (w.tcol) {
      tile_template_global(w, g_tmpl);
    } else {
      for (int i = tid; i < ta; i += nthr) {
        const float tv = -(float)(i == tid ? t_first : g_tmpl[i]);
        w.tmpl[i] = make_float2(tv, tv);
      }
      for (int i = tid; i < w.nvals; i += nthr) {
        w.tq[i] = i == tid ? q_first : g_tq[i];
        w.tv[i] = i == tid ? v_first : g_tv[i];
      }
    }
  }
  __syncthreads();
  // 2. histogram of grey levels + reflect-padded, row-paired copy of the window for the median
  if (!by_tma && !ranked)
    for (int i = tid; i < area; i += nthr) atomicAdd(&w.hist[w.raw[i]], 1u);
  const bool hp_plain = w.hp_mode == GB_HP_REFLECT && w.hp_org_r == 0 && w.hp_org_c == 0 && !w.hp_fp;
  const bool hp5 = w.mh == 5 && w.mw == 5 && hp_plain;
  if (!hp5) {
    // other median sizes / border modes (Tracker.highpass): a plain copy of the window, since hp overwrites raw
    uint16_t* copy = reinterpret_cast<uint16_t*>(w.packed);
    for (int i = tid; i < area; i += nthr) copy[i] = w.raw[i];
  } else {
    const int PW = Su + 4, PH = Sv + 4;
    for (int i = tid; i < PW * PH; i += nthr) {
      const int pr = i / PW, pc = i - pr * PW;
      const int cc = reflect_index(pc - 2, Su);
      const uint32_t lo = w.raw[reflect_index(pr - 2, Sv) * Su + cc], hi = w.raw[reflect_index(pr - 1, Sv) * Su + cc];
      w.packed[i] = lo | (hi << 16);
    }
  }
  __syncthreads();
  // 3. inclusive cumulative counts (one warp; nbins <= 1024); empty levels are marked with 0
  if (tid < 32) {
    const int per = (w.nbins + 31) / 32;
    const int b0 = tid * per, b1 = min(b0 + per, w.nbins);
    uint32_t sum = 0;
    for (int b = b0; b < b1; ++b) sum += w.hist[b];
    uint32_t incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
      if (tid >= d) incl += o;
    }
    uint32_t run = incl - sum;
    for (int b = b0; b < b1; ++b) {
      const uint32_t h = w.hist[b];
      run += h;
      w.hist[b] = h ? run : 0u;
    }
  }
  __syncthreads();
  // 4. look-up table: matched value of every occupied grey level (helpers.py:488-493)
  for (int b = tid; b < w.nbins; b += nthr) {
    const uint32_t cle = w.hist[b];
    if (cle) w.lut[b] = interp_clamped(quo((double)cle, (double)area), w.tq, w.tv, w.nvals);
  }
  __syncthreads();
  if (clk && threadIdx.x == 0) clk[0] = clock64();
  // 5. high-pass: matched value minus the matched 5x5 median (tracker.py:530-531), cast to float32
  //    as the reference does for matchTemplate (tracker.py:610).  One thread = pixels (r, c), (r+1, c).
  if (!hp5 && !hp_plain) {
    // general border mode / origin: the border constant takes its place among the grey levels through the matched values
    __shared__ int s_cval_level;
    if (tid == 0) s_cval_level = w.nbins;
    __syncthreads();
    for (int b = tid; b < w.nbins; b += nthr)
      if (w.hist[b] && !(w.lut[b] < w.hp_cval)) atomicMin(&s_cval_level, b);  // smallest occupied level whose value is >= cval
    __syncthreads();
    const int cval_code = 2 * s_cval_level;
    const uint16_t* copy = reinterpret_cast<const uint16_t*>(w.packed);
    for (int i = tid; i < area; i += nthr) {
      const int r = i / Su, c = i - r * Su;
      const int code = median_window_codes(copy, Su, Sv, r, c, w.mh, w.mw, w.hp_mode, w.hp_org_r, w.hp_org_c, cval_code, w.hp_fp, w.nbins);
      const double med = (code & 1) ? w.lut[code >> 1] : w.hp_cval;
      const float o = (float)sub(w.lut[copy[i]], med);
      w.hp[r * Sp + c] = o;
      if (dump_search && i < dump_cap) dump_search[i] = o;
    }
  } else if (!hp5) {
    const uint16_t* copy = reinterpret_cast<const uint16_t*>(w.packed);
    for (int i = tid; i < area; i += nthr) {
      const int r = i / Su, c = i - r * Su;
      const int med = median_window(copy, Su, Sv, r, c, w.mh, w.mw, w.nbins);
      const float o = (float)sub(w.lut[copy[i]], w.lut[med]);
      w.hp[r * Sp + c] = o;
      if (dump_search && i < dump_cap) dump_search[i] = o;
    }
  } else {
    const int PW = Su + 4, pairs = ((Sv + 1) / 2) * Su;
    for (int i = tid; i < pairs; i += nthr) {
      const int rp = i / Su, c = i - rp * Su, r = 2 * rp;
      uint32_t v[25];
#pragma unroll
      for (int a = 0; a < 5; ++a) {
        const uint32_t* row = w.packed + (r + a) * PW + c;
#pragma unroll
        for (int b = 0; b < 5; ++b) v[a * 5 + b] = row[b];
      }
      const uint32_t self = v[12];
      const uint32_t med = gb_median25_u16x2(v);
      {
        const float o = (float)sub(w.lut[self & 0xffffu], w.lut[med & 0xffffu]);
        w.hp[r * Sp + c] = o;
        if (dump_search && r * Su + c < dump_cap) dump_search[r * Su + c] = o;
      }
      if (r + 1 < Sv) {
        const float o = (float)sub(w.lut[self >> 16], w.lut[med >> 16]);
        w.hp[(r + 1) * Sp + c] = o;
        if (dump_search && (r + 1) * Su + c < dump_cap) dump_search[(r + 1) * Su + c] = o;
      }
    }
  }
  __syncthreads();
  if (clk && threadIdx.x == 0) clk[1] = clock64();
}

// How the 32 lanes of a warp tile the SSD surface: `cw` lanes along the columns, two adjacent output columns each, times
// 32 / cw groups of four output rows.  Narrow surfaces get more row groups so that lanes are not left idle.
struct SsdLanes {
  int cw, rh, RG, CB;  // lanes per row group, row groups per warp, item grid
  __device__ __forceinline__ SsdLanes(int Mu, int Mv) {
    cw = Mu > 32 ? 32 : (Mu > 16 ? 16 : 8);
    rh = 32 / cw;
    RG = (Mv + 4 * rh - 1) / (4 * rh);
    CB = (Mu + 2 * cw - 1) / (2 * cw);
  }
  // first output row / column of a lane in item (rg, cb)
  __device__ __forceinline__ int row(int rg, int lane) const { return (rg * rh + lane / cw) * 4; }
  __device__ __forceinline__ int col(int cb, int lane) const { return 2 * (cb * cw + (lane & (cw - 1))); }
};

// One pixel pair of the high-passed tile; the pair starts at an even float index when ALIGNED.
template <bool ALIGNED>
__device__ __forceinline__ float2 ssd_load(const float* p) {
  if (ALIGNED) return *reinterpret_cast<const float2*>(p);
  return make_float2(p[0], p[1]);
}

// One column of the template as the pairs (-t, -t), row by row: from the shared copy [th][tw] of small templates, or from the
// column-major float copy of a large one in global memory (every lane of the warp reads the same address: one broadcast
// load, and eight consecutive rows share a 32-byte sector).
struct TmplShared {
  const float2* p;
  int tw;
  __device__ __forceinline__ float2 operator[](int ip) const { return p[ip * tw]; }
};
struct TmplGlobal {
  const float* p;
  __device__ __forceinline__ float2 operator[](int ip) const {
    const float t = p[ip];
    return make_float2(t, t);
  }
};

// SSD of one lane: output rows r0 .. r0 + kmax - 1 (kmax <= 4), output columns c (even) and c + 1, template columns
// [jlo, jhi).  Packed FP32 arithmetic (FADD2 / FFMA2, new in sm_100): the two columns share every instruction, each half
// an ordinary IEEE operation, so the sums are bit-identical to scalar code.  The four row outputs stay in registers
// while the template column slides past; the template is stored negated (d = pixel + (-t)).
template <bool ALIGNED, class TC>
__device__ __forceinline__ void ssd_column(const TileWork& w, const float* Icol, const TC Tcol, int kmax, float2 (&a)[4]) {
  const int th = w.th, Sp = w.Sp;
  const int nrow = th + kmax - 1;
  if (th >= 4) {
    // ta, tb, tc = template rows ip-1, ip-2, ip-3; output row k pairs image row ip with template row ip-k
    float2 ta, tb, tc, d;
    {
      const float2 t_0 = Tcol[0], t_1 = Tcol[1], t_2 = Tcol[2];
      const float2 i_0 = ssd_load<ALIGNED>(Icol), i_1 = ssd_load<ALIGNED>(Icol + Sp), i_2 = ssd_load<ALIGNED>(Icol + 2 * Sp);
      d = __fadd2_rn(i_0, t_0); a[0] = __ffma2_rn(d, d, a[0]);
      d = __fadd2_rn(i_1, t_1); a[0] = __ffma2_rn(d, d, a[0]);
      d = __fadd2_rn(i_1, t_0); a[1] = __ffma2_rn(d, d, a[1]);
      d = __fadd2_rn(i_2, t_2); a[0] = __ffma2_rn(d, d, a[0]);
      d = __fadd2_rn(i_2, t_1); a[1] = __ffma2_rn(d, d, a[1]);
      d = __fadd2_rn(i_2, t_0); a[2] = __ffma2_rn(d, d, a[2]);
      ta = t_2; tb = t_1; tc = t_0;
    }
#pragma unroll 4
    for (int ip = 3; ip < th; ++ip) {
      const float2 tn = Tcol[ip];
      const float2 iv = ssd_load<ALIGNED>(Icol + ip * Sp);
      d = __fadd2_rn(iv, tn); a[0] = __ffma2_rn(d, d, a[0]);
      d = __fadd2_rn(iv, ta); a[1] = __ffma2_rn(d, d, a[1]);
      d = __fadd2_rn(iv, tb); a[2] = __ffma2_rn(d, d, a[2]);
      d = __fadd2_rn(iv, tc); a[3] = __ffma2_rn(d, d, a[3]);
      tc = tb; tb = ta; ta = tn;
    }
    // tail: image rows th .. th + kmax - 2 only feed output rows 1..3
    if (th < nrow) {
      const float2 iv = ssd_load<ALIGNED>(Icol + th * Sp);
      d = __fadd2_rn(iv, ta); a[1] = __ffma2_rn(d, d, a[1]);
      d = __fadd2_rn(iv, tb); a[2] = __ffma2_rn(d, d, a[2]);
      d = __fadd2_rn(iv, tc); a[3] = __ffma2_rn(d, d, a[3]);
    }
    if (th + 1 < nrow) {
      const float2 iv = ssd_load<ALIGNED>(Icol + (th + 1) * Sp);
      d = __fadd2_rn(iv, ta); a[2] = __ffma2_rn(d, d, a[2]);
      d = __fadd2_rn(iv, tb); a[3] = __ffma2_rn(d, d, a[3]);
    }
    if (th + 2 < nrow) {
      const float2 iv = ssd_load<ALIGNED>(Icol + (th + 2) * Sp);
      d = __fadd2_rn(iv, ta); a[3] = __ffma2_rn(d, d, a[3]);
    }
  } else {
    const float2 zero = make_float2(0.0f, 0.0f);
    float2 t0 = zero, t1 = zero, t2 = zero, t3 = zero;
    for (int ip = 0; ip < nrow; ++ip) {
      t3 = t2;
      t2 = t1;
      t1 = t0;
      t0 = ip < th ? Tcol[ip] : zero;
      const float2 iv = ssd_load<ALIGNED>(Icol + ip * Sp);
      if (ip < th) { const float2 d = __fadd2_rn(iv, t0); a[0] = __ffma2_rn(d, d, a[0]); }
      if (ip >= 1 && ip <= th) { const float2 d = __fadd2_rn(iv, t1); a[1] = __ffma2_rn(d, d, a[1]); }
      if (ip >= 2 && ip <= th + 1) { const float2 d = __fadd2_rn(iv, t2); a[2] = __ffma2_rn(d, d, a[2]); }
      if (ip >= 3 && ip <= th + 2) { const float2 d = __fadd2_rn(iv, t3); a[3] = __ffma2_rn(d, d, a[3]); }
    }
  }
}

// SSD of one lane of a warp item.  (r0, c) as given by SsdLanes; lanes beyond the surface are clamped onto it (their
// results are discarded by the caller) so that every load stays inside the tile.
__device__ __forceinline__ void ssd_warp_item(const TileWork& w, int r0, int c, int jlo, int jhi, float2 (&acc)[4]) {
  const float2 zero = make_float2(0.0f, 0.0f);
  acc[0] = acc[1] = acc[2] = acc[3] = zero;
  const int rc = min(r0, w.Mv - 1), cc = min(c, (w.Mu - 1) & ~1);
  const int kmax = max(1, min(4, w.Mv - rc));
  if (w.tcol) {
    for (int j = jlo; j < jhi; ++j) {
      const float* Icol = w.hp + rc * w.Sp + cc + j;
      const TmplGlobal Tcol{w.tcol + j * w.th};
      if (j & 1) ssd_column<false>(w, Icol, Tcol, kmax, acc);
      else ssd_column<true>(w, Icol, Tcol, kmax, acc);
    }
    return;
  }
  for (int j = jlo; j < jhi; ++j) {
    const float* Icol = w.hp + rc * w.Sp + cc + j;
    const TmplShared Tcol{w.tmpl + j, w.tw};
    if (j & 1) ssd_column<false>(w, Icol, Tcol, kmax, acc);  // cc is even and rows start 16-byte aligned: parity of j decides
    else ssd_column<true>(w, Icol, Tcol, kmax, acc);
  }
}

// SSD of one lane over every template column, for the organisations that give a warp item the whole template (planar, staged).
// A large template is summed in four column slices, added in the order tile_finish_interleaved adds its slices: one running
// float32 sum of up to 16 384 products drifts ~1.7e-5 from the exact SSD, four slices of a quarter stay within ~4e-6.
__device__ __forceinline__ void ssd_warp_item_all(const TileWork& w, int r0, int c, float2 (&acc)[4]) {
  if (!w.tcol) {
    ssd_warp_item(w, r0, c, 0, w.tw, acc);
    return;
  }
  const int jper = (w.tw + 3) / 4;
  ssd_warp_item(w, r0, c, 0, jper, acc);
#pragma unroll 1
  for (int jp = 1; jp < 4; ++jp) {
    float2 part[4];
    ssd_warp_item(w, r0, c, jp * jper, min((jp + 1) * jper, w.tw), part);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      acc[k].x = __fadd_rn(acc[k].x, part[k].x);
      acc[k].y = __fadd_rn(acc[k].y, part[k].y);
    }
  }
}

// Phases 6-7 with the surface in its final interleaved form (F, F_u, F_v, F_uv per cell) in `w.herm`.
__device__ inline void tile_finish_interleaved(TileWork& w, float* dump_sse, int64_t dump_cap, long long* clk) {
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
  const int Mu = w.Mu, Mv = w.Mv, Mp = w.Mp;
  // 6. area-normalised sum of squared differences (tracker.py:609-614).  One warp owns a block of
  //    4 output rows x 32 output columns and a slice of the template columns: lanes run along the
  //    image row (conflict-free loads, template values broadcast) and each lane keeps the four row
  //    outputs in registers while the template column slides past.  Slices land in the unused
  //    components of the Hermite cells and are summed in a fixed order (bit-reproducible).
  {
    const int tw = w.tw, th = w.th;
    const SsdLanes L(Mu, Mv);
    int JP = 1;
    while (JP < 4 && JP * 2 * L.RG * L.CB <= nwarp && JP * 2 <= tw) JP *= 2;
    const int jper = (tw + JP - 1) / JP;
    const int items = L.RG * L.CB * JP;
    float* hf = reinterpret_cast<float*>(w.herm);
    for (int item = warp; item < items; item += nwarp) {
      const int jp = item % JP, blk = item / JP;
      const int rg = blk / L.CB, cb = blk - rg * L.CB;
      const int r0 = L.row(rg, lane), c = L.col(cb, lane);
      const int jlo = jp * jper, jhi = min(jlo + jper, tw);
      float2 acc[4];
      ssd_warp_item(w, r0, c, jlo, jhi, acc);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (r0 + k < Mv) {
          if (c < Mu) hf[((r0 + k) * Mp + c) * 4 + jp] = acc[k].x;
          if (c + 1 < Mu) hf[((r0 + k) * Mp + c + 1) * 4 + jp] = acc[k].y;
        }
    }
    __syncthreads();
    const double inv_area = 1.0 / (double)(tw * th);
    for (int o = tid; o < Mu * Mv; o += nthr) {
      const int r = o / Mu, cc = o - r * Mu;
      const float4 part = w.herm[r * Mp + cc];
      float acc = part.x;
      if (JP > 1) acc += part.y;
      if (JP > 2) acc = (acc + part.z) + part.w;
      const float sse = (float)((double)acc * inv_area);
      w.herm[r * Mp + cc] = make_float4(sse, 0.0f, 0.0f, 0.0f);
      if (dump_sse && o < dump_cap) dump_sse[o] = sse;
    }
  }
  __syncthreads();
  if (clk && threadIdx.x == 0) clk[2] = clock64();
  if (!spline_is_hermite(w.ku, w.kv)) {
    // 7'. B-spline coefficients of the interpolating spline of degrees (ku, kv): rows, then columns, in place
    float* base = reinterpret_cast<float*>(w.herm);
    double* abu = w.band;
    double* abv = abu + (int64_t)Mu * (2 * w.ku + 1);
    if (tid == 0) bspline_factor(abu, Mu, w.ku);
    if (tid == 32) bspline_factor(abv, Mv, w.kv);
    __syncthreads();
    for (int r = tid; r < Mv; r += nthr) bspline_solve_line(abu, Mu, w.ku, base + (int64_t)r * Mp * 4, 4);
    __syncthreads();
    for (int c = tid; c < Mu; c += nthr) bspline_solve_line(abv, Mv, w.kv, base + (int64_t)c * 4, Mp * 4);
    __syncthreads();
    return;
  }
  // 7. Hermite data: dF/du along rows and dF/dv along columns, then the cross derivative
  {
    float* base = reinterpret_cast<float*>(w.herm);
    const int Mvp = 32 * ((Mv + 31) / 32);  // rows and columns on separate warps
    for (int line = tid; line < Mvp + Mu; line += nthr) {
      if (line < Mv) {
        spline_slopes_line(base + (int64_t)line * Mp * 4, base + (int64_t)line * Mp * 4 + 1, 4, Mu, w.cub_u);
      } else if (line >= Mvp) {
        const int c = line - Mvp;
        spline_slopes_line(base + (int64_t)c * 4, base + (int64_t)c * 4 + 2, Mp * 4, Mv, w.cub_v);
      }
    }
    __syncthreads();
    for (int c = tid; c < Mu; c += nthr) spline_slopes_line(base + (int64_t)c * 4 + 1, base + (int64_t)c * 4 + 3, Mp * 4, Mv, w.cub_v);
  }
  __syncthreads();
}

// Build the Hermite surface for one search window in `w.herm` (interleaved layout).
__device__ inline void tile_build_surface(const uint8_t* __restrict__ pixels, int pitch, int nchan, const int* box, const double* __restrict__ g_tmpl,
                                          const double* __restrict__ g_tq, const double* __restrict__ g_tv, TileWork& w,
                                          float* dump_search, float* dump_sse, int64_t dump_cap, long long* clk) {
  tile_prepare(pixels, pitch, nchan, box, g_tmpl, g_tq, g_tv, w, dump_search, dump_cap, clk);
  tile_finish_interleaved(w, dump_sse, dump_cap, clk);
}

// ---------------------------------------------------------------------------------------------
// Large search windows (k_s2_large): planar work arrays, so that windows up to ~140 px stay in the
// 200 KB of shared memory one CTA per SM can have.  Regions and lifetimes:
//   R1 = hp [Sv][Sp] float (median -> SSD); hosts the raw u16 window before and the row slopes F_u after
//   R2 = packed u32 [(Sv+4)][(Su+4)] (until the median) / F [Mv][Mq] + one scratch plane [Mv][Mq] (from the SSD on)
// The finished surface is written straight to its global region in the interleaved form k_s3 samples.
// ---------------------------------------------------------------------------------------------
struct TilePlanes {
  float *F, *Fu, *G;  // SSE surface, its row slopes, scratch plane for the column solves
  int Mq;             // plane pitch in floats (odd: row solves of different rows hit different banks)
};

__host__ __device__ inline int64_t tile_bytes_needed_planar(int Su, int Sv, int tw, int th, int nbins, int nvals) {
  const int64_t Mu = Su - tw + 1, Mv = Sv - th + 1, Mq = Mu | 1, Sp = (Su + 3) / 4 * 4;
  const int64_t r1 = align16((int64_t)Sv * Sp * 4);  // >= Mv * Mq * 4 (F_u) and >= Sv * Su * 2 (raw)
  const int64_t packed = (int64_t)(Sv + 4) * (Su + 4) * 4, planes = 2 * align16(Mv * Mq * 4);
  int64_t b = r1 + align16(packed > planes ? packed : planes);
  b += align16((int64_t)nbins * 8) + tile_template_bytes(tw, th, nvals);
  b += align16((int64_t)nbins * 4);
  return b;
}

__device__ inline void tile_carve_planar(char* base, TileWork& w, TilePlanes& pl) {
  w.Mp = w.Mu | 1;
  w.Sp = (w.Su + 3) / 4 * 4;
  w.Tp = (w.tw + 3) / 4 * 4;
  pl.Mq = w.Mu | 1;
  char* p = base;
  w.hp = reinterpret_cast<float*>(p);
  w.raw = reinterpret_cast<uint16_t*>(p);
  pl.Fu = reinterpret_cast<float*>(p);
  p += align16((int64_t)w.Sv * w.Sp * 4);
  const int64_t plane = align16((int64_t)w.Mv * pl.Mq * 4), packed = (int64_t)(w.Sv + 4) * (w.Su + 4) * 4;
  w.packed = reinterpret_cast<uint32_t*>(p);
  w.herm = nullptr;
  pl.F = reinterpret_cast<float*>(p);
  pl.G = reinterpret_cast<float*>(p + plane);
  p += align16(packed > 2 * plane ? packed : 2 * plane);
  w.lut = reinterpret_cast<double*>(p);
  p += align16((int64_t)w.nbins * 8);
  if (!w.tcol) {
    w.tq = reinterpret_cast<double*>(p);
    p += align16((int64_t)w.nvals * 8);
    w.tv = reinterpret_cast<double*>(p);
    p += align16((int64_t)w.nvals * 8);
    w.tmpl = reinterpret_cast<float2*>(p);
    p += align16((int64_t)w.th * w.tw * 8);
  }
  w.hist = reinterpret_cast<uint32_t*>(p);
}

// Phases 6-7 on planes; `out` = the surface's global region, float4 [Mv][Mp].  Same arithmetic as
// tile_finish_interleaved with one template slice (JP = 1), or four for a large template (ssd_warp_item_all).
__device__ inline void tile_finish_planar(TileWork& w, const TilePlanes& pl, float4* __restrict__ out, float* dump_sse,
                                          int64_t dump_cap, long long* clk) {
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
  const int Mu = w.Mu, Mv = w.Mv, Mp = w.Mp, Mq = pl.Mq;
  {
    const SsdLanes L(Mu, Mv);
    const double inv_area = 1.0 / (double)(w.tw * w.th);
    for (int item = warp; item < L.RG * L.CB; item += nwarp) {
      const int rg = item / L.CB, cb = item - rg * L.CB;
      const int r0 = L.row(rg, lane), c = L.col(cb, lane);
      float2 acc[4];
      ssd_warp_item_all(w, r0, c, acc);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (r0 + k < Mv) {
          const float sse[2] = {(float)((double)acc[k].x * inv_area), (float)((double)acc[k].y * inv_area)};
#pragma unroll
          for (int h = 0; h < 2; ++h)
            if (c + h < Mu) {
              pl.F[(r0 + k) * Mq + c + h] = sse[h];
              const int64_t o = (int64_t)(r0 + k) * Mu + c + h;
              if (dump_sse && o < dump_cap) dump_sse[o] = sse[h];
            }
        }
    }
  }
  __syncthreads();  // hp is dead from here on: F_u takes its place
  if (clk && threadIdx.x == 0) clk[2] = clock64();
  {
    // rows (F -> F_u) and columns (F -> F_v in the scratch plane) on separate warps
    const int Mvp = 32 * ((Mv + 31) / 32);
    for (int line = tid; line < Mvp + Mu; line += nthr) {
      if (line < Mv) {
        spline_slopes_line(pl.F + (int64_t)line * Mq, pl.Fu + (int64_t)line * Mq, 1, Mu, w.cub_u);
      } else if (line >= Mvp) {
        const int c = line - Mvp;
        spline_slopes_line(pl.F + c, pl.G + c, Mq, Mv, w.cub_v);
      }
    }
    __syncthreads();
    for (int o = tid; o < Mu * Mv; o += nthr) {
      const int r = o / Mu, c = o - r * Mu;
      out[r * Mp + c] = make_float4(pl.F[r * Mq + c], pl.Fu[r * Mq + c], pl.G[r * Mq + c], 0.0f);
    }
    __syncthreads();
    // cross derivative: columns of F_u into the scratch plane, then into the fourth component
    for (int c = tid; c < Mu; c += nthr) spline_slopes_line(pl.Fu + c, pl.G + c, Mq, Mv, w.cub_v);
    __syncthreads();
    float* outf = reinterpret_cast<float*>(out);
    for (int o = tid; o < Mu * Mv; o += nthr) {
      const int r = o / Mu, c = o - r * Mu;
      outf[((int64_t)r * Mp + c) * 4 + 3] = pl.G[r * Mq + c];
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// Largest search windows (up to ~128 px at 110 KB): every phase still runs out of shared memory, but the phases
// hand their results over through the window's global region, because no two of the big arrays fit at once:
//   prepare:  raw + packed + tables in shared memory, high-passed tile hp written to the region
//   SSD:      hp staged back into shared memory (raw / packed are dead), SSE plane F written to the region
//   Hermite:  two planes in shared memory; F_u, F_v, F_uv are produced one after the other and stored into the
//             interleaved surface as they appear (F_u is reloaded for the cross derivative)
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline int64_t tile_bytes_needed_staged(int Su, int Sv, int tw, int th, int nbins, int nvals) {
  int64_t b = align16((int64_t)Su * Sv * 2) + align16((int64_t)(Sv + 4) * (Su + 4) * 4);
  b += align16((int64_t)nbins * 8) + tile_template_bytes(tw, th, nvals);
  b += align16((int64_t)nbins * 4);
  const int64_t Mu = Su - tw + 1, Mv = Sv - th + 1, planes = 2 * align16(Mv * (Mu | 1) * 4);
  return b > planes ? b : planes;
}

__device__ inline void tile_build_surface_staged(char* smem, char* region, const uint8_t* __restrict__ pixels, int pitch, int nchan,
                                                 const int* box, const double* __restrict__ g_tmpl, const double* __restrict__ g_tq,
                                                 const double* __restrict__ g_tv, TileWork& w, float* dump_search, float* dump_sse,
                                                 int64_t dump_cap, long long* clk) {
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
  w.Mp = w.Mu | 1;
  w.Sp = (w.Su + 3) / 4 * 4;
  w.Tp = (w.tw + 3) / 4 * 4;
  const int Mu = w.Mu, Mv = w.Mv, Mp = w.Mp, Mq = w.Mu | 1;
  char* p = smem;
  w.raw = reinterpret_cast<uint16_t*>(p);
  p += align16((int64_t)w.Su * w.Sv * 2);
  w.packed = reinterpret_cast<uint32_t*>(p);
  p += align16((int64_t)(w.Sv + 4) * (w.Su + 4) * 4);
  w.lut = reinterpret_cast<double*>(p);
  p += align16((int64_t)w.nbins * 8);
  if (!w.tcol) {
    w.tq = reinterpret_cast<double*>(p);
    p += align16((int64_t)w.nvals * 8);
    w.tv = reinterpret_cast<double*>(p);
    p += align16((int64_t)w.nvals * 8);
    w.tmpl = reinterpret_cast<float2*>(p);
    p += align16((int64_t)w.th * w.tw * 8);
  }
  w.hist = reinterpret_cast<uint32_t*>(p);
  w.herm = nullptr;
  float* hp_global = reinterpret_cast<float*>(region);
  w.hp = hp_global;
  tile_prepare(pixels, pitch, nchan, box, g_tmpl, g_tq, g_tv, w, dump_search, dump_cap, clk);
  // hp back into shared memory, over raw / packed (4 Sv Sp <= their 6 S^2 bytes)
  float* hp_s = reinterpret_cast<float*>(smem);
  {
    const int n4 = w.Sv * w.Sp / 4;  // Sp is a multiple of 4
    const float4* src = reinterpret_cast<const float4*>(hp_global);
    float4* dst = reinterpret_cast<float4*>(hp_s);
    for (int i = tid; i < n4; i += nthr) dst[i] = src[i];
  }
  __syncthreads();
  w.hp = hp_s;
  // SSD plane F -> region (hp's global copy is dead)
  float* F_global = reinterpret_cast<float*>(region);
  {
    const SsdLanes L(Mu, Mv);
    const double inv_area = 1.0 / (double)(w.tw * w.th);
    for (int item = warp; item < L.RG * L.CB; item += nwarp) {
      const int rg = item / L.CB, cb = item - rg * L.CB;
      const int r0 = L.row(rg, lane), c = L.col(cb, lane);
      float2 acc[4];
      ssd_warp_item_all(w, r0, c, acc);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (r0 + k < Mv) {
          const float sse[2] = {(float)((double)acc[k].x * inv_area), (float)((double)acc[k].y * inv_area)};
#pragma unroll
          for (int h = 0; h < 2; ++h)
            if (c + h < Mu) {
              F_global[(r0 + k) * Mq + c + h] = sse[h];
              const int64_t o = (int64_t)(r0 + k) * Mu + c + h;
              if (dump_sse && o < dump_cap) dump_sse[o] = sse[h];
            }
        }
    }
  }
  __syncthreads();
  if (clk && threadIdx.x == 0) clk[2] = clock64();
  // Hermite on two planes
  float* P0 = reinterpret_cast<float*>(smem);
  float* P1 = reinterpret_cast<float*>(smem + align16((int64_t)Mv * Mq * 4));
  for (int i = tid; i < Mv * Mq; i += nthr) P0[i] = F_global[i];
  __syncthreads();  // F is in shared memory: the region is free for the final surface
  float* out = reinterpret_cast<float*>(region);
  for (int r = tid; r < Mv; r += nthr) spline_slopes_line(P0 + (int64_t)r * Mq, P1 + (int64_t)r * Mq, 1, Mu, w.cub_u);  // F -> F_u
  __syncthreads();
  for (int o = tid; o < Mu * Mv; o += nthr) {
    const int r = o / Mu, c = o - r * Mu;
    *reinterpret_cast<float2*>(out + ((int64_t)r * Mp + c) * 4) = make_float2(P0[r * Mq + c], P1[r * Mq + c]);
  }
  __syncthreads();
  for (int c = tid; c < Mu; c += nthr) spline_slopes_line(P0 + c, P1 + c, Mq, Mv, w.cub_v);  // F -> F_v
  __syncthreads();
  for (int o = tid; o < Mu * Mv; o += nthr) {
    const int r = o / Mu, c = o - r * Mu;
    out[((int64_t)r * Mp + c) * 4 + 2] = P1[r * Mq + c];
    P0[r * Mq + c] = out[((int64_t)r * Mp + c) * 4 + 1];  // F_u back in (written by this CTA before the last barrier)
  }
  __syncthreads();
  for (int c = tid; c < Mu; c += nthr) spline_slopes_line(P0 + c, P1 + c, Mq, Mv, w.cub_v);  // F_u -> F_uv
  __syncthreads();
  for (int o = tid; o < Mu * Mv; o += nthr) {
    const int r = o / Mu, c = o - r * Mu;
    out[((int64_t)r * Mp + c) * 4 + 3] = P1[r * Mq + c];
  }
  __syncthreads();
}

}  // namespace gb
