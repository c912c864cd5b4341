// Raster.viewshed (reference raster.py:1293-1389): binary visibility of every cell of a DEM from one origin.
//
// The reference bins the cells into rings by their rounded distance in cells, orders every ring by heading and sweeps the
// rings outwards: a cell is visible when its elevation ratio dz / distance exceeds the highest ratio seen so far along its
// heading — the previous ring's running maximum, interpolated periodically (np.interp(..., period=2 pi)) at the cell's
// heading.  The rings depend on each other, the cells of a ring do not.  On the device:
//   k_vs_cells    one thread per cell: ring, heading, ratio; range of the ring numbers
//   k_vs_count    cells per ring          k_vs_scan   ring offsets (one CTA)
//   k_vs_scatter  cells into their ring's bucket (any order)
//   k_vs_sort     one CTA per ring: bitonic sort of (heading, cell index) in shared memory = np.lexsort((heading, ring)); a
//                 ring of more than C cells (the capacity, GB_VS_MAX_RING) is sorted in chunks of C cells
//   k_vs_merge    rings of more than C cells only: pass p merges the sorted runs of C * 2^p cells pairwise, between the bucket
//                 arrays (b_head, b_idx) and the dead heading / ring arrays; a ring of m cells takes ceil(log2(m / C)) passes
//                 and ends in the second pair when that count is odd
//   k_vs_sweep    one CTA walks the rings in order; its threads share a ring's cells; the horizon of the previous ring =
//                 headings modulo 2 pi in increasing order with the two wrap-around entries np.interp adds (in shared memory:
//                 the binary search reads them ~14 times per cell; after a ring of more than C cells only every k-th of them,
//                 and the search ends in a k-entry segment of the global copy) and the running maxima (double-buffered in global
//                 memory)
// Everything but the heading (atan2) is IEEE-exact arithmetic in the reference's order, so the result equals the reference's
// unless a ratio sits within rounding of the interpolated horizon.
// (included by glimpse_b200.cu inside namespace gb, after common.cuh)
#pragma once

#define GB_VS_MAX_RING 16384  // C: cells per ring the sort holds in shared memory (a full circle of radius ~2 600 cells)
#define GB_VS_SORT_THREADS 1024
#define GB_VS_SWEEP_THREADS 1024

// Work buffer: 64 bytes per cell + 12 per ring + 2 KB of alignment and header (viewshed_layout).
struct ViewshedWork {
  int32_t* head;     // [8] status, rmin, rmax, largest ring over C cells (0: none), ...
  int32_t* ring;     // [n]  (after the scatter: the merge passes' second index buffer)
  double* heading;   // [n]  (after the sort: the merge passes' second heading buffer)
  double* ratio;     // [n]
  int32_t* count;    // [R + 1]
  int32_t* start;    // [R + 1]
  int32_t* fill;     // [R + 1]
  double* b_head;    // [n] bucketed, then sorted, headings
  int32_t* b_idx;    // [n] ... and their cells
  double* hx[2];     // [n + 2] a ring's abscissae (headings mod 2 pi, wrapped), double-buffered: the previous ring's stay readable
  double* hf[2];     // [n + 2] horizon ordinates (running maximum of the ratio)
};

__host__ __device__ inline int64_t vs_align(int64_t b) { return (b + 255) / 256 * 256; }

__host__ inline int64_t viewshed_layout(int64_t n, int64_t R, unsigned char* base, ViewshedWork* w) {
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    unsigned char* p = base ? base + off : nullptr;
    off += vs_align(bytes);
    return p;
  };
  unsigned char* p;
  p = take(8 * 4); if (w) w->head = reinterpret_cast<int32_t*>(p);
  p = take(n * 4); if (w) w->ring = reinterpret_cast<int32_t*>(p);
  p = take(n * 8); if (w) w->heading = reinterpret_cast<double*>(p);
  p = take(n * 8); if (w) w->ratio = reinterpret_cast<double*>(p);
  p = take((R + 1) * 4); if (w) w->count = reinterpret_cast<int32_t*>(p);
  p = take((R + 1) * 4); if (w) w->start = reinterpret_cast<int32_t*>(p);
  p = take((R + 1) * 4); if (w) w->fill = reinterpret_cast<int32_t*>(p);
  p = take(n * 8); if (w) w->b_head = reinterpret_cast<double*>(p);
  p = take(n * 4); if (w) w->b_idx = reinterpret_cast<int32_t*>(p);
  for (int k = 0; k < 2; ++k) {  // (a ring holds at most n cells)
    p = take((n + 2) * 8); if (w) w->hx[k] = reinterpret_cast<double*>(p);
    p = take((n + 2) * 8); if (w) w->hf[k] = reinterpret_cast<double*>(p);
  }
  return off;
}

struct ViewshedParams {
  const double* z;   // (ny, nx) row-major
  const double* xc;  // [nx] cell-centre x in array order
  const double* yc;  // [ny]
  int32_t nx, ny, R, has_corr;
  int32_t cap;       // C, 1..GB_VS_MAX_RING: rings of more cells take the chunked sort, the merge and the sampled search
  double ox, oy, oz, inv_cell, corr_c1, corr_c2;
  ViewshedWork w;
  uint8_t* visible;
};

__global__ void k_vs_init(const __grid_constant__ ViewshedParams q) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i == 0) {
    q.w.head[0] = 0;
    q.w.head[1] = 0x7fffffff;
    q.w.head[2] = -1;
    q.w.head[3] = 0;
  }
  if (i <= q.R) {
    q.w.count[i] = 0;
    q.w.fill[i] = 0;
  }
}

__global__ void k_vs_cells(const __grid_constant__ ViewshedParams q) {
  const int64_t n = (int64_t)q.nx * q.ny;
  int lo = 0x7fffffff, hi = -1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / q.nx), c = (int)(i - (int64_t)r * q.nx);
    const double dx = sub(q.xc[c], q.ox), dy = sub(q.yc[r], q.oy);
    double dz = sub(q.z[i], q.oz);
    const double d2 = add(mul(dx, dx), mul(dy, dy));
    if (q.has_corr) dz = add(dz, quo(mul(q.corr_c1, d2), q.corr_c2));  // helpers.elevation_corrections (helpers.py:1790)
    const double dist = sqrt(d2);
    const double cells = add(mul(dist, q.inv_cell), 0.5);
    const int ring = cells < 2147483000.0 ? (int)cells : 2147483000;
    q.w.ring[i] = ring;
    double h = atan2(dy, dx);
    if (h == 0.0) h = 0.0;  // (-0.0 and +0.0 are one key)
    q.w.heading[i] = h;
    q.w.ratio[i] = quo(dz, dist);
    lo = min(lo, ring);
    hi = max(hi, ring);
  }
  lo = __reduce_min_sync(0xffffffffu, lo);
  hi = __reduce_max_sync(0xffffffffu, hi);
  if ((threadIdx.x & 31) == 0 && hi >= 0) {
    atomicMin(&q.w.head[1], lo);
    atomicMax(&q.w.head[2], hi);
  }
}

__global__ void k_vs_count(const __grid_constant__ ViewshedParams q) {
  const int64_t n = (int64_t)q.nx * q.ny;
  const int rmin = q.w.head[1], span = q.w.head[2] - rmin + 1;
  if (span > q.R) {
    if (blockIdx.x == 0 && threadIdx.x == 0) q.w.head[0] = 2;  // more rings than the work buffer was sized for
    return;
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(&q.w.count[q.w.ring[i] - rmin], 1);
}

// Exclusive scan of the ring sizes (one CTA; R <= nx + ny + 2).
__global__ void k_vs_scan(const __grid_constant__ ViewshedParams q) {
  __shared__ int s_carry;
  __shared__ int s_warp[32];
  if (q.w.head[0] != 0) return;
  const int span = q.w.head[2] - q.w.head[1] + 1;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < span; base += blockDim.x) {
    const int i = base + tid;
    const int v = i < span ? q.w.count[i] : 0;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int x = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += x;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int off = s_carry;
    for (int k = 0; k < warp; ++k) off += s_warp[k];
    if (i < span) {
      q.w.start[i] = off + incl - v;
      if (v > q.cap) atomicMax(&q.w.head[3], v);  // a ring for the merge passes
    }
    __syncthreads();
    if (tid == blockDim.x - 1) s_carry = off + incl;
    __syncthreads();
  }
  if (tid == 0) q.w.start[span] = s_carry;
}

__global__ void k_vs_scatter(const __grid_constant__ ViewshedParams q) {
  if (q.w.head[0] != 0) return;
  const int64_t n = (int64_t)q.nx * q.ny;
  const int rmin = q.w.head[1];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = q.w.ring[i] - rmin;
    const int pos = q.w.start[b] + atomicAdd(&q.w.fill[b], 1);
    q.w.b_head[pos] = q.w.heading[i];
    q.w.b_idx[pos] = (int)i;
  }
}

__device__ __forceinline__ uint64_t vs_orderable(double v) {
  const uint64_t b = (uint64_t)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// One CTA per ring: (heading, cell) ascending — np.lexsort((heading, ring)) is stable, so equal headings keep cell order.  A
// ring of more than q.cap cells is sorted in runs of q.cap cells, which k_vs_merge joins.
__global__ void __launch_bounds__(GB_VS_SORT_THREADS) k_vs_sort(const __grid_constant__ ViewshedParams q) {
  extern __shared__ __align__(16) unsigned char vs_raw[];
  if (q.w.head[0] != 0) return;
  const int b = blockIdx.x;
  if (b > q.w.head[2] - q.w.head[1]) return;
  const int m_ring = q.w.count[b];
  if (m_ring <= 1) {
    // (the sweep wants the number of negative headings of every ring: they follow the others modulo 2 pi)
    if (threadIdx.x == 0) q.w.fill[b] = (m_ring == 1 && q.w.b_head[q.w.start[b]] < 0.0) ? 1 : 0;
    return;
  }
  int n_neg = 0;  // (thread 0's)
  for (int c0 = 0; c0 < m_ring; c0 += q.cap) {
    const int m = min(m_ring - c0, q.cap);
    const int s0 = q.w.start[b] + c0;
    int cap = 1;
    while (cap < m) cap <<= 1;
    uint64_t* key = reinterpret_cast<uint64_t*>(vs_raw);
    uint32_t* idx = reinterpret_cast<uint32_t*>(key + cap);
    if (c0 > 0) __syncthreads();  // the previous run's keys are read
    for (int i = threadIdx.x; i < cap; i += blockDim.x) {
      key[i] = i < m ? vs_orderable(q.w.b_head[s0 + i]) : ~0ull;
      idx[i] = i < m ? (uint32_t)q.w.b_idx[s0 + i] : 0xffffffffu;
    }
    __syncthreads();
    for (int k = 2; k <= cap; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < cap; i += blockDim.x) {
          const int l = i ^ j;
          if (l > i) {
            const bool up = (i & k) == 0;
            const uint64_t ka = key[i], kb = key[l];
            const uint32_t ia = idx[i], ib = idx[l];
            const bool greater = ka > kb || (ka == kb && ia > ib);
            if (greater == up) {
              key[i] = kb;
              key[l] = ka;
              idx[i] = ib;
              idx[l] = ia;
            }
          }
        }
        __syncthreads();
      }
    }
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      const uint32_t c = idx[i];
      q.w.b_idx[s0 + i] = (int)c;
      q.w.b_head[s0 + i] = q.w.heading[c];
    }
    if (threadIdx.x == 0) {
      // negative headings come first: their orderable keys have the top bit clear
      int lo = 0, hi = m;  // first i with the top bit set
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (key[mid] >> 63) hi = mid; else lo = mid + 1;
      }
      n_neg += lo;
    }
  }
  if (threadIdx.x == 0) q.w.fill[b] = n_neg;
}

// Merge passes of the rings of more than q.cap cells: k_vs_sort left runs of q.cap cells; pass p merges the runs of
// q.cap * 2^p cells pairwise.  Even passes read (b_head, b_idx) and write (heading, ring), odd passes the other way round, so a
// ring ends in the second pair when its number of passes (vs_merge_passes) is odd.  The keys (heading, cell) are all distinct,
// so a cell's place is its place in its run plus the number of cells of the partner run with a smaller key.
__host__ __device__ __forceinline__ int vs_merge_passes(int m, int cap) {
  int p = 0;
  for (int64_t run = cap; run < m; run <<= 1) ++p;
  return p;
}

__global__ void k_vs_merge(const __grid_constant__ ViewshedParams q, int pass) {
  if (q.w.head[0] != 0) return;
  const int64_t run = (int64_t)q.cap << pass;
  if (q.w.head[3] <= run) return;  // no ring needs this pass
  const int span = q.w.head[2] - q.w.head[1] + 1;
  const int total = q.w.start[span];
  const double* sh = (pass & 1) ? q.w.heading : q.w.b_head;
  const int32_t* si = (pass & 1) ? q.w.ring : q.w.b_idx;
  double* dh = (pass & 1) ? q.w.b_head : q.w.heading;
  int32_t* di = (pass & 1) ? q.w.b_idx : q.w.ring;
  for (int64_t pos = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; pos < total; pos += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = span;  // the ring of pos: the last b with start[b] <= pos (empty rings share their successor's start)
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (q.w.start[mid] <= pos) lo = mid; else hi = mid;
    }
    const int m = q.w.count[lo];
    if (m <= run) continue;
    const int64_t s0 = q.w.start[lo], e = pos - s0;
    const double h = sh[pos];
    const int32_t c = si[pos];
    const uint64_t key = vs_orderable(h);
    const int64_t r = e / run, left = (r & ~1ll) * run;  // first cell of the pair
    const bool in_left = (r & 1) == 0;
    int64_t p0 = in_left ? left + run : left, p1 = in_left ? min(left + 2 * run, (int64_t)m) : left + run;  // the partner run
    int64_t out = in_left ? e : e - run;
    if (p0 < p1) {  // cells of the partner run below (h, c)
      int64_t a = p0, z = p1;
      while (a < z) {
        const int64_t mid = (a + z) >> 1;
        const uint64_t km = vs_orderable(sh[s0 + mid]);
        if (km < key || (km == key && si[s0 + mid] < c)) a = mid + 1; else z = mid;
      }
      out += a - p0;
    }
    dh[s0 + out] = h;
    di[s0 + out] = c;
  }
}

// np.interp's compiled loop for one abscissa (numpy compiled_base.c arr_interp): xp increasing, n >= 1.  vs_interp_at: from
// the j the search found.
template <typename XP>
__device__ __forceinline__ double vs_interp_at(double x, int j, XP xp, const double* __restrict__ fp, int n) {
  if (j == n - 1 || xp(j) == x) return fp[j];
  const double slope = quo(sub(fp[j + 1], fp[j]), sub(xp(j + 1), xp(j)));
  double r = add(mul(slope, sub(x, xp(j))), fp[j]);
  if (isnan(r)) {  // "if we get nan in one direction, try the other"
    r = add(mul(slope, sub(x, xp(j + 1))), fp[j + 1]);
    if (isnan(r) && fp[j] == fp[j + 1]) r = fp[j];
  }
  return r;
}

// The same for a horizon of more entries than shared memory holds: xs = xp[0], xp[k], xp[2k], ... in shared memory, xp and fp
// in global memory (xp written by this CTA: read through L2).  The search ends in the k-entry segment xs brackets, so j is again
// the largest with xp[j] <= x.
__device__ inline double vs_interp_sampled(double x, const double* __restrict__ xs, int k, const double* xp,
                                           const double* __restrict__ fp, int n) {
  const auto xg = [xp](int i) { return __ldcg(xp + i); };
  if (isnan(x)) return x;
  if (x < xs[0]) return fp[0];
  if (x > xg(n - 1)) return fp[n - 1];
  int lo = 0, hi = (n - 1) / k + 1;  // largest t with xs[t] <= x
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (xs[mid] <= x) lo = mid; else hi = mid;
  }
  lo *= k;
  hi = min(lo + k, n);
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (xg(mid) <= x) lo = mid; else hi = mid;
  }
  return vs_interp_at(x, lo, xg, fp, n);
}

__device__ inline double vs_interp(double x, const double* __restrict__ xp, const double* __restrict__ fp, int n) {
  if (isnan(x)) return x;
  if (x < xp[0]) return fp[0];
  if (x > xp[n - 1]) return fp[n - 1];
  int lo = 0, hi = n;  // largest j with xp[j] <= x
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (xp[mid] <= x) lo = mid; else hi = mid;
  }
  return vs_interp_at(x, lo, [xp](int i) { return xp[i]; }, fp, n);
}

#define GB_VS_TWO_PI 6.283185307179586

__device__ __forceinline__ double vs_mod_period(double h) {  // np.remainder(h, 2 pi) for |h| <= pi
  if (h < 0.0) return add(h, GB_VS_TWO_PI);
  return h == 0.0 ? 0.0 : h;
}

// LARGE = false: every ring has at most q.cap cells (head[3] == 0); LARGE = true: some ring has more, so a ring may sit in the
// merge passes' second buffer pair, and the ring after one searches the sampled horizon.  Both are launched; the one that does
// not apply returns at once, so the common case keeps a kernel of its own registers.
template <bool LARGE>
__global__ void __launch_bounds__(GB_VS_SWEEP_THREADS) k_vs_sweep(const __grid_constant__ ViewshedParams q) {
  extern __shared__ __align__(16) unsigned char vs_sweep_raw[];
  // [prev_m + 2] abscissae of the previous ring's horizon; after a ring of more than q.cap cells every prev_k-th of them
  double* xp_s = reinterpret_cast<double*>(vs_sweep_raw);
  __shared__ int s_cnt[2];  // unknown horizons, newly opened cells (only while the horizon still has NaN)
  constexpr int VS_BATCH = 4;
  const int64_t n = (int64_t)q.nx * q.ny;
  const int tid = threadIdx.x, nthr = GB_VS_SWEEP_THREADS;
  if (q.w.head[0] != 0 || (q.w.head[3] != 0) != LARGE) return;
  const int rmin = q.w.head[1], span = q.w.head[2] - rmin + 1;
  // a raster that is one ring: all visible if that ring is ring 0 (raster.py:1343-1345), otherwise that ring is the first
  int rings_with_cells = 0;  // (of this thread's rings: there are ~15 000 rings in a DEM of 10^8 cells)
  for (int b = tid; b < span; b += nthr) rings_with_cells += q.w.count[b] > 0;
  const bool one_ring = __syncthreads_count(rings_with_cells > 0) == 1 && !__syncthreads_or(rings_with_cells > 1);
  if (one_ring && rmin == 0) {
    for (int64_t i = tid; i < n; i += nthr) q.visible[i] = 1;
    return;
  }
  for (int64_t i = tid; i < n; i += nthr) q.visible[i] = 0;
  bool first = true, has_nan = false;
  int prev_m = 0, prev_k = 1, cur = 0;
  for (int b = 0; b < span; ++b) {
    const int m = q.w.count[b];
    if (m == 0) continue;
    if (b == 0 && rmin == 0) continue;  // the cells within half a cell of the origin are not visited (raster.py:1336-1338)
    const int s0 = q.w.start[b], n_neg = q.w.fill[b];
    const double* r_head = q.w.b_head;
    const int32_t* r_idx = q.w.b_idx;
    if constexpr (LARGE) {
      if (vs_merge_passes(m, q.cap) & 1) {  // k_vs_merge left the ring in its second buffer pair
        r_head = q.w.heading;
        r_idx = q.w.ring;
      }
    }
    const double* pf = q.w.hf[cur ^ 1];
    const double* px = q.w.hx[cur ^ 1];
    double* nf_ = q.w.hf[cur];
    double* nx_ = q.w.hx[LARGE ? cur : 0];  // this ring's abscissae on their way to shared memory
    if (has_nan) {
      if (tid < 2) s_cnt[tid] = 0;
      __syncthreads();
    }
    int unknown = 0, opened = 0, nans = 0;
    // the ring's cells of this thread, four at a time: their loads are issued before the first use (two memory round trips)
    for (int k0 = 0; k0 * nthr < m; k0 += VS_BATCH) {
      double h[VS_BATCH], r[VS_BATCH];
      int cell[VS_BATCH];
#pragma unroll
      for (int k = 0; k < VS_BATCH; ++k) {
        const int j = tid + (k0 + k) * nthr;
        if (j < m) {
          h[k] = r_head[s0 + j];
          cell[k] = r_idx[s0 + j];
        }
      }
#pragma unroll
      for (int k = 0; k < VS_BATCH; ++k)
        if (tid + (k0 + k) * nthr < m) r[k] = q.w.ratio[cell[k]];
#pragma unroll
      for (int k = 0; k < VS_BATCH; ++k) {
        const int j = tid + (k0 + k) * nthr;
        if (j < m) {
          const double x = vs_mod_period(h[k]);
          double hor;
          bool seen;
          if (first) {
            seen = !isnan(r[k]);
            hor = r[k];
            nans |= isnan(r[k]);
          } else {
            if (LARGE && prev_k > 1)
              hor = vs_interp_sampled(x, xp_s, prev_k, px, pf, prev_m + 2);
            else
              hor = vs_interp(x, xp_s, pf, prev_m + 2);
            seen = r[k] > hor;
            if (has_nan) {
              const bool unk = isnan(hor);
              const bool open = unk && !isnan(r[k]);
              seen |= open;
              unknown += unk;
              opened += open;
            }
            if (seen) hor = r[k];
          }
          q.visible[cell[k]] = seen ? 1 : 0;
          // np.interp's periodic preparation for the next ring: abscissae modulo 2 pi in increasing order (the negatives,
          // shifted by 2 pi, follow the non-negatives) with one wrapped entry at either end
          const int pos = j >= n_neg ? j - n_neg : j + (m - n_neg);
          nf_[1 + pos] = hor;
          nx_[1 + pos] = x;
          if (pos == m - 1) {
            nf_[0] = hor;
            nx_[0] = sub(x, GB_VS_TWO_PI);
          }
          if (pos == 0) {
            nf_[m + 1] = hor;
            nx_[m + 1] = add(x, GB_VS_TWO_PI);
          }
        }
      }
    }
    if (first) {
      has_nan = __syncthreads_or(nans) != 0;
    } else if (has_nan) {
      if (unknown) atomicAdd(&s_cnt[0], unknown);
      if (opened) atomicAdd(&s_cnt[1], opened);
      __syncthreads();
      if (s_cnt[0] == s_cnt[1]) has_nan = false;
      __syncthreads();
    } else {
      __syncthreads();
    }
    // everybody is done with the previous abscissae: this ring's take their place in shared memory (every prev_k-th of them
    // when there are more than q.cap + 2: then at most q.cap + 2 samples)
    if (LARGE && m > q.cap) {
      prev_k = (m + 2 + q.cap + 1) / (q.cap + 2);
      for (int i = tid; i <= (m + 1) / prev_k; i += nthr) xp_s[i] = __ldcg(nx_ + (int64_t)i * prev_k);
    } else {
      prev_k = 1;
      for (int i = tid; i < m + 2; i += nthr) xp_s[i] = __ldcg(nx_ + i);
    }
    __syncthreads();
    first = false;
    prev_m = m;
    cur ^= 1;
  }
}
