// glimpse_b200 — kernels and C ABI of the Tracker hot path (see include/glimpse_b200.h).
//
// The per-update kernels are in stream.cuh (one update = kernels over all points of a batch; batches of points advance
// on their own streams); this file holds the kernel parameters, the first-frame / template kernels, the stand-alone
// stage entry points and the host side of the C ABI.
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <nvjpeg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "camera.cuh"
#include "common.cuh"
#include "motion.cuh"
#include "tile.cuh"

#define GB_THREADS 512
#define GB_MAX_TEMPLATE 1024 /* template pixels a plan admits without GB_PLAN_LARGE_TEMPLATES */
#define GB_MAX_HIGHPASS 31   /* rows / columns of the median high-pass */

namespace gb {

static thread_local char g_error[512] = "";

static int fail(int code, const char* fmt, const char* detail = "") {
  snprintf(g_error, sizeof(g_error), fmt, detail);
  return code;
}
#define GB_CUDA(expr)                                                               \
  do {                                                                              \
    cudaError_t err_ = (expr);                                                      \
    if (err_ != cudaSuccess) return fail(GB_E_CUDA, #expr ": %s", cudaGetErrorString(err_)); \
  } while (0)

// ---------------------------------------------------------------------------------------------
// Kernel parameters
// ---------------------------------------------------------------------------------------------
struct StepParams {
  int64_t P, N;
  int T, O, S, t;
  int tile_w, tile_h;
  int hp_rows;                // hp_rows x hp_cols: size of the median high-pass (Tracker.highpass['size'], tracker.py:59, 530)
  int skip_evolve, viewshed, rng_mode, hp_cols;
  int hp_mode, hp_org_r, hp_org_c;  // border mode (GB_HP_*) and origin of the median high-pass
  double hp_cval;
  int hp_has_fp;
  uint32_t hp_fp[GB_MAX_HIGHPASS];  // footprint of the median high-pass, one word per window row
  uint64_t seed;
  int64_t point_offset;
  double tau, tau2;
  // Slots of time t: what a time step uses once and discards (the arrays below, the scratch regions, the grids of k_s2_surface
  // and k_template) is indexed by slot; templates, masks and outputs by observer obs[s].  A call of up to GB_MAX_OBS observers
  // has the identity table (n_slots = O, obs[s] = s); a larger one lists the observers with a frame at t in ascending order.
  int n_slots, slot_stride;  // slots in use at t; slots per point in the scratch layout (plan.n_observers)
  int obs[GB_MAX_OBS];       // observer of each slot
  int img[GB_MAX_OBS];       // global image index of each slot's observer at time t, -1 = none
  CamK cam[GB_MAX_OBS];      // that image's camera (constant bank: operands without loads)
  const uint8_t* pixels[GB_MAX_OBS];
  int pitch[GB_MAX_OBS], nchan[GB_MAX_OBS], pixdtype[GB_MAX_OBS];
  int tmpl_frame[GB_MAX_OBS]; // time index at which each slot's observer's template is cut
  double obs_scale[GB_MAX_OBS];
  const gb_image* images;
  const uint8_t* mask;
  const int32_t* first;
  const int32_t* last;
  const gb_motion* motion;
  const gb_surface* surfaces;
  const double* init_normals;
  const double* step_normals;
  const double* uniforms;
  double* state_a;
  double* state_b;
  double* weight_state;
  double* tmpl_tile;
  double* tmpl_values;
  double* tmpl_quantiles;
  int32_t* tmpl_nvalues;
  int32_t* tmpl_box;
  double* tmpl_duv;
  double* means;
  double* sigmas;
  double* covariances;
  double* out_particles;
  double* out_weights;
  int32_t* status;
  int32_t* status_time;
  uint8_t* obs_flags;
  int32_t* window_stats;
  double* final_weights;  // [N] weights of the last point's resampled particles at its last time, or NULL
  gb_stage_io io;
  // GB_MODE_STREAM buffers (carved from `scratch` by the host)
  double* s_ev;      // [P][6][N]   particles after the motion step (this time's parity)
  double* s_ev_next; // [P][6][N]   pipelined flow: particles advanced to the next time (other parity)
  double* s_ref;     // [P][6]      pipelined flow: fixed origin of the moment sums
  int* s_pflags_next; // [P]        pipelined flow: flags of the next time
  double* s_uv;      // [P][slot][2][N] projected particles
  double* s_w;       // [P][N]      weights
  double* s_bsum;    // [P][nblk]   per-CTA weight totals
  double* s_pm;      // [P][nblk][28] per-CTA moment sums
  double* s_pre;     // [P][nblk + 4] prefix of the CTA totals (0 .. total), 1 / total, uniform draw, 1 / N (written by k_s3b_publish)
  int* s_ibox;       // [P][slot][5] integer cloud box (left, top, -right, -bottom, -(any NaN))
  int* s_pflags;     // [P]         GB_F_* raised during this update
  uint8_t* s_act;    // [P]         GB_ACT_* bits of this update
  int* s_meta;       // [P][slot][8] surface meta: box[4], Mu, Mv, Mp, ok
  char* s_surf;      // [P][slot] surface regions of surf_bytes each (Hermite array first)
  int64_t surf_bytes;
  int s_block, s_nblk;
  int tmpl_from_ev;  // k_template: staggered templates read the evolved particles from s_ev (pipelined flow)
  int resample_method;  // GB_RESAMPLE_*
  int s2_budget;        // shared-memory bytes k_s2_surface may use for one window (negative: planar path forced, tests)
  int s2_smem;          // dynamic shared memory k_s2_surface is launched with (s2_smem_bytes)
  int64_t p0, pb;    // batch of points handled by this launch
  int interp_rows, interp_cols;  // spline degree along the rows (kx) / columns (ky) of the SSE surface: 3 or 1 (Tracker.interpolation)
};

// What k_s4p needs to know about the NEXT time to advance the particles to it.
struct NextParams {
  double tau, tau2;
  int spec_update;  // no point starts at this time: every active point is resampled, k_s4p may request its parents early
  int n_slots;      // the slot table of the next time (see StepParams)
  int obs[GB_MAX_OBS];
  int img[GB_MAX_OBS];
  CamK cam[GB_MAX_OBS];
};

// Tensor maps (TMA descriptors) of the frames the slots show at time t: a kernel parameter of k_s2_surface, so the
// descriptors live in the constant bank of the launch.  ok[s] = 0: that frame is read with ordinary loads.
struct alignas(64) FrameMaps {
  CUtensorMap map[GB_MAX_OBS];
  int ok[GB_MAX_OBS];
};

__device__ __forceinline__ double* state_buffer(const StepParams& prm, int t) { return (t & 1) ? prm.state_b : prm.state_a; }

__device__ __forceinline__ int status_from_flags(uint32_t f) {
  if (f & GB_F_EVOLVE_OOB) return GB_ST_DEM_BOUNDS;  // raised inside evolve_particles, before the particle tests
  if (f & GB_F_VIEW_OOB) return GB_ST_DEM_BOUNDS;
  if (f & GB_F_NOT_VISIBLE) return GB_ST_NOT_VISIBLE;
  if (f & GB_F_NAN) return GB_ST_NAN;
  if (f & GB_F_TEMPLATE) return GB_ST_TEMPLATE_BOUNDS;
  if (f & GB_F_WINDOW) return GB_ST_WINDOW_TOO_LARGE;
  if (f & GB_F_SAMPLE_OUTSIDE) return GB_ST_SAMPLE_OUTSIDE;
  if (f & GB_F_DEM_OOB) return GB_ST_DEM_BOUNDS;
  return GB_ST_OK;
}

// tracker.py:106-119 for one particle
__device__ __forceinline__ uint32_t test_particle(const StepParams& prm, const double (&s)[6]) {
  uint32_t f = 0;
  if (prm.viewshed >= 0) {
    bool oob;
    const double vis = surface_sample(prm.surfaces[prm.viewshed], s[0], s[1], 0, oob);
    if (oob) f |= GB_F_VIEW_OOB;
    else if (vis == 0.0) f |= GB_F_NOT_VISIBLE;
  }
  if (isnan(s[0]) | isnan(s[1]) | isnan(s[2]) | isnan(s[3]) | isnan(s[4]) | isnan(s[5])) f |= GB_F_NAN;
  return f;
}

// ---------------------------------------------------------------------------------------------
// Weighted moments (tracker.py:72-104).  Sums are taken of d = particle - ref so that map-scale
// coordinates do not cancel; NM = 13 (sigmas) or 28 (covariances) accumulators.
// ---------------------------------------------------------------------------------------------
template <bool COV>
struct Moments {
  static constexpr int NM = COV ? 28 : 13;
  double a[NM];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int k = 0; k < NM; ++k) a[k] = 0.0;
  }
  __device__ __forceinline__ void accumulate(double w, const double (&s)[6], const double* ref) {
    double d[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) d[k] = s[k] - ref[k];
    a[0] += w;
#pragma unroll
    for (int k = 0; k < 6; ++k) a[1 + k] = fma(w, d[k], a[1 + k]);
    if (COV) {
      int idx = 7;
#pragma unroll
      for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int l = k; l < 6; ++l) a[idx++] = fma(w * d[k], d[l], a[idx]);
    } else {
#pragma unroll
      for (int k = 0; k < 6; ++k) a[7 + k] = fma(w * d[k], d[k], a[7 + k]);
    }
  }
};

// Finalise from the summed accumulators `a` (NM doubles): mean[6], sigma[6] or cov[36].
template <bool COV>
__device__ inline void finalize_moments(const double* a, const double* ref, double* mean, double* sigma, double* cov) {
  const double inv = 1.0 / a[0];
  double m1[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    m1[k] = a[1 + k] * inv;
    mean[k] = ref[k] + m1[k];
  }
  if (COV) {
    int idx = 7;
    for (int k = 0; k < 6; ++k)
      for (int l = k; l < 6; ++l) {
        const double c = a[idx++] * inv - m1[k] * m1[l];
        cov[k * 6 + l] = c;
        cov[l * 6 + k] = c;
      }
  } else {
    for (int k = 0; k < 6; ++k) sigma[k] = sqrt(fmax(a[7 + k] * inv - m1[k] * m1[k], 0.0));
  }
}

// ---------------------------------------------------------------------------------------------
// Small stand-alone kernels
// ---------------------------------------------------------------------------------------------
__global__ void k_project(const __grid_constant__ gb_camera cam, const double* __restrict__ xyz, int64_t n,
                          double* __restrict__ uv) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double u, v;
    project(cam, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], u, v);
    uv[2 * i] = u;
    uv[2 * i + 1] = v;
  }
}

__global__ void k_unproject(const __grid_constant__ gb_camera cam, const double* __restrict__ uv, int64_t n,
                            int directions, const double* __restrict__ depth, double* __restrict__ xyz) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double dx, dy, dz;
    unproject(cam, uv[2 * i], uv[2 * i + 1], dx, dy, dz);
    if (depth) {
      const double d = depth[i];
      dx = mul(dx, d);
      dy = mul(dy, d);
      dz = mul(dz, d);
    }
    if (!directions) {
      dx = add(dx, cam.xyz[0]);
      dy = add(dy, cam.xyz[1]);
      dz = add(dz, cam.xyz[2]);
    }
    xyz[3 * i] = dx;
    xyz[3 * i + 1] = dy;
    xyz[3 * i + 2] = dz;
  }
}

// Image.project (image.py:301-361): one thread per pixel of the target camera.  The pixel centre is cast out through the
// target camera, projected into the source camera as a direction, and every band of the source frame is sampled there the
// way scipy.interpolate.RegularGridInterpolator does on the pixel-centre grid (bounds_error=False: NaN outside, which an
// integer frame stores as 0).  Arithmetic per band type as restated in oracle/tracker_oracle.py::project_image.
__device__ __forceinline__ double band_value(const uint8_t* pixels, int64_t pitch, int nchan, int dtype, int row, int col, int ch) {
  const uint8_t* base = pixels + (int64_t)row * pitch;
  const int64_t e = (int64_t)col * nchan + ch;
  switch (dtype) {
    case GB_PIX_U16: return (double)reinterpret_cast<const uint16_t*>(base)[e];
    case GB_PIX_F32: return (double)reinterpret_cast<const float*>(base)[e];
    case GB_PIX_F64: return reinterpret_cast<const double*>(base)[e];
    default: return (double)base[e];
  }
}

__device__ __forceinline__ void grid_interval(double x, int n, int& i, double& y) {
  double f = floor(x - 0.5);
  if (!(f >= 0.0)) f = 0.0;  // (NaN too: the distance below stays NaN)
  i = (int)fmin(f, (double)(n - 2));
  y = sub(x, (double)i + 0.5);
}

__global__ void k_project_image(const __grid_constant__ gb_image src, const __grid_constant__ gb_camera dst, int method,
                                uint8_t* __restrict__ out) {
  const int W = dst.imgsz[0], H = dst.imgsz[1], C = src.nchan, sw = src.width, sh = src.height;
  const int64_t total = (int64_t)W * H;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(i / W), col = (int)(i - (int64_t)row * W);
    double dx, dy, dz, pu, pv;
    unproject(dst, (double)col + 0.5, (double)row + 0.5, dx, dy, dz);
    project_direction(src.cam, dx, dy, dz, pu, pv);
    const bool nan = isnan(pu) || isnan(pv);
    const bool outside = pv < 0.5 || pv > (double)sh - 0.5 || pu < 0.5 || pu > (double)sw - 0.5;
    int i0 = 0, i1 = 0;
    double y0 = 0.0, y1 = 0.0;
    if (!nan && !outside) {
      grid_interval(pv, sh, i0, y0);
      grid_interval(pu, sw, i1, y1);
    }
    for (int ch = 0; ch < C; ++ch) {
      double val = CUDART_NAN;
      if (!nan && !outside) {
        if (method == 0) {
          val = band_value(src.pixels, src.pitch, C, src.dtype, y0 <= 0.5 ? i0 : i0 + 1, y1 <= 0.5 ? i1 : i1 + 1, ch);
        } else {
          const double v00 = band_value(src.pixels, src.pitch, C, src.dtype, i0, i1, ch);
          const double v01 = band_value(src.pixels, src.pitch, C, src.dtype, i0, i1 + 1, ch);
          const double v10 = band_value(src.pixels, src.pitch, C, src.dtype, i0 + 1, i1, ch);
          const double v11 = band_value(src.pixels, src.pitch, C, src.dtype, i0 + 1, i1 + 1, ch);
          const double a0 = sub(1.0, y0), a1 = sub(1.0, y1);
          if (src.dtype == GB_PIX_F32) {  // generic form: value * (wy * wx), summed in corner order
            val = mul(v00, mul(a0, a1));
            val = add(val, mul(v01, mul(a0, y1)));
            val = add(val, mul(v10, mul(y0, a1)));
            val = add(val, mul(v11, mul(y0, y1)));
          } else {  // integer and float64 bands: v * wy * wx, left to right
            val = mul(mul(v00, a0), a1);
            val = add(val, mul(mul(v01, a0), y1));
            val = add(val, mul(mul(v10, y0), a1));
            val = add(val, mul(mul(v11, y0), y1));
          }
        }
      }
      const int64_t e = i * C + ch;
      switch (src.dtype) {
        case GB_PIX_U16: reinterpret_cast<uint16_t*>(out)[e] = isnan(val) ? (uint16_t)0 : (uint16_t)(int)val; break;
        case GB_PIX_F32: reinterpret_cast<float*>(out)[e] = (float)val; break;
        case GB_PIX_F64: reinterpret_cast<double*>(out)[e] = val; break;
        default: out[e] = isnan(val) ? (uint8_t)0 : (uint8_t)(int)val; break;
      }
    }
  }
}

__global__ void k_state_from_rows(const double* __restrict__ rows, int64_t npoints, int64_t n, double* __restrict__ state) {
  const int64_t total = npoints * n;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / n, j = i - p * n;
#pragma unroll
    for (int c = 0; c < 6; ++c) state[(p * 6 + c) * n + j] = rows[i * 6 + c];
  }
}

__global__ void k_state_to_rows(const double* __restrict__ state, int64_t npoints, int64_t n, double* __restrict__ rows) {
  const int64_t total = npoints * n;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / n, j = i - p * n;
#pragma unroll
    for (int c = 0; c < 6; ++c) rows[i * 6 + c] = state[(p * 6 + c) * n + j];
  }
}

// Motion.evolve_particles on SoA state with supplied normals (stage entry point + staggered
// template path of gb_track, where t/first/last select the points that step at time t).
__global__ void k_evolve(const gb_motion* __restrict__ motion, const gb_surface* __restrict__ surfaces, int64_t P, int64_t N,
                         double tau, double tau2, const double* __restrict__ normals, int64_t normals_point_stride,
                         double* __restrict__ state, const int32_t* first, const int32_t* last, int32_t* status, int32_t* status_time,
                         int t, int rng_mode, uint64_t seed, int S, int64_t point_offset) {
  const int64_t p = blockIdx.y;
  if (first && (status[p] != 0 || t <= first[p] || t > last[p])) return;
  const gb_motion m = motion[p];
  const double* zn = normals ? normals + p * normals_point_stride + (first ? (int64_t)(t - first[p] - 1) * N * 3 : 0) : nullptr;
  (void)S;
  uint32_t flags = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    double s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) s[c] = state[(p * 6 + c) * N + i];
    double z0, z1, z2;
    if (rng_mode == GB_RNG_SUPPLIED) {
      z0 = zn[3 * i];
      z1 = zn[3 * i + 1];
      z2 = zn[3 * i + 2];
    } else {
      philox_normals3(seed, (uint64_t)(p + point_offset), (uint32_t)t, (uint32_t)i, 2u, z0, z1, z2);
    }
    evolve_particle(m, surfaces, tau, tau2, z0, z1, z2, s, flags);
#pragma unroll
    for (int c = 0; c < 6; ++c) state[(p * 6 + c) * N + i] = s[c];
  }
  // (stand-alone call: the failure is reported after the fact; inside gb_track_step the step kernels see the status)
  if (flags && status) {
    atomicCAS(&status[p], 0, GB_ST_DEM_BOUNDS);
    if (status_time) status_time[p] = t;
  }
}

// Tracker.particle_mean / sigma / covariance for one row-major particle set (stage entry point).
__global__ void __launch_bounds__(GB_THREADS) k_moments(const double* __restrict__ particles,
                                                        const double* __restrict__ weights, int64_t n, double* mean,
                                                        double* sigma, double* cov) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemHeader* hdr = reinterpret_cast<SmemHeader*>(smem_raw);
  double ref[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) ref[c] = particles[c];
  Moments<true> mom;
  mom.clear();
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    double s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) s[c] = particles[i * 6 + c];
    mom.accumulate(weights[i], s, ref);
  }
  block_reduce<28, 0>(mom.a, hdr);
  if (threadIdx.x == 0) {
    double m[6], cv[36];
    finalize_moments<true>(hdr->bcast, ref, m, nullptr, cv);
    for (int c = 0; c < 6; ++c) {
      mean[c] = m[c];
      if (sigma) sigma[c] = sqrt(fmax(cv[c * 7], 0.0));
    }
    if (cov)
      for (int c = 0; c < 36; ++c) cov[c] = cv[c];
  }
}

// The device draws of gb_track's philox mode, read back through the very functions the step kernels call (stand-alone
// entry point gb_philox_draws; element i is particle first + i, or time `time + i` for the systematic uniform).
__global__ void k_philox_draws(uint64_t seed, uint64_t point, uint32_t time, uint32_t first, int64_t n, int kind, uint32_t rng_stream,
                               void* out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t particle = first + (uint32_t)i;
    if (kind == GB_DRAW_WORDS) {
      uint32_t r[4];
      Philox{(uint32_t)seed, (uint32_t)(seed >> 32)}.generate(particle, time, (uint32_t)point,
                                                             ((uint32_t)(point >> 32) << 8) | rng_stream, r);
      uint32_t* dst = static_cast<uint32_t*>(out) + 4 * i;
#pragma unroll
      for (int c = 0; c < 4; ++c) dst[c] = r[c];
    } else if (kind == GB_DRAW_NORMALS) {
      double* dst = static_cast<double*>(out) + 3 * i;
      philox_normals3(seed, point, time, particle, rng_stream, dst[0], dst[1], dst[2]);
    } else if (kind == GB_DRAW_UNIFORM) {
      static_cast<double*>(out)[i] = philox_uniform(seed, point, time + (uint32_t)i);
    } else {
      static_cast<double*>(out)[i] = philox_uniform_particle(seed, point, time, particle);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// First frame: initialize_particles + test_particles + unit weights + moments
// (motion.py:149-163, 260-283; tracker.py:327-330, 350-357).  One CTA per point.
// ---------------------------------------------------------------------------------------------
template <bool COV>
__global__ void __launch_bounds__(GB_THREADS) k_init(const __grid_constant__ StepParams prm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemHeader* hdr = reinterpret_cast<SmemHeader*>(smem_raw);
  const int64_t p = blockIdx.x;
  const int t = prm.t;
  if (prm.status[p] != 0 || prm.first[p] != t || prm.last[p] < t) return;
  const int64_t N = prm.N;
  const gb_motion m = prm.motion[p];
  double* state = state_buffer(prm, t) + p * 6 * N;
  bool oob0, oob1;
  double ref[6] = {m.xy[0], m.xy[1], surface_sample(prm.surfaces[m.dem], m.xy[0], m.xy[1], 1, oob0), 0.0, 0.0, 0.0};
  (void)oob1;
  if (isnan(ref[2])) ref[2] = 0.0;
  if (m.kind == GB_MOTION_CYLINDRICAL) {
    ref[3] = m.v[0] * cos(m.v[1]);
    ref[4] = m.v[0] * sin(m.v[1]);
  } else {
    ref[3] = m.v[0];
    ref[4] = m.v[1];
  }
  ref[5] = m.v[2];
  if (prm.s_ref && threadIdx.x < 6) prm.s_ref[p * 6 + threadIdx.x] = ref[threadIdx.x];
  Moments<COV> mom;
  mom.clear();
  uint32_t flags = 0;
  for (int64_t i = threadIdx.x; i < N; i += blockDim.x) {
    double zn[6];
    if (prm.rng_mode == GB_RNG_SUPPLIED) {
      const double* src = prm.init_normals + (p * N + i) * 6;
#pragma unroll
      for (int c = 0; c < 6; ++c) zn[c] = src[c];
    } else {
      philox_normals3(prm.seed, (uint64_t)(p + prm.point_offset), (uint32_t)t, (uint32_t)i, 0u, zn[0], zn[1], zn[2]);
      philox_normals3(prm.seed, (uint64_t)(p + prm.point_offset), (uint32_t)t, (uint32_t)i, 1u, zn[3], zn[4], zn[5]);
    }
    double s[6];
    init_particle(m, prm.surfaces, zn, s, flags);
    flags |= test_particle(prm, s);
#pragma unroll
    for (int c = 0; c < 6; ++c) state[c * N + i] = s[c];
    if (prm.weight_state) prm.weight_state[p * N + i] = 1.0;
    if (prm.out_particles) {
      double* dst = prm.out_particles + ((p * prm.T + t) * N + i) * 6;
#pragma unroll
      for (int c = 0; c < 6; ++c) dst[c] = s[c];
    }
    if (prm.out_weights) prm.out_weights[(p * prm.T + t) * N + i] = 1.0;
    mom.accumulate(1.0, s, ref);
  }
  const int any = (int)block_or(flags, reinterpret_cast<unsigned*>(&hdr->iflags[1]));
  if (any) {
    if (threadIdx.x == 0) {
      prm.status[p] = status_from_flags((uint32_t)any);
      prm.status_time[p] = t;
    }
    return;
  }
  block_reduce<Moments<COV>::NM, 0>(mom.a, hdr);
  if (threadIdx.x == 0) {
    double mean[6], sg[6], cv[36];
    finalize_moments<COV>(hdr->bcast, ref, mean, sg, cv);
    double* mo = prm.means + (p * prm.T + t) * 6;
    for (int c = 0; c < 6; ++c) mo[c] = mean[c];
    if (COV) {
      double* co = prm.covariances + (p * prm.T + t) * 36;
      for (int c = 0; c < 36; ++c) co[c] = cv[c];
    } else {
      double* so = prm.sigmas + (p * prm.T + t) * 6;
      for (int c = 0; c < 6; ++c) so[c] = sg[c];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Template construction (tracker.py:536-561, 494-534): one CTA per (point, slot) of time t; the template of the slot's
// observer is cut when t is its template frame.
// LARGE: templates above GB_SMEM_TEMPLATE pixels (GB_PLAN_LARGE_TEMPLATES).  Their levels, histogram and representatives
// live in dynamic shared memory (template_smem_bytes), the grey values of ranked frames in the (point, slot)'s surface
// region, which no kernel uses while templates are cut.  Otherwise the two variants run the same code.
// ---------------------------------------------------------------------------------------------
// histogram bins: one per rank of a ranked template, one per band sum of a uint8 frame of up to 8 bands
__host__ __device__ inline int template_bins(int area) { return area > GB_MAX_U8_BINS ? area : GB_MAX_U8_BINS; }
__host__ __device__ inline int template_smem_bytes(int area) {
  return (int)(align16((int64_t)template_bins(area) * 4) + 2 * align16((int64_t)area * 2));
}

template <bool LARGE>
__global__ void __launch_bounds__(256) k_template(const __grid_constant__ StepParams prm) {
  __shared__ double s_red[8][8];
  __shared__ int s_box[4];
  __shared__ int s_ok;
  __shared__ double s_stats[2];
  const int64_t p = blockIdx.x / prm.n_slots;
  const int slot = (int)(blockIdx.x - p * prm.n_slots), o = prm.obs[slot];
  const int64_t po = p * prm.O + o;
  uint16_t* s_raw;   // grey level of every pixel
  uint32_t* s_hist;  // pixels per level
  double* s_vals;    // frames other than uint8: the tile's grey values ...
  uint16_t* s_rep;   // ... and one pixel of every level
  if constexpr (LARGE) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int a = prm.tile_w * prm.tile_h;
    s_hist = reinterpret_cast<uint32_t*>(smem_raw);
    s_raw = reinterpret_cast<uint16_t*>(smem_raw + align16((int64_t)template_bins(a) * 4));
    s_rep = reinterpret_cast<uint16_t*>(smem_raw + align16((int64_t)template_bins(a) * 4) + align16((int64_t)a * 2));
    s_vals = reinterpret_cast<double*>(prm.s_surf + (p * prm.slot_stride + slot) * prm.surf_bytes);
  } else {
    __shared__ uint16_t a_raw[GB_SMEM_TEMPLATE];
    __shared__ uint32_t a_hist[GB_MAX_U8_BINS];
    __shared__ double a_vals[GB_SMEM_TEMPLATE];
    __shared__ uint16_t a_rep[GB_SMEM_TEMPLATE];
    s_raw = a_raw;
    s_hist = a_hist;
    s_vals = a_vals;
    s_rep = a_rep;
  }
  const int t = prm.t;
  if (prm.status[p] != 0 || prm.tmpl_frame[slot] != t || !prm.mask[po] || prm.img[slot] < 0) return;
  if (t < prm.first[p] || t > prm.last[p]) return;
  const int64_t N = prm.N;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // particles as they are when the template is cut: just initialised (t == first) or evolved in place
  const double* state = prm.first[p] == t ? state_buffer(prm, t) + p * 6 * N
                        : (prm.tmpl_from_ev ? prm.s_ev + p * 6 * N : state_buffer(prm, t - 1) + p * 6 * N);
  const double* wts = prm.weight_state ? prm.weight_state + p * N : nullptr;
  const double ref[3] = {state[0], state[N], state[2 * N]};
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int64_t i = tid; i < N; i += blockDim.x) {
    const double w = wts ? wts[i] : 1.0;
    acc[0] += w;
    acc[1] = fma(w, state[i] - ref[0], acc[1]);
    acc[2] = fma(w, state[N + i] - ref[1], acc[2]);
    acc[3] = fma(w, state[2 * N + i] - ref[2], acc[3]);
  }
  for (int k = 0; k < 4; ++k) {
    const double x = warp_sum(acc[k]);
    if (lane == 0) s_red[warp][k] = x;
  }
  __syncthreads();
  const gb_image* img = prm.images + prm.img[slot];
  const int tw = prm.tile_w, th = prm.tile_h;
  if (tid == 0) {
    double tot[4] = {0, 0, 0, 0};
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w)
      for (int k = 0; k < 4; ++k) tot[k] += s_red[w][k];
    const double mx = ref[0] + tot[1] / tot[0], my = ref[1] + tot[2] / tot[0], mz = ref[2] + tot[3] / tot[0];
    double u, v;
    project(img->cam, mx, my, mz, u, v);
    // Observer.tile_box -> Grid.snap_box (observer.py:115-130, raster.py:390-421)
    const double hw = tw * 0.5, hh = th * 0.5;
    const double l = sub(u, hw), tp = sub(v, hh), r = add(u, hw), b = add(v, hh);
    const double W = (double)img->cam.imgsz[0], H = (double)img->cam.imgsz[1];
    const bool ok = (l >= 0.0) & (l <= W) & (r >= 0.0) & (r <= W) & (tp >= 0.0) & (tp <= H) & (b >= 0.0) & (b <= H);
    s_ok = ok ? 1 : 0;
    if (ok) {
      s_box[0] = (int)floor(l + 0.5);
      s_box[1] = (int)floor(tp + 0.5);
      s_box[2] = (int)floor(r + 0.5);
      s_box[3] = (int)floor(b + 0.5);
      int32_t* gbox = prm.tmpl_box + po * 4;
      for (int k = 0; k < 4; ++k) gbox[k] = s_box[k];
      double* duv = prm.tmpl_duv + po * 2;
      duv[0] = sub(u, (double)(s_box[0] + s_box[2]) / 2.0);
      duv[1] = sub(v, (double)(s_box[1] + s_box[3]) / 2.0);
    } else {
      if (atomicCAS(&prm.status[p], 0, GB_ST_TEMPLATE_BOUNDS) == 0) prm.status_time[p] = t;
      // the reference raises inside initialize_template, before the moments of this time are stored (tracker.py:336-354)
      double* mo = prm.means + (p * prm.T + t) * 6;
      for (int c = 0; c < 6; ++c) mo[c] = CUDART_NAN;
      if (prm.sigmas) for (int c = 0; c < 6; ++c) prm.sigmas[(p * prm.T + t) * 6 + c] = CUDART_NAN;
      if (prm.covariances) for (int c = 0; c < 36; ++c) prm.covariances[(p * prm.T + t) * 36 + c] = CUDART_NAN;
    }
  }
  __syncthreads();
  if (!s_ok) return;
  // the snapped box always spans tile_w x tile_h pixels for integer sizes
  const int bw = s_box[2] - s_box[0], bh = s_box[3] - s_box[1];
  const int area = bw * bh;
  const int nchan = img->nchan;
  // uint8 frames: grey levels are the band sums (value = level / bands).  Other types: the tile's grey values are kept and every
  // pixel's level is the number of tile pixels below it (same order, equal values share a level), one representative per level.
  const bool ranked = img->dtype != GB_PIX_U8;
  const int nbins = ranked ? area : 255 * nchan + 1;
  for (int i = tid; i < nbins; i += blockDim.x) s_hist[i] = 0u;
  for (int i = tid; i < area; i += blockDim.x) {
    const int r = i / bw, c = i - r * bw;
    // a box snapped onto the frame edge can reach one pixel outside only through rounding; clamp
    const int rr = min(max(s_box[1] + r, 0), img->height - 1), cc = min(max(s_box[0] + c, 0), img->width - 1);
    if (ranked) {
      s_vals[i] = pixel_gray(img->pixels, img->pitch, nchan, img->dtype, rr, cc);
    } else {
      const uint8_t* px = img->pixels + (int64_t)rr * img->pitch + (int64_t)cc * img->nchan;
      unsigned sum = 0;
      for (int k = 0; k < img->nchan; ++k) sum += px[k];
      s_raw[i] = (uint16_t)sum;
    }
  }
  __syncthreads();
  if (ranked) {
    for (int i = tid; i < area; i += blockDim.x) {
      const double v = s_vals[i];
      int below = 0;
      for (int j = 0; j < area; ++j) below += s_vals[j] < v;
      s_raw[i] = (uint16_t)below;
      s_rep[below] = (uint16_t)i;  // (any pixel of the level: they hold the same value)
    }
    __syncthreads();
  }
  auto gray_of = [&](int i) { return ranked ? s_vals[i] : quo((double)s_raw[i], (double)nchan); };
  auto level_value = [&](int b) { return ranked ? s_vals[s_rep[b]] : quo((double)b, (double)nchan); };
  // grey mean and population std (helpers.py:324-344)
  double sum = 0.0;
  for (int i = tid; i < area; i += blockDim.x) {
    sum += gray_of(i);
    atomicAdd(&s_hist[s_raw[i]], 1u);
  }
  sum = warp_sum(sum);
  if (lane == 0) s_red[warp][0] = sum;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_red[w][0];
    s_stats[0] = quo(tot, (double)area);
  }
  __syncthreads();
  const double mean = s_stats[0];
  double ss = 0.0;
  for (int i = tid; i < area; i += blockDim.x) {
    const double d = sub(gray_of(i), mean);
    ss += mul(d, d);
  }
  ss = warp_sum(ss);
  if (lane == 0) s_red[warp][1] = ss;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_red[w][1];
    s_stats[1] = quo(1.0, sqrt(quo(tot, (double)area)));
  }
  __syncthreads();
  const double inv_std = s_stats[1];
  // CDF over occupied grey levels (helpers.py:433-464): levels are visited in increasing order, and
  // the normalised value is an increasing function of the level, so this is np.unique's order.
  if (tid == 0) {
    double* vals = prm.tmpl_values + po * (int64_t)(tw * th);
    double* qs = prm.tmpl_quantiles + po * (int64_t)(tw * th);
    int n = 0;
    uint32_t run = 0;
    for (int b = 0; b < nbins; ++b) {
      if (!s_hist[b]) continue;
      run += s_hist[b];
      vals[n] = mul(sub(level_value(b), mean), inv_std);
      qs[n] = quo((double)run, (double)area);
      ++n;
    }
    prm.tmpl_nvalues[po] = n;
  }
  // high-pass (tracker.py:530-531): value minus the reflected median (5x5 unless Tracker.highpass says otherwise), taken
  // on grey levels
  double* tile = prm.tmpl_tile + po * (int64_t)(tw * th);
  const bool hp_plain = prm.hp_mode == GB_HP_REFLECT && prm.hp_org_r == 0 && prm.hp_org_c == 0 && !prm.hp_has_fp;
  const bool hp5 = prm.hp_rows == 5 && prm.hp_cols == 5 && hp_plain;
  // (general border mode: the constant beyond the border takes its place among the grey levels through the normalised values)
  int cval_level = nbins;
  if (!hp_plain)
    for (int b = nbins - 1; b >= 0; --b)
      if ((!ranked || s_hist[b]) && !(mul(sub(level_value(b), mean), inv_std) < prm.hp_cval)) cval_level = b;
  for (int i = tid; i < area; i += blockDim.x) {
    const int r = i / bw, c = i - r * bw;
    const double vn = mul(sub(gray_of(i), mean), inv_std);
    double vm;
    if (hp_plain) {
      const int med = hp5 ? median5x5(s_raw, bw, bh, r, c) : median_window(s_raw, bw, bh, r, c, prm.hp_rows, prm.hp_cols, nbins);
      vm = mul(sub(level_value(med), mean), inv_std);
    } else {
      const int code = median_window_codes(s_raw, bw, bh, r, c, prm.hp_rows, prm.hp_cols, prm.hp_mode, prm.hp_org_r, prm.hp_org_c,
                                           2 * cval_level, prm.hp_has_fp ? prm.hp_fp : nullptr, nbins);
      vm = (code & 1) ? mul(sub(level_value(code >> 1), mean), inv_std) : prm.hp_cval;
    }
    tile[i] = sub(vn, vm);
  }
}

// ---------------------------------------------------------------------------------------------
// Resampling positions (tracker.py:168-186), shared by the kernels of stream.cuh
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double resample_position(int j, double u, double inv_n) {
  // (np.arange(n) + u) * (1 / n)  (tracker.py:173)
  return mul(add((double)j, u), inv_n);
}

// Number of resampling positions <= c, i.e. the end of the child range of a particle whose
// normalised cumulative weight is c (np.searchsorted(cumsum, positions, side='left')).  The guess
// from c * N - u is verified against the reference's own position formula and walked if needed.
__device__ __forceinline__ int count_positions_le(double c, double u, double inv_n, int N) {
  int e = __double2int_rd(c * (double)N - u) + 1;
  e = min(max(e, 0), N);
  const bool ok = (e == 0 || resample_position(e - 1, u, inv_n) <= c) && (e == N || resample_position(e, u, inv_n) > c);
  if (!ok) {
    while (e > 0 && resample_position(e - 1, u, inv_n) > c) --e;
    while (e < N && resample_position(e, u, inv_n) <= c) ++e;
  }
  return e;
}

// Stratified resampling (tracker.py:178-186): position j = (j + u_j) / N with one uniform per particle, taken from
// the supplied draws or from Philox.  Positions still increase with j, so a parent's child range ends at the number
// of positions <= its normalised cumulative weight: j < floor(c N) always qualify, the stratum containing c decides
// with its own uniform; the guess is verified against the reference's position formula like the systematic one.
struct StratifiedDraws {
  const double* supplied;  // [N] uniforms of this (point, update), or nullptr: Philox
  uint64_t seed, point;
  uint32_t time;
  __device__ __forceinline__ double u(int j) const {
    return supplied ? supplied[j] : philox_uniform_particle(seed, point, time, (uint32_t)j);
  }
};
__device__ __noinline__ int count_positions_le_stratified(double c, StratifiedDraws d, double inv_n, int N) {
  int e = __double2int_rd(c * (double)N);
  e = min(max(e, 0), N);
  while (e > 0 && resample_position(e - 1, d.u(e - 1), inv_n) > c) --e;
  while (e < N && resample_position(e, d.u(e), inv_n) <= c) ++e;
  return e;
}
__device__ __forceinline__ StratifiedDraws stratified_draws(const StepParams& prm, int64_t p, int t) {
  StratifiedDraws d;
  d.supplied = prm.rng_mode == GB_RNG_SUPPLIED ? prm.uniforms + ((int64_t)p * prm.S + (t - prm.first[p] - 1)) * prm.N : nullptr;
  d.seed = prm.seed;
  d.point = (uint64_t)(p + prm.point_offset);
  d.time = (uint32_t)t;
  return d;
}

__device__ __forceinline__ double warp_inclusive_scan(double v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const double o = shfl_up(v, d);
    if (lane >= d) v += o;
  }
  return v;
}

#include "stream.cuh"
#include "viewshed.cuh"

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
static int grid_for(int64_t n, int threads) {
  int64_t g = (n + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > 148 * 16) g = 148 * 16;
  return (int)g;
}

static constexpr int kMaxSlots = 8;   // side streams / scratch slots of GB_MODE_STREAM
static constexpr int kMaxSmem = 232448;  // 227 KB opt-in dynamic shared memory per CTA on sm_100
static constexpr int kHeaderBytes = (int)((sizeof(SmemHeader) + 15) / 16 * 16);

// ---------------------------------------------------------------------------------------------
// Tensor maps of the frames (TMA): one CUtensorMap per image of the current descriptor, kept in a per-device table in
// global memory.  A frame qualifies when its base and pitch are multiples of 16 bytes; the box is GB_TMA_BOXW bytes x
// GB_TMA_BOXH rows of uint8.  cuTensorMapEncodeTiled is looked up at run time (no link-time dependency on the driver, so
// the library still loads on a machine without one).
// ---------------------------------------------------------------------------------------------
struct TensorMapTable {
  std::vector<CUtensorMap> host;
  std::vector<gb_image> seen;   // what each entry was encoded from
  std::vector<uint8_t> ok;
};
static thread_local TensorMapTable g_tmaps;
static thread_local bool g_tmaps_on = false;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    cudaGetLastError();
  });
  return fn;
}

// Encode (or reuse) the maps of the images the descriptor references; GB_TMA=0 switches the TMA path off (A/B runs).
static int ensure_tensor_maps(const gb_track_desc& d) {
  TensorMapTable& tb = g_tmaps;
  g_tmaps_on = false;
  const char* env = getenv("GB_TMA");
  EncodeTiledFn encode = (env && !strcmp(env, "0")) ? nullptr : encode_tiled_fn();
  if (!encode || !d.images_host) return GB_OK;
  int n_images = 0;
  for (int64_t k = 0; k < (int64_t)d.T * d.O; ++k) {
    const int o = (int)(k % d.O), idx = d.image_index_host[k];
    if (idx >= 0 && d.image_offset_host[o] + idx + 1 > n_images) n_images = d.image_offset_host[o] + idx + 1;
  }
  if ((size_t)n_images > tb.host.size()) {
    const size_t old = tb.host.size();
    tb.host.resize(n_images);
    tb.seen.resize(n_images);
    tb.ok.resize(n_images, 0);
    for (size_t k = old; k < (size_t)n_images; ++k) memset(&tb.seen[k], 0, sizeof(gb_image));
  }
  for (int k = 0; k < n_images; ++k) {
    const gb_image& im = d.images_host[k];
    if (tb.seen[k].pixels == im.pixels && tb.seen[k].width == im.width && tb.seen[k].height == im.height && tb.seen[k].pitch == im.pitch &&
        tb.seen[k].nchan == im.nchan && tb.seen[k].dtype == im.dtype)
      continue;
    tb.seen[k] = im;
    tb.ok[k] = 0;
    if (!im.pixels || im.dtype != GB_PIX_U8 || (reinterpret_cast<uintptr_t>(im.pixels) & 15) || (im.pitch & 15) || im.width <= 0 || im.height <= 0)
      continue;
    const cuuint64_t dims[2] = {(cuuint64_t)im.width * (cuuint64_t)im.nchan, (cuuint64_t)im.height};
    const cuuint64_t strides[1] = {(cuuint64_t)im.pitch};
    const cuuint32_t box[2] = {GB_TMA_BOXW, GB_TMA_BOXH}, estr[2] = {1, 1};
    if (encode(&tb.host[k], CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(im.pixels), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
      tb.ok[k] = 1;
  }
  g_tmaps_on = true;
  return GB_OK;
}

// The maps of the frames of time prm.t, as k_s2_surface's kernel parameter.
static void frame_maps(const StepParams& prm, FrameMaps& fm) {
  memset(&fm, 0, sizeof(fm));
  if (!g_tmaps_on) return;
  for (int s = 0; s < prm.n_slots; ++s) {
    const int image = prm.img[s];
    if (image >= 0 && (size_t)image < g_tmaps.ok.size() && g_tmaps.ok[image]) {
      fm.map[s] = g_tmaps.host[image];
      fm.ok[s] = 1;
    }
  }
}

// Time index at which observer o's template is cut: its first frame (-1: none).
static int template_frame(const gb_track_desc& d, int o) {
  for (int t = 0; t < d.T; ++t)
    if (d.image_index_host[(int64_t)t * d.O + o] >= 0) return t;
  return -1;
}

// Most observers with a frame at one time (image_index_host >= 0).
static int max_active_observers(const gb_track_desc& d) {
  int most = 0;
  for (int t = 0; t < d.T; ++t) {
    int n = 0;
    for (int o = 0; o < d.O; ++o) n += d.image_index_host[(int64_t)t * d.O + o] >= 0;
    if (n > most) most = n;
  }
  return most;
}

static void fill_params(const gb_track_desc& d, int t, StepParams& prm) {
  memset(&prm, 0, sizeof(prm));
  prm.P = d.P;
  prm.N = d.N;
  prm.T = d.T;
  prm.O = d.O;
  prm.S = d.T - 1;
  prm.t = t;
  prm.tile_w = d.tile_w;
  prm.tile_h = d.tile_h;
  prm.interp_rows = d.interp_rows ? d.interp_rows : 3;
  prm.interp_cols = d.interp_cols ? d.interp_cols : 3;
  prm.hp_rows = d.highpass_size ? (d.highpass_size & 0xffff) : 5;
  prm.hp_cols = d.highpass_size ? (d.highpass_size >> 16 & 0xffff) : 5;
  prm.hp_mode = d.highpass_mode;
  prm.hp_org_r = (int16_t)(d.highpass_origin & 0xffff);
  prm.hp_org_c = (int16_t)(d.highpass_origin >> 16 & 0xffff);
  prm.hp_cval = d.highpass_cval;
  prm.hp_has_fp = d.highpass_footprint_host != nullptr;
  if (prm.hp_has_fp)
    for (int a = 0; a < GB_MAX_HIGHPASS; ++a) prm.hp_fp[a] = a < prm.hp_rows ? d.highpass_footprint_host[a] : 0u;
  prm.viewshed = d.viewshed;
  prm.rng_mode = d.rng_mode;
  prm.seed = d.seed;
  prm.point_offset = d.point_offset;
  if (t > 0) {
    prm.tau = d.tau_host[t - 1];
    prm.tau2 = d.tau2_host[t - 1];
  }
  // the slot table (check_desc has bounded the observers with a frame at t by the plan's slots)
  prm.slot_stride = d.plan.n_observers;
  int n = 0;
  for (int o = 0; o < d.O; ++o) {
    const int idx = d.image_index_host[(int64_t)t * d.O + o];
    if (d.O > GB_MAX_OBS && idx < 0) continue;
    const int s = n++;
    prm.obs[s] = o;
    prm.img[s] = idx >= 0 ? d.image_offset_host[o] + idx : -1;
    if (idx >= 0 && d.images_host) {
      const gb_image& im = d.images_host[prm.img[s]];
      camk_from(im.cam, prm.cam[s]);
      prm.pixels[s] = im.pixels;
      prm.pitch[s] = im.pitch;
      prm.nchan[s] = im.nchan;
      prm.pixdtype[s] = im.dtype;
    }
    prm.obs_scale[s] = d.obs_scale_host[o];
    prm.tmpl_frame[s] = template_frame(d, o);
  }
  if (n == 0) {  // no frame at t: one empty slot keeps the grids non-empty (it flags its observer GB_OBS_NO_IMAGE, as it has no frame)
    prm.obs[0] = 0;
    prm.img[0] = -1;
    prm.tmpl_frame[0] = -1;
    n = 1;
  }
  prm.n_slots = n;
  prm.images = d.images;
  prm.mask = d.mask;
  prm.first = d.first;
  prm.last = d.last;
  prm.motion = d.motion;
  prm.surfaces = d.surfaces;
  prm.init_normals = d.init_normals;
  prm.step_normals = d.step_normals;
  prm.uniforms = d.uniforms;
  prm.resample_method = d.resample_method;
  prm.state_a = d.state_a;
  prm.state_b = d.state_b;
  prm.weight_state = d.weight_state;
  prm.tmpl_tile = d.tmpl_tile;
  prm.tmpl_values = d.tmpl_values;
  prm.tmpl_quantiles = d.tmpl_quantiles;
  prm.tmpl_nvalues = d.tmpl_nvalues;
  prm.tmpl_box = d.tmpl_box;
  prm.tmpl_duv = d.tmpl_duv;
  prm.means = d.means;
  prm.sigmas = d.sigmas;
  prm.covariances = d.covariances;
  prm.out_particles = d.out_particles;
  prm.out_weights = d.out_weights;
  prm.status = d.status;
  prm.status_time = d.status_time;
  prm.obs_flags = d.obs_flags;
  prm.window_stats = d.window_stats;
  prm.final_weights = d.final_weights;
}

static int check_desc(const gb_track_desc& d) {
  if (d.P <= 0 || d.N <= 0 || d.T < 2) return fail(GB_E_INVALID, "P, N must be positive and T >= 2%s");
  if (d.O < 1) return fail(GB_E_INVALID, "at least one observer is required%s");
  if (d.tile_w < 1 || d.tile_h < 1 || (int64_t)d.tile_w * d.tile_h > GB_MAX_TEMPLATE) {
    if (d.tile_w < 1 || d.tile_h < 1 || (int64_t)d.tile_w * d.tile_h > d.plan.max_template)
      return fail(GB_E_RESOURCE, "template larger than 1024 pixels (or than the plan's max_template)%s");
    if (d.tile_w > GB_MAX_TEMPLATE_SIDE || d.tile_h > GB_MAX_TEMPLATE_SIDE)
      return fail(GB_E_RESOURCE, "template above 1024 pixels and wider or taller than 128 pixels%s");
  }
  if (d.highpass_size != 0 && ((d.highpass_size & 0xffff) < 1 || (d.highpass_size & 0xffff) > GB_MAX_HIGHPASS ||
                               (d.highpass_size >> 16 & 0xffff) < 1 || (d.highpass_size >> 16 & 0xffff) > GB_MAX_HIGHPASS))
    return fail(GB_E_INVALID, "highpass_size: rows and columns must be between 1 and 31%s");
  {
    const int rows = d.highpass_size ? (d.highpass_size & 0xffff) : 5, cols = d.highpass_size ? (d.highpass_size >> 16 & 0xffff) : 5;
    const int org_r = (int16_t)(d.highpass_origin & 0xffff), org_c = (int16_t)(d.highpass_origin >> 16 & 0xffff);
    if (d.highpass_mode < GB_HP_REFLECT || d.highpass_mode > GB_HP_WRAP) return fail(GB_E_INVALID, "highpass_mode: unknown border mode%s");
    if (d.highpass_footprint_host) {
      uint32_t any = 0;
      for (int a = 0; a < rows; ++a) any |= d.highpass_footprint_host[a] & (cols >= 32 ? 0xffffffffu : ((1u << cols) - 1u));
      if (!any) return fail(GB_E_INVALID, "highpass_footprint_host: empty footprint%s");
    }
    // scipy.ndimage: -(size // 2) <= origin <= (size - 1) // 2
    if (org_r < -(rows / 2) || org_r > (rows - 1) / 2 || org_c < -(cols / 2) || org_c > (cols - 1) / 2)
      return fail(GB_E_INVALID, "highpass_origin: the shifted window must still cover its pixel%s");
  }
  if (d.interp_rows < 0 || d.interp_rows > 5 || d.interp_cols < 0 || d.interp_cols > 5)
    return fail(GB_E_INVALID, "interp_rows / interp_cols: spline degrees 1 to 5 (0 = the default 3)%s");
  if (!d.sigmas == !d.covariances) return fail(GB_E_INVALID, "exactly one of sigmas / covariances must be given%s");
  if (!d.images_host) return fail(GB_E_INVALID, "images_host is required%s");
  if (!d.image_offset_host || !d.image_index_host) return fail(GB_E_INVALID, "image_offset_host and image_index_host are required%s");
  // the tile kernels size their grey-level histograms for 1 to GB_MAX_BANDS bands (frames no time references are not read)
  for (int64_t k = 0; k < (int64_t)d.T * d.O; ++k) {
    const int idx = d.image_index_host[k];
    if (idx < 0) continue;
    const int nchan = d.images_host[d.image_offset_host[k % d.O] + idx].nchan;
    if (nchan < 1 || nchan > GB_MAX_BANDS) return fail(GB_E_INVALID, "frames must have 1 to 8 bands (gb_image.nchan)%s");
  }
  if (!d.images || !d.mask || !d.first || !d.last || !d.motion || !d.surfaces || !d.state_a || !d.state_b || !d.means ||
      !d.status || !d.status_time || !d.obs_flags || !d.tmpl_tile || !d.tmpl_values || !d.tmpl_quantiles ||
      !d.tmpl_nvalues || !d.tmpl_box || !d.tmpl_duv)
    return fail(GB_E_INVALID, "missing required buffer%s");
  if (d.rng_mode == GB_RNG_SUPPLIED && (!d.init_normals || !d.step_normals || !d.uniforms))
    return fail(GB_E_INVALID, "supplied-draw mode needs init_normals, step_normals and uniforms%s");
  if (d.plan.mode != GB_MODE_STREAM || d.plan.threads != GB_THREADS || d.plan.n_local < 1)
    return fail(GB_E_INVALID, "invalid launch plan (use gb_step_plan)%s");
  // up to GB_MAX_OBS observers: one slot each; more: one slot per observer with a frame at the same time, up to GB_MAX_OBS
  if (d.O > GB_MAX_OBS) {
    const int active = max_active_observers(d);
    if (active > GB_MAX_OBS) return fail(GB_E_RESOURCE, "more than 8 observers have a frame at the same time%s");
    if (d.plan.n_observers < (active > 1 ? active : 1) || d.plan.n_observers > GB_MAX_OBS)
      return fail(GB_E_INVALID, "plan.n_observers must cover the observers with a frame at the same time (use gb_step_plan)%s");
  } else if (d.plan.n_observers != d.O) {
    return fail(GB_E_INVALID, "streaming plan does not match the descriptor (use gb_step_plan)%s");
  }
  if ((d.plan.stream_nblk < 1 || d.plan.surf_bytes <= 0 ||
                                        d.plan.stream_batch < 1 || d.plan.stream_slots < 1 || d.plan.stream_slots > kMaxSlots))
    return fail(GB_E_INVALID, "streaming plan does not match the descriptor (use gb_step_plan)%s");
  if (d.plan.stream_block > GB_S4P_CAP || (d.plan.stream_block & 1)) return fail(GB_E_INVALID, "plan: stream_block must be even and <= 768%s");
  if (d.plan.stream_batch > 65535) return fail(GB_E_INVALID, "plan: stream_batch must be <= 65535%s");
  if (d.plan.scratch_bytes > 0 && !d.scratch) return fail(GB_E_INVALID, "plan needs a scratch buffer%s");
  if ((int64_t)d.plan.n_local < d.N) return fail(GB_E_INVALID, "plan does not cover N particles%s");
  return GB_OK;
}

// dynamic shared memory of k_s2_surface: windows up to ~66 px with the interleaved surface, up to ~80 px on planes;
// larger ones work in their global region
#ifndef GB_S2_SMEM_KB
#define GB_S2_SMEM_KB 110
#endif
static constexpr int kSurfaceSmem = GB_S2_SMEM_KB * 1024;
// ... and for large templates whose usual windows (the template plus 10-40 px) would not fit that: one CTA an SM with
// 224 KB, where a 128 x 128 template's windows up to ~165 px stay interleaved in shared memory and up to ~210 px staged
static constexpr int kSurfaceSmemLarge = 224 * 1024;

static int s2_smem_bytes(int tw, int th) {
  if ((int64_t)tw * th <= GB_SMEM_TEMPLATE) return kSurfaceSmem;
  return tile_bytes_needed(tw + 40, th + 40, tw, th, GB_MAX_BINS, 0) <= kSurfaceSmem ? kSurfaceSmem : kSurfaceSmemLarge;
}

struct StreamLayout {
  int64_t ev[2], uv, w, bsum, pre, pm, ibox, pflags[2], act, meta, ref, surf, total;
};

// Scratch of GB_MODE_STREAM for `B` points.
static StreamLayout stream_layout(int64_t B, int64_t N, int64_t O, int64_t nblk, int64_t surf_bytes) {
  StreamLayout L;
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    const int64_t at = off;
    off += (bytes + 255) / 256 * 256;
    return at;
  };
  L.ev[0] = take(B * 6 * N * 8);
  L.ev[1] = take(B * 6 * N * 8);
  L.uv = take(B * O * 2 * N * 8);
  L.w = take(B * N * 8);
  L.bsum = take(B * nblk * 8);
  L.pre = take(B * (nblk + 4) * 8);  // per point: prefix[0..nblk], 1/total, uniform draw, 1/N
  L.pm = take(B * nblk * 28 * 8);
  L.ibox = take(B * O * 5 * 4);
  L.pflags[0] = take(B * 4);
  L.pflags[1] = take(B * 4);
  L.act = take(B);
  L.meta = take(B * O * 8 * 4);
  L.ref = take(B * 6 * 8);
  L.surf = take(B * O * surf_bytes);
  L.total = off;
  return L;
}

// Point the kernels at the scratch arrays (indexed by the global point number) for time parity `par`, and at
// the batch of points [p0, p0 + pb).
static void stream_bind(const gb_track_desc& d, StepParams& prm, int par, int64_t p0, int64_t pb) {
  const gb_plan& pl = d.plan;
  const StreamLayout L = stream_layout(d.P, d.N, pl.n_observers, pl.stream_nblk, pl.surf_bytes);
  char* base = reinterpret_cast<char*>(d.scratch);
  prm.s_ev = reinterpret_cast<double*>(base + L.ev[par & 1]);
  prm.s_ev_next = reinterpret_cast<double*>(base + L.ev[(par + 1) & 1]);
  prm.s_uv = reinterpret_cast<double*>(base + L.uv);
  prm.s_w = reinterpret_cast<double*>(base + L.w);
  prm.s_bsum = reinterpret_cast<double*>(base + L.bsum);
  prm.s_pre = reinterpret_cast<double*>(base + L.pre);
  prm.s_pm = reinterpret_cast<double*>(base + L.pm);
  prm.s_ibox = reinterpret_cast<int*>(base + L.ibox);
  prm.s_pflags = reinterpret_cast<int*>(base + L.pflags[par & 1]);
  prm.s_pflags_next = reinterpret_cast<int*>(base + L.pflags[(par + 1) & 1]);
  prm.s_act = reinterpret_cast<uint8_t*>(base + L.act);
  prm.s_meta = reinterpret_cast<int*>(base + L.meta);
  prm.s_ref = reinterpret_cast<double*>(base + L.ref);
  prm.s_surf = base + L.surf;
  prm.surf_bytes = pl.surf_bytes;
  prm.s_block = pl.stream_block;
  prm.s_nblk = pl.stream_nblk;
  {
    const int mag = pl.tile_bytes < 0 ? -pl.tile_bytes : pl.tile_bytes;
    prm.s2_smem = s2_smem_bytes(d.tile_w, d.tile_h);
    prm.s2_budget = (pl.tile_bytes < 0 ? -1 : 1) * (mag < prm.s2_smem ? mag : prm.s2_smem);
  }
  prm.p0 = p0;
  prm.pb = pb;
}


// Side streams on which batches of points advance independently (points never interact).  One pool per device.
struct StreamPool {
  std::mutex busy;  // one call at a time per device: the fork / join events are shared
  cudaStream_t side[kMaxSlots] = {};
  cudaEvent_t fork = nullptr, join[kMaxSlots] = {};
  bool ready = false;
};
static StreamPool g_pools[16];
static std::mutex g_pool_mutex;

static int get_pool(StreamPool** out) {
  int dev = 0;
  GB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 16) return fail(GB_E_INVALID, "device index out of range%s");
  std::lock_guard<std::mutex> lock(g_pool_mutex);
  StreamPool& pool = g_pools[dev];
  if (!pool.ready) {
    for (int k = 0; k < kMaxSlots; ++k) {
      GB_CUDA(cudaStreamCreateWithFlags(&pool.side[k], cudaStreamNonBlocking));
      GB_CUDA(cudaEventCreateWithFlags(&pool.join[k], cudaEventDisableTiming));
    }
    GB_CUDA(cudaEventCreateWithFlags(&pool.fork, cudaEventDisableTiming));
    pool.ready = true;
  }
  *out = &pool;
  return GB_OK;
}

// Optional per-kernel timing of the pipelined flow (gb_kernel_timing): every launch is bracketed by CUDA events
// on the stream it is launched on; durations are accumulated per kernel kind when the track has finished.
enum { GB_K_ACTIVITY = 0, GB_K_SURFACE, GB_K_WEIGHTS, GB_K_RESAMPLE_PROPAGATE, GB_K_FINALIZE, GB_K_INIT, GB_K_TEMPLATE, GB_K_PUBLISH, GB_K_KINDS };
struct KernelTimer {
  std::mutex mu;
  bool on = false;
  std::vector<cudaEvent_t> ev;
  std::vector<int> kind;
  size_t used = 0;
  double ms[GB_K_KINDS] = {0};
  int64_t n[GB_K_KINDS] = {0};
  cudaEvent_t next() {
    if (used == ev.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev.push_back(e);
    }
    return ev[used++];
  }
  void begin(int k, cudaStream_t s) {
    if (!on) return;
    kind.push_back(k);
    cudaEventRecord(next(), s);
  }
  void end(cudaStream_t s) {
    if (!on) return;
    cudaEventRecord(next(), s);
  }
  // after the streams have been synchronised
  void collect() {
    for (size_t i = 0; i < kind.size(); ++i) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, ev[2 * i], ev[2 * i + 1]) == cudaSuccess) {
        ms[kind[i]] += t;
        n[kind[i]] += 1;
      }
    }
    kind.clear();
    used = 0;
  }
};
static KernelTimer g_ktimer;

// Per-device set-up of the gb_track* entry points and gb_sample_surface: the spline tables, and the dynamic shared memory of
// every kernel that may need more than 48 KB.  The outcome is kept, so a failure reaches every call, not only the first.
static int ensure_device() {
  static std::once_flag once[16];
  static cudaError_t result[16];
  int dev = 0;
  GB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 16) return fail(GB_E_INVALID, "device index out of range%s");
  std::call_once(once[dev], [dev]() {
    static double cp[GB_MAX_SURFACE], inv[GB_MAX_SURFACE];
    cp[0] = 2.0;
    inv[0] = 1.0;
    for (int i = 1; i < GB_MAX_SURFACE; ++i) {
      inv[i] = 1.0 / (4.0 - cp[i - 1]);
      cp[i] = inv[i];
    }
    cudaError_t err = cudaMemcpyToSymbol(c_spline_cp, cp, sizeof(cp));
    if (err == cudaSuccess) err = cudaMemcpyToSymbol(c_spline_inv, inv, sizeof(inv));
    auto smem = [&err](const void* kernel, int bytes) {
      if (err == cudaSuccess) err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    };
    smem((const void*)k_s2_surface<false>, kSurfaceSmem);
    smem((const void*)k_s2_surface<true>, kSurfaceSmemLarge);
    smem((const void*)k_s4p_resample_propagate<true, true>, kS4pSmem);
    smem((const void*)k_s4p_resample_propagate<false, true>, kS4pSmem);
    smem((const void*)k_s4p_resample_propagate<true, false>, kS4pSmem);
    smem((const void*)k_s4p_resample_propagate<false, false>, kS4pSmem);
    smem((const void*)k_template<true>, template_smem_bytes(GB_MAX_TEMPLATE_SIDE * GB_MAX_TEMPLATE_SIDE));
    result[dev] = err;
  });
  if (result[dev] != cudaSuccess) return fail(GB_E_CUDA, "spline tables or kernel attributes: %s", cudaGetErrorString(result[dev]));
  return GB_OK;
}

// `s` waits for the uploads of the frames of time prm.t (gb_track_desc.image_events_host).
static int wait_frames(const gb_track_desc& d, const StepParams& prm, cudaStream_t s) {
  if (!d.image_events_host) return GB_OK;
  for (int k = 0; k < prm.n_slots; ++k)
    if (prm.img[k] >= 0 && d.image_events_host[prm.img[k]])
      GB_CUDA(cudaStreamWaitEvent(s, (cudaEvent_t)d.image_events_host[prm.img[k]], 0));
  return GB_OK;
}

// The side streams of a call.  Points never interact, so batches of them advance on their own streams: batch b runs on side
// stream b % slots with scratch slot b % slots.  The caller's stream forks them after its own kernels (first-frame
// initialisation, templates) and joins them before the next such kernel and at the end.
struct SideStreams {
  const gb_track_desc& d;
  cudaStream_t stream;  // the caller's
  StreamPool* pool = nullptr;
  std::unique_lock<std::mutex> busy;
  int used = 0;  // side streams that receive a batch
  bool forked = false;

  SideStreams(const gb_track_desc& desc, cudaStream_t caller) : d(desc), stream(caller) {}
  int open() {
    if (int rc = get_pool(&pool)) return rc;
    busy = std::unique_lock<std::mutex>(pool->busy);
    const int64_t nbatch = (d.P + d.plan.stream_batch - 1) / d.plan.stream_batch;
    used = (int)(nbatch < d.plan.stream_slots ? nbatch : d.plan.stream_slots);
    return GB_OK;
  }
  // the side streams wait for what the caller's stream holds now (once until the next join)
  int fork() {
    if (forked) return GB_OK;
    GB_CUDA(cudaEventRecord(pool->fork, stream));
    for (int k = 0; k < used; ++k) GB_CUDA(cudaStreamWaitEvent(pool->side[k], pool->fork, 0));
    forked = true;
    return GB_OK;
  }
  // the caller's stream waits for what the side streams hold
  int join() {
    if (!forked) return GB_OK;
    for (int k = 0; k < used; ++k) {
      GB_CUDA(cudaEventRecord(pool->join[k], pool->side[k]));
      GB_CUDA(cudaStreamWaitEvent(stream, pool->join[k], 0));
    }
    forked = false;
    return GB_OK;
  }
  int wait_frames(const StepParams& prm) {
    for (int k = 0; k < used; ++k)
      if (int rc = gb::wait_frames(d, prm, pool->side[k])) return rc;
    return GB_OK;
  }
  // launch(prm bound to the batch, its side stream) for every batch of points
  template <class Launch>
  int each_batch(StepParams& prm, Launch&& launch) {
    const int64_t batch = d.plan.stream_batch;
    for (int64_t b = 0, p0 = 0; p0 < d.P; ++b, p0 += batch) {
      stream_bind(d, prm, prm.t, p0, p0 + batch <= d.P ? batch : d.P - p0);
      if (int rc = launch(prm, pool->side[b % d.plan.stream_slots])) return rc;
    }
    return GB_OK;
  }
};

// Each launch helper below adds the kernels it enqueues to `launches`.
static int launch_init(const StepParams& prm, bool cov, cudaStream_t stream, int64_t& launches) {
  if (cov)
    k_init<true><<<(unsigned)prm.P, GB_THREADS, kHeaderBytes, stream>>>(prm);
  else
    k_init<false><<<(unsigned)prm.P, GB_THREADS, kHeaderBytes, stream>>>(prm);
  ++launches;
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

static int launch_template(const gb_track_desc& d, StepParams prm, cudaStream_t stream, int64_t& launches) {
  const int area = prm.tile_w * prm.tile_h;
  if (area <= GB_SMEM_TEMPLATE) {
    k_template<false><<<(unsigned)(prm.P * prm.n_slots), 256, 0, stream>>>(prm);
  } else {
    // the work area of ranked frames: the surface regions (plan.surf_bytes >= 8 B a template pixel)
    prm.s_surf = reinterpret_cast<char*>(d.scratch) + stream_layout(d.P, d.N, d.plan.n_observers, d.plan.stream_nblk, d.plan.surf_bytes).surf;
    prm.surf_bytes = d.plan.surf_bytes;
    k_template<true><<<(unsigned)(prm.P * prm.n_slots), 256, template_smem_bytes(area), stream>>>(prm);
  }
  ++launches;
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

static void launch_surface(const StepParams& prm, const FrameMaps& fm, cudaStream_t s, int64_t& launches) {
  if (prm.tile_w * prm.tile_h > GB_SMEM_TEMPLATE)
    k_s2_surface<true><<<(unsigned)(prm.pb * prm.n_slots), GB_S2_THREADS, prm.s2_smem, s>>>(prm, fm, prm.s2_budget);
  else
    k_s2_surface<false><<<(unsigned)(prm.pb * prm.n_slots), GB_S2_THREADS, prm.s2_smem, s>>>(prm, fm, prm.s2_budget);
  ++launches;
}

static void launch_weights(const StepParams& prm, cudaStream_t s, int64_t& launches) {
  if (spline_is_hermite(prm.interp_cols, prm.interp_rows))
    k_s3_weights<false><<<dim3((unsigned)prm.s_nblk, (unsigned)prm.pb), s3_threads(prm.s_block), 0, s>>>(prm);
  else
    k_s3_weights<true><<<dim3((unsigned)prm.s_nblk, (unsigned)prm.pb), s3_threads(prm.s_block), 0, s>>>(prm);
  ++launches;
}

// One batch of the step-by-step flow: k_s0 k_s1 k_s2 k_s3 k_s4* k_s5 (gb_track for choice / residual, gb_track_step).
template <bool COV>
static int step_batch(const StepParams& prm, const FrameMaps& fm, cudaStream_t s, int64_t& launches) {
  const unsigned nb = (unsigned)(prm.pb * prm.s_nblk);
  k_s0_reset<<<grid_for(prm.pb * prm.slot_stride * 5, 256), 256, 0, s>>>(prm);
  ++launches;
  k_s1_propagate<<<nb, GB_SBLOCK_THREADS, 0, s>>>(prm);
  ++launches;
  launch_surface(prm, fm, s, launches);
  launch_weights(prm, s, launches);
  if (prm.resample_method == GB_RESAMPLE_CHOICE || prm.resample_method == GB_RESAMPLE_RESIDUAL) {
    if (prm.resample_method == GB_RESAMPLE_CHOICE)
      k_s4c_scan<<<nb, GB_SBLOCK_THREADS, 0, s>>>(prm);
    else
      k_s4r_residual<<<(unsigned)prm.pb, GB_SBLOCK_THREADS, 0, s>>>(prm);
    ++launches;
    k_s4c_gather<COV><<<nb, GB_SBLOCK_THREADS, 0, s>>>(prm);
  } else {
    k_s4_resample<COV><<<nb, GB_SBLOCK_THREADS, 0, s>>>(prm);
  }
  ++launches;
  k_s5_finalize<COV><<<(unsigned)((prm.pb + 3) / 4), 128, 0, s>>>(prm);
  ++launches;
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

// One batch of the pipelined flow: [k_s0p] k_s2 k_s3 k_s3b k_s4p k_s5p, k_s4p advancing the particles to the time `nxt`
// describes.  `activity`: k_s0p writes the activity of this time; `update`: some point of the call is updated at it.
static int pipelined_batch(const StepParams& prm, const FrameMaps& fm, const NextParams& nxt, bool activity, bool update, bool cov,
                           bool tangent, cudaStream_t s, int64_t& launches) {
  KernelTimer& kt = g_ktimer;
  if (activity) {
    kt.begin(GB_K_ACTIVITY, s);
    k_s0p_activity<<<grid_for(prm.pb, 256), 256, 0, s>>>(prm);
    kt.end(s);
    ++launches;
  }
  if (update) {
    kt.begin(GB_K_SURFACE, s);
    launch_surface(prm, fm, s, launches);
    kt.end(s);
    kt.begin(GB_K_WEIGHTS, s);
    launch_weights(prm, s, launches);
    kt.end(s);
    kt.begin(GB_K_PUBLISH, s);
    k_s3b_publish<<<(unsigned)((prm.pb + 7) / 8), 256, 0, s>>>(prm);
    kt.end(s);
    ++launches;
  }
  kt.begin(GB_K_RESAMPLE_PROPAGATE, s);
  const dim3 grid((unsigned)prm.s_nblk, (unsigned)prm.pb);
  if (cov && tangent)
    k_s4p_resample_propagate<true, true><<<grid, GB_S4P_THREADS, kS4pSmem, s>>>(prm, nxt);
  else if (cov)
    k_s4p_resample_propagate<true, false><<<grid, GB_S4P_THREADS, kS4pSmem, s>>>(prm, nxt);
  else if (tangent)
    k_s4p_resample_propagate<false, true><<<grid, GB_S4P_THREADS, kS4pSmem, s>>>(prm, nxt);
  else
    k_s4p_resample_propagate<false, false><<<grid, GB_S4P_THREADS, kS4pSmem, s>>>(prm, nxt);
  kt.end(s);
  ++launches;
  kt.begin(GB_K_FINALIZE, s);
  if (cov)
    k_s5p_finalize<true><<<(unsigned)((prm.pb + 3) / 4), 128, 0, s>>>(prm);
  else
    k_s5p_finalize<false><<<(unsigned)((prm.pb + 3) / 4), 128, 0, s>>>(prm);
  kt.end(s);
  ++launches;
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

// What k_s4p needs of time t + 1 (no slots after the last time).  `spec_update`: no point starts at t.
static NextParams next_params(const gb_track_desc& d, int t, bool spec_update) {
  NextParams nxt;
  memset(&nxt, 0, sizeof(nxt));
  for (int o = 0; o < GB_MAX_OBS; ++o) nxt.img[o] = -1;
  nxt.spec_update = spec_update;
  if (t + 1 < d.T) {
    StepParams pn;
    fill_params(d, t + 1, pn);
    nxt.tau = pn.tau;
    nxt.tau2 = pn.tau2;
    nxt.n_slots = pn.n_slots;
    for (int s = 0; s < pn.n_slots; ++s) {
      nxt.obs[s] = pn.obs[s];
      nxt.img[s] = pn.img[s];
      nxt.cam[s] = pn.cam[s];
    }
  }
  return nxt;
}

// What gb_track does at each time, from the host copies of first / last / mask (tracker.py:321-347).  A time without init
// or update work is idle: a point is advanced from t to t + 1 only at times it starts or is updated at.
struct TimeWork {
  bool init;       // a point starts (k_init)
  bool tmpl;       // an observer's template is cut (k_template)
  bool update;     // a point that started earlier is updated
  bool staggered;  // a template is cut after its point's first frame
};
struct Schedule {
  std::vector<TimeWork> at;
  bool staggered = false;  // at any time
};

static Schedule schedule(const gb_track_desc& d) {
  Schedule s;
  s.at.assign(d.T, TimeWork{});
  std::vector<int> tmpl_frame(d.O);
  for (int o = 0; o < d.O; ++o) tmpl_frame[o] = template_frame(d, o);
  for (int64_t p = 0; p < d.P; ++p) {
    const int f = d.first_host[p], l = d.last_host[p] < d.T ? d.last_host[p] : d.T - 1;
    if (f < 0 || f >= d.T || l < f) continue;
    s.at[f].init = true;
    for (int t = f + 1; t <= l; ++t) s.at[t].update = true;
    for (int o = 0; o < d.O; ++o) {
      const int tf = tmpl_frame[o];
      if (tf >= f && tf <= l && d.mask_host[p * d.O + o]) {
        s.at[tf].tmpl = true;
        if (tf > f) s.at[tf].staggered = s.staggered = true;
      }
    }
  }
  return s;
}

// gb_track.  The pipelined flow (systematic / stratified resampling) advances the particles to the next time in k_s4p of
// this one; the step-by-step flow (choice / residual) moves them in k_s1 of the next update, or on the caller's stream
// ahead of a template that is cut after a point's first frame.  The flows differ only in what the caller's stream runs at
// a time and in the kernels of one batch.
static int track(const gb_track_desc& d, cudaStream_t stream, int64_t& launches) {
  const bool pipelined = d.resample_method != GB_RESAMPLE_CHOICE && d.resample_method != GB_RESAMPLE_RESIDUAL;
  const bool cov = d.covariances != nullptr;
  // kernels without the tangent models' DEM gathers when the caller says no point uses them (0 = unknown: assume any kind)
  const bool tangent = d.motion_kinds == 0 || (d.motion_kinds & ((1 << GB_MOTION_TANGENT_CARTESIAN) | (1 << GB_MOTION_TANGENT_CYLINDRICAL))) != 0;
  const Schedule work = schedule(d);
  if (work.staggered && !d.weight_state)
    return fail(GB_E_INVALID, "weight_state is required when a template starts after a point's first frame%s");
  SideStreams sides(d, stream);
  int rc = sides.open();
  if (rc) return rc;
  if (pipelined) {
    StepParams prm;
    fill_params(d, 0, prm);
    stream_bind(d, prm, 0, 0, d.P);
    k_s0p_reset<<<grid_for(d.P * prm.slot_stride * 5, 256), 256, 0, stream>>>(prm);
    ++launches;
    GB_CUDA(cudaGetLastError());
  }
  bool have_activity = false;
  for (int t = 0; t < d.T; ++t) {
    const TimeWork& w = work.at[t];
    if (!w.init && !w.update) {
      have_activity = false;  // a gap: the last k_s5p wrote the activity of a time that is not processed
      continue;
    }
    StepParams prm;
    fill_params(d, t, prm);
    FrameMaps fm;
    frame_maps(prm, fm);
    if (w.init || w.tmpl) {
      if ((rc = sides.join()) || (rc = wait_frames(d, prm, stream))) return rc;
      if (pipelined) {
        stream_bind(d, prm, t, 0, d.P);
        prm.tmpl_from_ev = 1;
        if (w.init) {
          g_ktimer.begin(GB_K_INIT, stream);
          if ((rc = launch_init(prm, cov, stream, launches))) return rc;
          g_ktimer.end(stream);
        }
        if (w.tmpl) {
          g_ktimer.begin(GB_K_TEMPLATE, stream);
          if ((rc = launch_template(d, prm, stream, launches))) return rc;
          g_ktimer.end(stream);
        }
      } else {
        if (w.init && (rc = launch_init(prm, cov, stream, launches))) return rc;
        if (w.staggered) {
          dim3 grid((unsigned)grid_for(d.N, 256), (unsigned)d.P, 1);
          k_evolve<<<grid, 256, 0, stream>>>(d.motion, d.surfaces, d.P, d.N, prm.tau, prm.tau2, d.step_normals,
                                             (int64_t)(d.T - 1) * d.N * 3, ((t - 1) & 1) ? d.state_b : d.state_a, d.first, d.last,
                                             d.status, d.status_time, t, d.rng_mode, d.seed, d.T - 1, d.point_offset);
          ++launches;
          GB_CUDA(cudaGetLastError());
          prm.skip_evolve = 1;
        }
        if (w.tmpl && (rc = launch_template(d, prm, stream, launches))) return rc;
      }
    }
    if (!pipelined && !w.update) continue;  // (that flow's batches only update)
    if ((rc = sides.fork())) return rc;
    if (w.update && (rc = sides.wait_frames(prm))) return rc;
    if (pipelined) {
      const NextParams nxt = next_params(d, t, !w.init);
      // activity of time t: written by k_s5p of the previous processed time unless statuses may have changed since
      const bool activity = !have_activity || w.init || w.tmpl;
      have_activity = true;
      rc = sides.each_batch(prm, [&](const StepParams& b, cudaStream_t s) {
        return pipelined_batch(b, fm, nxt, activity, w.update, cov, tangent, s, launches);
      });
    } else {
      rc = sides.each_batch(prm, [&](const StepParams& b, cudaStream_t s) {
        return cov ? step_batch<true>(b, fm, s, launches) : step_batch<false>(b, fm, s, launches);
      });
    }
    if (rc) return rc;
  }
  if ((rc = sides.join())) return rc;
  if (g_ktimer.on) {
    GB_CUDA(cudaStreamSynchronize(stream));
    g_ktimer.collect();
  }
  return GB_OK;
}

// Motion.initialize_particles as a stand-alone call (motion.py:149-163, 260-283, 378-390, 485-505): one thread per particle,
// normals[p][i][6] in the reference's draw order (see init_particle).  Grid: (blocks over N, P).
__global__ void k_init_particles(const gb_motion* __restrict__ motion, const gb_surface* __restrict__ surfaces, int64_t N,
                                 const double* __restrict__ normals, double* __restrict__ state, int32_t* status) {
  const int64_t p = blockIdx.y;
  const gb_motion m = motion[p];
  uint32_t flags = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    double zn[6], s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) zn[c] = normals[(p * N + i) * 6 + c];
    init_particle(m, surfaces, zn, s, flags);
#pragma unroll
    for (int c = 0; c < 6; ++c) state[(p * 6 + c) * N + i] = s[c];
  }
  if (flags && status) atomicCAS(&status[p], 0, GB_ST_DEM_BOUNDS);
}

// Motion.compute_log_likelihoods as a stand-alone call (motion.py:181-204) on SoA state [P][6][N] -> ll[P][N].
__global__ void k_motion_log_likelihoods(const gb_motion* __restrict__ motion, const gb_surface* __restrict__ surfaces, int64_t N,
                                         const double* __restrict__ state, double* __restrict__ ll, int32_t* status) {
  const int64_t p = blockIdx.y;
  const gb_motion m = motion[p];
  uint32_t flags = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    const double* s = state + p * 6 * N;
    ll[p * N + i] = surface_log_likelihood(m, surfaces, s[i], s[N + i], s[2 * N + i], flags);
  }
  if (flags && status) atomicCAS(&status[p], 0, GB_ST_DEM_BOUNDS);
}

// Observer.sample_tile as a stand-alone call (observer.py:178-214): interpolating spline (degree 3 not-a-knot = FITPACK's, or
// degree 1) through the cell centres of `tile` (Mv rows x Mu columns), evaluated at n points given relative to the first cell
// centre in cell units.  One CTA: Hermite data (F, F_u, F_v, F_uv) in the caller's work area `herm` [Mv][Mu | 1] float4.
__global__ void __launch_bounds__(256) k_sample_surface(const double* __restrict__ tile, int Mu, int Mv, int ku, int kv,
                                                        const double* __restrict__ xy, int64_t n, float4* __restrict__ herm,
                                                        double* __restrict__ out) {
  const int tid = threadIdx.x, nthr = blockDim.x, Mp = Mu | 1;
  const int lin_u = ku == 1, lin_v = kv == 1;
  for (int i = tid; i < Mu * Mv; i += nthr) {
    const int r = i / Mu, c = i - r * Mu;
    herm[r * Mp + c] = make_float4((float)tile[i], 0.0f, 0.0f, 0.0f);
  }
  __syncthreads();
  float* base = reinterpret_cast<float*>(herm);
  if (!spline_is_hermite(ku, kv)) {  // degrees 2 / 4 / 5: B-spline coefficients (work area behind the Hermite array)
    double* abu = reinterpret_cast<double*>(herm + (int64_t)Mv * Mp);
    double* abv = abu + (int64_t)Mu * (2 * ku + 1);
    if (tid == 0) bspline_factor(abu, Mu, ku);
    if (tid == 32) bspline_factor(abv, Mv, kv);
    __syncthreads();
    for (int r = tid; r < Mv; r += nthr) bspline_solve_line(abu, Mu, ku, base + (int64_t)r * Mp * 4, 4);
    __syncthreads();
    for (int c = tid; c < Mu; c += nthr) bspline_solve_line(abv, Mv, kv, base + (int64_t)c * 4, Mp * 4);
    __syncthreads();
    for (int64_t i = tid; i < n; i += nthr) out[i] = (double)bspline_eval(herm, Mp, Mu, Mv, xy[2 * i], xy[2 * i + 1], ku, kv);
    return;
  }
  for (int line = tid; line < Mv + Mu; line += nthr) {
    if (line < Mv) spline_slopes_line(base + (int64_t)line * Mp * 4, base + (int64_t)line * Mp * 4 + 1, 4, Mu, !lin_u);
    else spline_slopes_line(base + (int64_t)(line - Mv) * 4, base + (int64_t)(line - Mv) * 4 + 2, Mp * 4, Mv, !lin_v);
  }
  __syncthreads();
  for (int c = tid; c < Mu; c += nthr) spline_slopes_line(base + (int64_t)c * 4 + 1, base + (int64_t)c * 4 + 3, Mp * 4, Mv, !lin_v);
  __syncthreads();
  for (int64_t i = tid; i < n; i += nthr) out[i] = (double)hermite_eval_sat(herm, Mp, Mu, Mv, xy[2 * i], xy[2 * i + 1], lin_u != 0, lin_v != 0);
}

}  // namespace gb

using namespace gb;

extern "C" {

int gb_version(void) { return GB_VERSION; }
const char* gb_last_error(void) { return g_error; }
int64_t gb_struct_size(int32_t which) {
  switch (which) {
    case 0: return sizeof(gb_camera);
    case 1: return sizeof(gb_image);
    case 2: return sizeof(gb_surface);
    case 3: return sizeof(gb_motion);
    case 4: return sizeof(gb_plan);
    case 5: return sizeof(gb_track_desc);
    case 6: return sizeof(gb_stage_io);
    default: return -1;
  }
}

int gb_kernel_timing(int32_t enable) {
  std::lock_guard<std::mutex> guard(gb::g_ktimer.mu);
  gb::g_ktimer.on = enable != 0;
  gb::g_ktimer.kind.clear();
  gb::g_ktimer.used = 0;
  for (int k = 0; k < gb::GB_K_KINDS; ++k) {
    gb::g_ktimer.ms[k] = 0.0;
    gb::g_ktimer.n[k] = 0;
  }
  return GB_OK;
}

int gb_kernel_timing_read(double* ms, int64_t* launches, int32_t n) {
  if (!ms || !launches || n < 0) return gb::fail(GB_E_INVALID, "null argument%s");
  std::lock_guard<std::mutex> guard(gb::g_ktimer.mu);
  for (int k = 0; k < n; ++k) {
    ms[k] = k < gb::GB_K_KINDS ? gb::g_ktimer.ms[k] : 0.0;
    launches[k] = k < gb::GB_K_KINDS ? gb::g_ktimer.n[k] : 0;
  }
  return GB_OK;
}

int gb_camera_from_vector(const double* v, const double* corr, gb_camera* out) {
  if (!v || !out) return fail(GB_E_INVALID, "null argument%s");
  memset(out, 0, sizeof(*out));
  const double d2r = 3.14159265358979323846 / 180.0;
  const double c1 = cos(v[3] * d2r), c2 = cos(v[4] * d2r), c3 = cos(v[5] * d2r);
  const double s1 = sin(v[3] * d2r), s2 = sin(v[4] * d2r), s3 = sin(v[5] * d2r);
  const double R[9] = {c1 * c3 + s1 * s2 * s3, c1 * s2 * s3 - c3 * s1, -c2 * s3,
                       c3 * s1 * s2 - c1 * s3, s1 * s3 + c1 * c3 * s2, -c2 * c3,
                       c2 * s1,                c1 * c2,                s2};
  for (int i = 0; i < 9; ++i) out->R[i] = R[i];
  for (int i = 0; i < 3; ++i) out->xyz[i] = v[i];
  out->imgsz[0] = (int32_t)v[6];
  out->imgsz[1] = (int32_t)v[7];
  out->f[0] = v[8];
  out->f[1] = v[9];
  out->cc[0] = out->imgsz[0] / 2.0 + v[10];
  out->cc[1] = out->imgsz[1] / 2.0 + v[11];
  for (int i = 0; i < 6; ++i) out->k[i] = v[12 + i];
  out->p[0] = v[18];
  out->p[1] = v[19];
  if (corr) {
    out->has_corr = 1;
    out->corr_c1 = corr[1] - 1.0;
    out->corr_c2 = 2.0 * corr[0];
  }
  return GB_OK;
}

int gb_project(const gb_camera* cam, const double* xyz, int64_t n, double* uv, void* stream) {
  if (!cam || (n > 0 && (!xyz || !uv))) return fail(GB_E_INVALID, "null argument%s");
  if (n <= 0) return GB_OK;
  k_project<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(*cam, xyz, n, uv);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_unproject(const gb_camera* cam, const double* uv, int64_t n, int directions, const double* depth, double* xyz,
                 void* stream) {
  if (!cam || (n > 0 && (!xyz || !uv))) return fail(GB_E_INVALID, "null argument%s");
  if (n <= 0) return GB_OK;
  k_unproject<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(*cam, uv, n, directions, depth, xyz);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

// ---------------------------------------------------------------------------------------------
// Frame ingest: JPEG bytes -> pixels in device memory through nvJPEG (a library call, like the reference's own decode through
// GDAL / libjpeg, image.py:137-214).  The library is opened at run time, so libglimpse_b200.so itself does not depend on it.
// ---------------------------------------------------------------------------------------------
namespace {
struct NvJpeg {
  void* lib = nullptr;
  nvjpegStatus_t (*create)(nvjpegHandle_t*) = nullptr;
  nvjpegStatus_t (*state_create)(nvjpegHandle_t, nvjpegJpegState_t*) = nullptr;
  nvjpegStatus_t (*info)(nvjpegHandle_t, const unsigned char*, size_t, int*, nvjpegChromaSubsampling_t*, int*, int*) = nullptr;
  nvjpegStatus_t (*decode)(nvjpegHandle_t, nvjpegJpegState_t, const unsigned char*, size_t, nvjpegOutputFormat_t, nvjpegImage_t*,
                           cudaStream_t) = nullptr;
  nvjpegHandle_t handle = nullptr;
  nvjpegJpegState_t state = nullptr;
  int device = -1;
  bool tried = false;
};
thread_local NvJpeg t_nvjpeg;

int nvjpeg_ready(NvJpeg** out) {
  NvJpeg& j = t_nvjpeg;
  if (!j.tried) {
    j.tried = true;
    for (const char* name : {"libnvjpeg.so.12", "/usr/local/cuda/lib64/libnvjpeg.so.12", "libnvjpeg.so"}) {
      j.lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
      if (j.lib) break;
    }
    if (j.lib) {
      j.create = reinterpret_cast<decltype(j.create)>(dlsym(j.lib, "nvjpegCreateSimple"));
      j.state_create = reinterpret_cast<decltype(j.state_create)>(dlsym(j.lib, "nvjpegJpegStateCreate"));
      j.info = reinterpret_cast<decltype(j.info)>(dlsym(j.lib, "nvjpegGetImageInfo"));
      j.decode = reinterpret_cast<decltype(j.decode)>(dlsym(j.lib, "nvjpegDecode"));
    }
  }
  if (!j.lib || !j.create || !j.state_create || !j.info || !j.decode)
    return fail(GB_E_RESOURCE, "decode_jpeg: libnvjpeg.so.12 could not be opened%s");
  int dev = 0;
  GB_CUDA(cudaGetDevice(&dev));
  if (!j.handle || j.device != dev) {  // (one handle per calling thread; a thread that changes device gets a new one)
    if (j.create(&j.handle) != NVJPEG_STATUS_SUCCESS || j.state_create(j.handle, &j.state) != NVJPEG_STATUS_SUCCESS)
      return fail(GB_E_RESOURCE, "decode_jpeg: nvjpegCreateSimple failed%s");
    j.device = dev;
  }
  *out = &j;
  return GB_OK;
}
}  // namespace

int gb_jpeg_info(const uint8_t* jpeg, int64_t nbytes, int32_t* width, int32_t* height, int32_t* nchan) {
  if (!jpeg || nbytes <= 0 || !width || !height || !nchan) return fail(GB_E_INVALID, "null argument%s");
  NvJpeg* j = nullptr;
  if (int rc = nvjpeg_ready(&j)) return rc;
  int ncomp = 0, ws[NVJPEG_MAX_COMPONENT], hs[NVJPEG_MAX_COMPONENT];
  nvjpegChromaSubsampling_t sub;
  if (j->info(j->handle, jpeg, (size_t)nbytes, &ncomp, &sub, ws, hs) != NVJPEG_STATUS_SUCCESS)
    return fail(GB_E_INVALID, "decode_jpeg: not a JPEG stream nvJPEG can read%s");
  *width = ws[0];
  *height = hs[0];
  *nchan = ncomp >= 3 ? 3 : 1;
  return GB_OK;
}

int gb_decode_jpeg(const uint8_t* jpeg, int64_t nbytes, int32_t width, int32_t height, int32_t nchan, uint8_t* out, void* stream) {
  if (!jpeg || nbytes <= 0 || !out) return fail(GB_E_INVALID, "null argument%s");
  if (nchan != 1 && nchan != 3) return fail(GB_E_INVALID, "decode_jpeg: 1 (grey) or 3 (RGB) output bands%s");
  int32_t w = 0, h = 0, c = 0;
  if (int rc = gb_jpeg_info(jpeg, nbytes, &w, &h, &c)) return rc;
  if (w != width || h != height) return fail(GB_E_INVALID, "decode_jpeg: the stream's size differs from the frame's%s");
  NvJpeg* j = nullptr;
  if (int rc = nvjpeg_ready(&j)) return rc;
  nvjpegImage_t img;
  memset(&img, 0, sizeof(img));
  img.channel[0] = out;
  img.pitch[0] = (size_t)width * nchan;
  const nvjpegStatus_t st = j->decode(j->handle, j->state, jpeg, (size_t)nbytes, nchan == 3 ? NVJPEG_OUTPUT_RGBI : NVJPEG_OUTPUT_Y, &img,
                                      (cudaStream_t)stream);
  if (st != NVJPEG_STATUS_SUCCESS) return fail(GB_E_CUDA, "decode_jpeg: nvjpegDecode failed%s");
  return GB_OK;
}

int64_t gb_viewshed_work_bytes(int32_t nx, int32_t ny, int32_t max_rings) {
  if (nx < 1 || ny < 1 || max_rings < 1) return 0;
  return viewshed_layout((int64_t)nx * ny, max_rings, nullptr, nullptr);
}

int gb_viewshed(const double* z, int32_t nx, int32_t ny, const double* x_centres, const double* y_centres, double cell,
                const double* origin, const double* corr, int32_t max_rings, void* work, int64_t work_bytes, uint8_t* visible,
                void* stream) {
  if (!z || !x_centres || !y_centres || !origin || !work || !visible) return fail(GB_E_INVALID, "null argument%s");
  if (nx < 1 || ny < 1 || max_rings < 1 || !(cell > 0.0)) return fail(GB_E_INVALID, "viewshed: empty raster or cell size%s");
  if ((int64_t)nx * ny > 0x7fffffff) return fail(GB_E_RESOURCE, "viewshed: more than 2^31 cells%s");
  ViewshedParams q;
  memset(&q, 0, sizeof(q));
  const int64_t n = (int64_t)nx * ny;
  if (viewshed_layout(n, max_rings, reinterpret_cast<unsigned char*>(work), &q.w) > work_bytes)
    return fail(GB_E_INVALID, "viewshed: work buffer smaller than gb_viewshed_work_bytes%s");
  q.z = z;
  q.xc = x_centres;
  q.yc = y_centres;
  q.nx = nx;
  q.ny = ny;
  q.R = max_rings;
  q.ox = origin[0];
  q.oy = origin[1];
  q.oz = origin[2];
  q.inv_cell = 1.0 / cell;
  if (corr) {
    q.has_corr = 1;
    q.corr_c1 = corr[1] - 1.0;
    q.corr_c2 = 2.0 * corr[0];
  }
  q.visible = visible;
  // GB_VS_RING_CAP (test hook): a lower ring capacity sends small rasters through the large-ring sort, merge and search; the
  // result is the same
  q.cap = GB_VS_MAX_RING;
  if (const char* e = getenv("GB_VS_RING_CAP")) {
    const int c = atoi(e);
    q.cap = c < 1 ? 1 : c > GB_VS_MAX_RING ? GB_VS_MAX_RING : c;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int sort_smem = GB_VS_MAX_RING * 12, sweep_smem = (GB_VS_MAX_RING + 2) * 8;
  // (per device and cheap: set on every call rather than remembered per process)
  GB_CUDA(cudaFuncSetAttribute(k_vs_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, sort_smem));
  GB_CUDA(cudaFuncSetAttribute(k_vs_sweep<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sweep_smem));
  GB_CUDA(cudaFuncSetAttribute(k_vs_sweep<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sweep_smem));
  k_vs_init<<<grid_for(max_rings + 1, 256), 256, 0, s>>>(q);
  k_vs_cells<<<grid_for(n, 256), 256, 0, s>>>(q);
  k_vs_count<<<grid_for(n, 256), 256, 0, s>>>(q);
  k_vs_scan<<<1, 1024, 0, s>>>(q);
  k_vs_scatter<<<grid_for(n, 256), 256, 0, s>>>(q);
  k_vs_sort<<<max_rings, GB_VS_SORT_THREADS, sort_smem, s>>>(q);
  // enough passes for a ring of all n cells; a pass no ring needs returns at once (the ring sizes stay on the device)
  for (int pass = 0, passes = vs_merge_passes((int)n, q.cap); pass < passes; ++pass)
    k_vs_merge<<<grid_for(n, 256), 256, 0, s>>>(q, pass);
  k_vs_sweep<false><<<1, GB_VS_SWEEP_THREADS, sweep_smem, s>>>(q);  // (one of the two returns at once)
  k_vs_sweep<true><<<1, GB_VS_SWEEP_THREADS, sweep_smem, s>>>(q);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_project_image(const gb_image* src, const gb_camera* dst, int32_t method, void* out, void* stream) {
  if (!src || !dst || !out || !src->pixels) return fail(GB_E_INVALID, "null argument%s");
  if (method != 0 && method != 1) return fail(GB_E_INVALID, "project_image: method must be 0 (nearest) or 1 (linear)%s");
  if (src->cam.affine || dst->affine) return fail(GB_E_INVALID, "project_image: both cameras must be frame cameras%s");
  if (src->cam.xyz[0] != dst->xyz[0] || src->cam.xyz[1] != dst->xyz[1] || src->cam.xyz[2] != dst->xyz[2])
    return fail(GB_E_INVALID, "Source and target cameras have different positions ('xyz')%s");
  if (src->width < 2 || src->height < 2 || src->nchan < 1 || dst->imgsz[0] < 1 || dst->imgsz[1] < 1 || src->dtype < GB_PIX_U8 ||
      src->dtype > GB_PIX_F64)
    return fail(GB_E_INVALID, "project_image: the source frame needs two pixels per axis and a supported pixel type%s");
  const int64_t total = (int64_t)dst->imgsz[0] * dst->imgsz[1];
  k_project_image<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(*src, *dst, method, reinterpret_cast<uint8_t*>(out));
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_state_from_rows(const double* rows, int64_t npoints, int64_t n, double* state, void* stream) {
  if (!rows || !state) return fail(GB_E_INVALID, "null argument%s");
  k_state_from_rows<<<grid_for(npoints * n, 256), 256, 0, (cudaStream_t)stream>>>(rows, npoints, n, state);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_state_to_rows(const double* state, int64_t npoints, int64_t n, double* rows, void* stream) {
  if (!rows || !state) return fail(GB_E_INVALID, "null argument%s");
  k_state_to_rows<<<grid_for(npoints * n, 256), 256, 0, (cudaStream_t)stream>>>(state, npoints, n, rows);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_step_plan(int64_t n_particles, int32_t tile_w, int32_t tile_h, int64_t npoints, int32_t n_observers,
                 int32_t flags, int32_t mode, gb_plan* plan) {
  return gb_step_plan_ex(n_particles, tile_w, tile_h, npoints, n_observers, flags, mode, 191, plan);
}

int gb_step_plan_ex(int64_t n_particles, int32_t tile_w, int32_t tile_h, int64_t npoints, int32_t n_observers,
                    int32_t flags, int32_t mode, int32_t window_margin, gb_plan* plan) {
  if (window_margin < 4 || window_margin > GB_MAX_SURFACE - 1) return fail(GB_E_INVALID, "window_margin must be between 4 and 1023%s");
  if (!plan || n_particles <= 0 || tile_w < 1 || tile_h < 1) return fail(GB_E_INVALID, "bad plan arguments%s");
  if ((int64_t)tile_w * tile_h > GB_MAX_TEMPLATE && !(flags & GB_PLAN_LARGE_TEMPLATES))
    return fail(GB_E_RESOURCE, "template larger than 1024 pixels (GB_PLAN_LARGE_TEMPLATES admits up to 128 x 128)%s");
  if ((int64_t)tile_w * tile_h > GB_MAX_TEMPLATE && (tile_w > GB_MAX_TEMPLATE_SIDE || tile_h > GB_MAX_TEMPLATE_SIDE))
    return fail(GB_E_RESOURCE, "template above 1024 pixels and wider or taller than 128 pixels%s");
  if (flags & ~(GB_PLAN_RANKED_FRAMES | GB_PLAN_LARGE_TEMPLATES)) return fail(GB_E_INVALID, "unknown plan flags%s");
  if (n_observers < 1 || n_observers > GB_MAX_OBS) return fail(GB_E_INVALID, "between 1 and 8 observers are supported%s");
  if (mode != GB_MODE_STREAM) return fail(GB_E_INVALID, "unknown mode (the cluster-per-point organisation of round 1 was removed)%s");
  memset(plan, 0, sizeof(*plan));
  plan->mode = mode;
  plan->n_observers = n_observers;
  plan->threads = GB_THREADS;
  plan->max_template = tile_w * tile_h;
  plan->smem_bytes = kMaxSmem;
  if (mode == GB_MODE_STREAM) {
    if (n_particles > 0x7fffffff / 4) return fail(GB_E_RESOURCE, "too many particles per point%s");
    plan->cluster = 1;
    plan->n_local = (int32_t)n_particles;
    plan->particles_in_smem = 0;
    plan->tile_bytes = s2_smem_bytes(tile_w, tile_h);
    // particles of a point are cut into equal even-sized blocks that fit k_s4p's shared memory (<= 768 parents)
    plan->stream_nblk = (int32_t)((n_particles + GB_S4P_CAP - 1) / GB_S4P_CAP);
    plan->stream_block = (int32_t)(((n_particles + plan->stream_nblk - 1) / plan->stream_nblk + 1) / 2 * 2);
    plan->stream_nblk = (int32_t)((n_particles + plan->stream_block - 1) / plan->stream_block);
    // surface regions sized for search windows up to `window_margin` (191 by default) px larger than the template
    {
      // largest window + (ranked frames: rank histograms with one bin per window pixel, and the window's grey values) +
      // the collocation factors of spline degrees 2 / 4 / 5
      const int64_t Su = tile_w + window_margin, Sv = tile_h + window_margin;
      const bool ranked = (flags & GB_PLAN_RANKED_FRAMES) != 0;
      // (uint8 frames: one bin per band sum, 255 * bands + 1 for up to GB_MAX_BANDS bands; a ranked plan may hold them too)
      const int64_t ranks = Su * Sv < 65535 ? Su * Sv : 65535;
      const int64_t bins = ranked && ranks > GB_MAX_U8_BINS ? ranks : GB_MAX_U8_BINS;
      int64_t bytes = tile_bytes_needed((int)Su, (int)Sv, tile_w, tile_h, (int)bins, tile_w * tile_h) + 16;
      bytes += bspline_band_bytes((int)(Su - tile_w + 1), (int)(Sv - tile_h + 1), 5, 5) + 16;
      if (ranked) bytes += bins * 8 + 16;
      const int64_t ta = (int64_t)tile_w * tile_h;
      if (ta > GB_SMEM_TEMPLATE) {
        bytes += ta * 4 + 16;                       // the template's column-major copy behind the window's data
        if (bytes < ta * 8) bytes = ta * 8;         // k_template's grey values of a ranked template
      }
      plan->surf_bytes = (bytes + 255) / 256 * 256;
    }
    // Points are independent: they are cut into `slots` batches that advance on their own side streams, so the
    // low-occupancy tails of one batch's kernels (a few very large search windows) overlap the other batches' work.
    // (Batches small enough to keep the intermediates L2-resident were measured slower: launch-bound.)
    // Fewer batches for few points, where a batch no longer fills the device and every extra launch shows: measured (40
    // frames, ms per track, 1 / 2 / 4 batches) 10 points 1.31 / 1.36 / 2.40 (20 frames), 100 points 5.96 / 5.67 / 5.74,
    // 250 points 8.76 / 7.99 / 7.85, 500 points 14.3 / 12.8 / 12.7 — a batch should hold at least ~50 points.
    int slots = (int)(npoints / 50);
    if (slots < 1) slots = 1;
    if (slots > 4) slots = 4;
    int64_t batch = (npoints + slots - 1) / slots;
    if (const char* e = getenv("GB_STREAM_BATCH")) batch = atoll(e);   // tuning overrides
    if (const char* e = getenv("GB_STREAM_SLOTS")) slots = atoi(e);
    if (batch < 1) batch = 1;
    if (batch > npoints) batch = npoints;
    if (batch > 65535) batch = 65535;  // a batch is the y extent of the k_s4p grid
    if (slots < 1) slots = 1;
    if (slots > kMaxSlots) slots = kMaxSlots;
    plan->stream_batch = (int32_t)batch;
    plan->stream_slots = slots;
    plan->scratch_bytes = stream_layout(npoints, n_particles, n_observers, plan->stream_nblk, plan->surf_bytes).total;
    return GB_OK;
  }
  return fail(GB_E_INVALID, "unknown mode%s");
}

int gb_track_init(const gb_track_desc* d, int32_t t, void* stream) {
  if (!d) return fail(GB_E_INVALID, "null descriptor%s");
  int rc = check_desc(*d);
  if (rc) return rc;
  if (t < 0 || t >= d->T) return fail(GB_E_INVALID, "time index out of range%s");
  if ((rc = ensure_device())) return rc;
  StepParams prm;
  fill_params(*d, t, prm);
  int64_t launches = 0;
  if ((rc = launch_init(prm, d->covariances != nullptr, (cudaStream_t)stream, launches))) return rc;
  return launch_template(*d, prm, (cudaStream_t)stream, launches);
}

int gb_track_step(const gb_track_desc* d, int32_t t, const gb_stage_io* io, void* stream) {
  if (!d) return fail(GB_E_INVALID, "null descriptor%s");
  int rc = check_desc(*d);
  if (rc) return rc;
  if (t < 1 || t >= d->T) return fail(GB_E_INVALID, "time index out of range%s");
  if ((rc = ensure_device())) return rc;
  if ((rc = ensure_tensor_maps(*d))) return rc;
  StepParams prm;
  fill_params(*d, t, prm);
  if (io) prm.io = *io;
  FrameMaps fm;
  frame_maps(prm, fm);
  const bool cov = d->covariances != nullptr;
  int64_t launches = 0;
  SideStreams sides(*d, (cudaStream_t)stream);
  if ((rc = sides.open()) || (rc = sides.fork()) || (rc = sides.wait_frames(prm))) return rc;
  rc = sides.each_batch(prm, [&](const StepParams& b, cudaStream_t s) {
    return cov ? step_batch<true>(b, fm, s, launches) : step_batch<false>(b, fm, s, launches);
  });
  return rc ? rc : sides.join();
}

int gb_track(const gb_track_desc* d, void* stream, int64_t* launches_out) {
  if (!d) return fail(GB_E_INVALID, "null descriptor%s");
  int rc = check_desc(*d);
  if (rc) return rc;
  if (!d->mask_host || !d->first_host || !d->last_host) return fail(GB_E_INVALID, "host copies of mask/first/last required%s");
  if ((rc = ensure_device())) return rc;
  if ((rc = ensure_tensor_maps(*d))) return rc;
  int64_t launches = 0;
  if ((rc = track(*d, (cudaStream_t)stream, launches))) return rc;
  if (launches_out) *launches_out = launches;
  return GB_OK;
}

int gb_evolve(const gb_motion* motion, const gb_surface* surfaces, int64_t P, int64_t N, double tau, double tau2,
              const double* normals, double* state, int32_t* status, void* stream) {
  if (!motion || !normals || !state || P <= 0 || N <= 0) return fail(GB_E_INVALID, "bad arguments%s");
  dim3 grid((unsigned)grid_for(N, 256), (unsigned)P, 1);
  k_evolve<<<grid, 256, 0, (cudaStream_t)stream>>>(motion, surfaces, P, N, tau, tau2, normals, N * 3, state, nullptr, nullptr, status,
                                                   nullptr, 0, GB_RNG_SUPPLIED, 0, 0, 0);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_init_particles(const gb_motion* motion, const gb_surface* surfaces, int64_t P, int64_t N, const double* normals, double* state,
                      int32_t* status, void* stream) {
  if (!motion || !surfaces || !normals || !state || P <= 0 || N <= 0 || P > 65535) return fail(GB_E_INVALID, "bad arguments%s");
  dim3 grid((unsigned)grid_for(N, 256), (unsigned)P, 1);
  k_init_particles<<<grid, 256, 0, (cudaStream_t)stream>>>(motion, surfaces, N, normals, state, status);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_motion_log_likelihoods(const gb_motion* motion, const gb_surface* surfaces, int64_t P, int64_t N, const double* state, double* ll,
                              int32_t* status, void* stream) {
  if (!motion || !surfaces || !state || !ll || P <= 0 || N <= 0 || P > 65535) return fail(GB_E_INVALID, "bad arguments%s");
  dim3 grid((unsigned)grid_for(N, 256), (unsigned)P, 1);
  k_motion_log_likelihoods<<<grid, 256, 0, (cudaStream_t)stream>>>(motion, surfaces, N, state, ll, status);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_sample_surface(const double* tile, int32_t rows, int32_t cols, int32_t kx, int32_t ky, const double* xy, int64_t n, void* work,
                      double* out, void* stream) {
  if (!tile || !xy || !work || !out || n <= 0) return fail(GB_E_INVALID, "bad arguments%s");
  if (kx < 1 || kx > 5 || ky < 1 || ky > 5) return fail(GB_E_INVALID, "spline degrees 1 to 5 are supported%s");
  if (rows < kx + 1 || cols < ky + 1 || rows > GB_MAX_SURFACE || cols > GB_MAX_SURFACE)
    return fail(GB_E_INVALID, "tile must have between degree + 1 and 1024 cells per axis%s");
  int rc = ensure_device();
  if (rc) return rc;
  k_sample_surface<<<1, 256, 0, (cudaStream_t)stream>>>(tile, cols, rows, ky, kx, xy, n, reinterpret_cast<float4*>(work), out);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_moments(const double* particles, const double* weights, int64_t n, double* mean, double* sigma, double* cov,
               void* stream) {
  if (!particles || !weights || !mean || n <= 0) return fail(GB_E_INVALID, "bad arguments%s");
  k_moments<<<1, GB_THREADS, kHeaderBytes, (cudaStream_t)stream>>>(particles, weights, n, mean, sigma, cov);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

int gb_philox_draws(uint64_t seed, uint64_t point, uint32_t time, uint32_t first_particle, int64_t n, int32_t kind, int32_t rng_stream,
                    void* out, void* stream) {
  if (!out || n <= 0 || n > ((int64_t)1 << 32) || kind < GB_DRAW_WORDS || kind > GB_DRAW_UNIFORM_PARTICLE || rng_stream < 0 ||
      rng_stream > 255)
    return fail(GB_E_INVALID, "bad arguments%s");
  k_philox_draws<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(seed, point, time, first_particle, n, kind, (uint32_t)rng_stream,
                                                                     out);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

}  // extern "C"
