/* glimpse_b200 — C ABI of the B200-native `glimpse.Tracker` hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / C++ types.  Every entry point
 * names the reference interface it replaces (paths relative to /root/reference/src/glimpse).  The
 * Python host layer (`glimpse_b200/`) binds these with ctypes; INTEGRATION.md shows the stub a
 * reference maintainer would add.
 *
 * Conventions
 *  - All functions return 0 on success, a negative GB_E_* code on API misuse / CUDA failure
 *    (text via gb_last_error()).  Per-point algorithmic failures (the reference's exceptions) are
 *    reported in `status[P]` as positive GB_ST_* codes, never by the return value.
 *  - Pointers are DEVICE pointers unless the parameter name ends in `_host`.  The caller owns every
 *    buffer; the library keeps no pointer after a call returns and never frees caller memory.
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are stream-ordered
 *    and asynchronous unless stated otherwise.
 *  - Particle state layout ("SoA"): double state[P][6][N], component-major (x, y, z, vx, vy, vz),
 *    so a warp reads 32 consecutive particles of one component.  The reference's (n, 6) row-major
 *    arrays (track/tracker.py:37-38) are converted with gb_state_from_rows / gb_state_to_rows.
 */
#ifndef GLIMPSE_B200_H
#define GLIMPSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GB_VERSION 1

/* ---- return codes ---- */
#define GB_OK 0
#define GB_E_INVALID (-1)   /* bad argument */
#define GB_E_CUDA (-2)      /* CUDA runtime error */
#define GB_E_RESOURCE (-3)  /* problem does not fit the on-chip layout (see gb_step_plan) */

/* ---- per-point status (reference exceptions on the path; SURVEY.md §5) ---- */
#define GB_ST_OK 0
#define GB_ST_NOT_VISIBLE 1     /* ValueError: particles on non-visible viewshed cells (tracker.py:114-117) */
#define GB_ST_NAN 2             /* ValueError: particles have missing (NaN) values (tracker.py:118-119) */
#define GB_ST_DEM_BOUNDS 3      /* ValueError: sampling coordinates out of bounds (raster.py:961-973) */
#define GB_ST_SAMPLE_OUTSIDE 4  /* ValueError: sampling points are outside box (observer.py:201-202) */
#define GB_ST_TEMPLATE_BOUNDS 5 /* IndexError: box extends beyond grid bounds (raster.py:417-418) */
#define GB_ST_WINDOW_TOO_LARGE 6 /* search window exceeds the on-chip tile capacity of this launch plan */

/* ---- per-(point, time, observer) flags ---- */
#define GB_OBS_USED 0
#define GB_OBS_NO_IMAGE 1    /* masked or no matching image (tracker.py:574-575) */
#define GB_OBS_OUT_OF_FRAME 2 /* warning: particles too close to or beyond image bounds (tracker.py:597-601) */

#define GB_MOTION_CARTESIAN 0   /* track/motion.py:92-204 */
#define GB_MOTION_CYLINDRICAL 1 /* track/motion.py:207-311 */
#define GB_MOTION_TANGENT_CARTESIAN 2   /* track/motion.py:314-420 */
#define GB_MOTION_TANGENT_CYLINDRICAL 3 /* track/motion.py:423-522 */

#define GB_RESAMPLE_SYSTEMATIC 0 /* tracker.py:168-176: one uniform per update */
#define GB_RESAMPLE_STRATIFIED 1 /* tracker.py:178-186: one uniform per particle and update */
#define GB_RESAMPLE_CHOICE 2     /* tracker.py:205-209: np.random.choice with replacement = inverse-CDF sampling, one uniform per particle */
#define GB_RESAMPLE_RESIDUAL 3   /* tracker.py:188-203: int(n w) copies of every particle, the rest by np.searchsorted on the cumulative
                                  * residuals exactly as the reference computes them; uniforms [P][S][N], the first n - sum(int(n w)) used */

#define GB_RNG_SUPPLIED 0 /* normals / uniforms provided in the reference's draw order */
#define GB_RNG_PHILOX 1   /* counter-based Philox4x32-10 on device */

/* What gb_philox_draws writes */
#define GB_DRAW_WORDS 0              /* uint32 [n][4]: the four Philox4x32-10 output words */
#define GB_DRAW_NORMALS 1            /* double [n][3]: the three float32 Box-Muller normals of those words */
#define GB_DRAW_UNIFORM 2            /* double [n]: the systematic resampler's uniform (stream 3) */
#define GB_DRAW_UNIFORM_PARTICLE 3   /* double [n]: the per-particle uniform of the other resamplers (stream 4) */

/* Camera of one image, already lowered from the reference's 20-vector
 * [xyz, viewdir, imgsz, f, c, k1..k6, p1, p2] (camera.py:101,127-198): R is `Camera.R`
 * (camera.py:239-280), cc = imgsz / 2 + c (camera.py:1507).  corr_* implement
 * helpers.elevation_corrections (helpers.py:1771-1790): dz += corr_c1 * d2 / corr_c2 with
 * corr_c1 = refraction - 1 and corr_c2 = 2 * radius; has_corr = 0 disables it. */
typedef struct gb_camera {
  double R[9];
  double xyz[3];
  double f[2];
  double cc[2];
  double k[6];
  double p[2];
  double corr_c1, corr_c2;
  int32_t imgsz[2];
  int32_t has_corr;
  int32_t affine;                  /* 1 = a raster observer (an orthoimage on a regular grid, raster.py:423-459):
                                    * u = (x - xyz[0]) / f[0], v = (y - xyz[1]) / f[1] with xyz = (xlim[0], ylim[0], -) and
                                    * f = the signed cell size d; z, R, cc, k, p are unused */
} gb_camera;

/* One cached frame (image.py:137-214 with cache=True): the pixel array exactly as the host holds it, (height, width, nchan)
 * row-major with `pitch` BYTES per row, of type `dtype`.  uint8 frames (the usual case) are summed over their bands on the fly
 * (tile.mean(axis=2), tracker.py:523-524, is that sum / nchan) and take the integer tile pipeline; the other types take a rank
 * pipeline (every window pixel is replaced by the number of window pixels below it — CDF matching and the median only depend on
 * the order).  No converted copy of a frame is ever written. */
#define GB_PIX_U8 0
#define GB_PIX_U16 1
#define GB_PIX_F32 2
#define GB_PIX_F64 3
typedef struct gb_image {
  const uint8_t* pixels;
  int32_t width, height, pitch, nchan;
  int32_t dtype;                   /* GB_PIX_* */
  int32_t pad_;
  gb_camera cam;
} gb_image;

/* DEM / DEM-sigma / viewshed raster in point-sampling form (raster.py:891-1027).  A constant
 * surface (reference 0-D raster, motion.py:136-141) has z == NULL and returns `value` everywhere.
 * Otherwise z[ix * ny + iy] on cell centres x0 + ix * dx, y0 + iy * dy (dx, dy > 0, increasing),
 * and [xmin, xmax] x [ymin, ymax] are the outer limits used for the bounds error. */
typedef struct gb_surface {
  const double* z;
  int32_t nx, ny;
  double x0, dx, y0, dy;
  double xmin, xmax, ymin, ymax;
  double value;
} gb_surface;

/* Motion-model parameters of one tracked point (CartesianMotion motion.py:122-147 /
 * CylindricalMotion motion.py:239-258 / TangentCartesianMotion motion.py:350-376 /
 * TangentCylindricalMotion motion.py:457-483).  For the cylindrical kinds v/a are (vr, theta, vz) and
 * (ar, dtheta/dt, az); the tangent kinds use the first two components of v/a (the third must be 0) and
 * slope_sigma.  dem / dem_sigma index the `surfaces` table of the call. */
typedef struct gb_motion {
  int32_t kind;
  int32_t dem, dem_sigma;
  int32_t pad_;
  double xy[2], xy_sigma[2];
  double v[3], v_sigma[3];
  double a[3], a_sigma[3];
  double slope_sigma; /* tangent kinds: sigma of the slope of small-scale features (motion.py:345-346) */
} gb_motion;

/* ------------------------------------------------------------------------------------------
 * Library
 * ------------------------------------------------------------------------------------------ */
int gb_version(void);
const char* gb_last_error(void);
/* sizeof() of the public structs as this library was compiled, so that a binding can verify its mirror of the layouts:
 * which = 0 gb_camera, 1 gb_image, 2 gb_surface, 3 gb_motion, 4 gb_plan, 5 gb_track_desc, 6 gb_stage_io; -1 for anything else. */
int64_t gb_struct_size(int32_t which);

/* Measurement aid (no reference counterpart): when enabled, every kernel launch of gb_track's streaming
 * flow is bracketed by CUDA events on the stream it is launched on; gb_kernel_timing_read returns the
 * accumulated milliseconds and launch counts per kernel kind, index = GB_KERNEL_*.  Enabling resets the sums. */
#define GB_KERNEL_ACTIVITY 0            /* k_s0p_activity */
#define GB_KERNEL_SURFACE 1             /* k_s2_surface */
#define GB_KERNEL_WEIGHTS 2             /* k_s3_weights */
#define GB_KERNEL_RESAMPLE_PROPAGATE 3  /* k_s4p_resample_propagate */
#define GB_KERNEL_FINALIZE 4            /* k_s5p_finalize */
#define GB_KERNEL_INIT 5                /* k_init */
#define GB_KERNEL_TEMPLATE 6            /* k_template */
#define GB_KERNEL_PUBLISH 7             /* k_s3b_publish */
#define GB_KERNEL_KINDS 8
int gb_kernel_timing(int32_t enable);
int gb_kernel_timing_read(double* ms, int64_t* launches, int32_t n);
/* Build a gb_camera from the reference 20-vector on the host (libm sin/cos).  corr_host = {radius,
 * refraction} or NULL.  Replaces Camera.__init__ + Camera.R (camera.py:74-123, 239-280). */
int gb_camera_from_vector(const double* vec20_host, const double* corr_host, gb_camera* out_host);

/* ------------------------------------------------------------------------------------------
 * Camera (stage entry points; also used by the host-side Camera class)
 * ------------------------------------------------------------------------------------------ */
/* Camera.xyz_to_uv (camera.py:591-628): xyz[n][3] -> uv[n][2]; NaN behind the camera. */
int gb_project(const gb_camera* cam_host, const double* xyz, int64_t n, double* uv, void* stream);
/* Camera.uv_to_xyz (camera.py:630-663): uv[n][2] -> xyz[n][3].  depth == NULL means depth 1;
 * otherwise depth[n].  directions != 0 returns ray directions, else adds the camera position. */
int gb_unproject(const gb_camera* cam_host, const double* uv, int64_t n, int directions, const double* depth,
                 double* xyz, void* stream);

/* Image.project (image.py:301-361): resample a frame into the frame of another camera at the same position (sequence
 * stabilisation warps; also optimize.project_images, optimize.py:2776-2872).  src_host->pixels is device memory; out is device
 * memory of dst_cam_host->imgsz[1] x imgsz[0] x src nchan pixels of the source's type.  method 0 = 'nearest', 1 = 'linear'
 * (scipy.interpolate.RegularGridInterpolator on pixel centres); pixels that fall outside the source are NaN (0 in an integer
 * frame).  GB_E_INVALID if the cameras' positions differ (the reference's ValueError). */
int gb_project_image(const gb_image* src_host, const gb_camera* dst_cam_host, int32_t method, void* out, void* stream);

/* Frame ingest (Image.read, image.py:137-214: the reference decodes through GDAL / libjpeg on the host): a JPEG stream in HOST
 * memory decoded by nvJPEG straight into device memory, `out` = height x width x nchan uint8 (nchan 3: interleaved RGB, 1: luma),
 * the layout gb_image describes.  The library is opened at run time (GB_E_RESOURCE if it is not installed); decoders differ in
 * their IDCT and chroma upsampling, so the pixels are within a few grey levels of libjpeg's, not identical.  gb_jpeg_info reads the
 * size and the number of bands (1 or 3) of a stream.  The decode is asynchronous on `stream`; jpeg_host must stay valid until then. */
int gb_jpeg_info(const uint8_t* jpeg_host, int64_t nbytes, int32_t* width, int32_t* height, int32_t* nchan);
int gb_decode_jpeg(const uint8_t* jpeg_host, int64_t nbytes, int32_t width, int32_t height, int32_t nchan, uint8_t* out, void* stream);

/* Raster.viewshed (raster.py:1293-1389): cells of the DEM z (ny x nx doubles, row-major, device memory) visible from
 * origin_host = (x, y, z).  x_centres[nx] / y_centres[ny] (device) are the cell-centre coordinates in array order (Grid.x, Grid.y,
 * raster.py:139-174), cell = |d[0]|, corr_host = {radius, refraction} or NULL (helpers.elevation_corrections).  max_rings bounds
 * the number of distance rings between the nearest and the farthest cell (the host knows it from the raster's corners); work =
 * gb_viewshed_work_bytes(nx, ny, max_rings) bytes of device scratch (64 per cell, 12 per ring and 2 KB) whose first int32 is the
 * status the caller reads back after the stream: 0 ok, 2 more rings than max_rings.  Rings of any size; GB_E_RESOURCE, before
 * any device work, for more than 2^31 cells.  The call only enqueues work on `stream`.  visible[ny * nx] = 1 / 0.
 * Test hook: the environment variable GB_VS_RING_CAP (1 up to the default capacity) lowers the number of cells a ring may have
 * before it takes the large-ring sort and horizon search; the result is the same. */
int64_t gb_viewshed_work_bytes(int32_t nx, int32_t ny, int32_t max_rings);
int gb_viewshed(const double* z, int32_t nx, int32_t ny, const double* x_centres, const double* y_centres, double cell,
                const double* origin_host, const double* corr_host, int32_t max_rings, void* work, int64_t work_bytes,
                uint8_t* visible, void* stream);

/* ------------------------------------------------------------------------------------------
 * State layout helpers
 * ------------------------------------------------------------------------------------------ */
int gb_state_from_rows(const double* rows, int64_t npoints, int64_t n, double* state, void* stream);
int gb_state_to_rows(const double* state, int64_t npoints, int64_t n, double* rows, void* stream);

/* ------------------------------------------------------------------------------------------
 * The filter
 * ------------------------------------------------------------------------------------------ */
/* Device organisation of an update: kernels over all points.  gb_track pipelines them: per update and batch of points
 *   [k_s0p_activity ->] k_s2_surface -> k_s3_weights -> k_s3b_publish -> k_s4p_resample_propagate (the resampling of
 *   time t fused with the motion step to t + 1) -> k_s5p_finalize, batches on their own streams; gb_track_step runs the
 *   same stages unfused so that intermediates can be forced / dumped.
 * (Mode 0 was round 1's cluster-per-point kernel, which kept a point's particles in distributed shared memory; it ran at
 *  a third of this organisation's rate and was removed.  gb_step_plan rejects it.) */
#define GB_MODE_STREAM 1

/* Launch plan chosen by gb_step_plan: cluster size (CTAs per tracked point), threads per CTA,
 * dynamic shared memory and how it is split between particle arrays and tile buffers. */
typedef struct gb_plan {
  int32_t cluster;          /* CTAs per point (1, 2, 4 or 8) */
  int32_t threads;          /* threads per CTA */
  int32_t n_local;          /* particles per CTA */
  int32_t particles_in_smem; /* 1: evolved state / uv / weights live in shared memory; 0: in `scratch` */
  int32_t smem_bytes;       /* dynamic shared memory per CTA */
  int32_t tile_bytes;       /* bytes of it available to the tile pipeline (GB_MODE_STREAM: shared memory one search window may use
                             * in k_s2_surface; negative = skip the interleaved organisation, parity tests) */
  int32_t max_template;     /* template pixels the plan was sized for */
  int32_t n_slabs;          /* per-SM overflow slabs for search windows that do not fit tile_bytes */
  int64_t slab_bytes;       /* bytes per slab (windows up to 256 + template - 1 pixels a side) */
  int64_t particle_scratch_bytes; /* global particle arrays when !particles_in_smem */
  int64_t scratch_bytes;    /* total global scratch the caller must provide */
  int32_t mode;             /* GB_MODE_* */
  int32_t stream_block;     /* GB_MODE_STREAM: particles per CTA of the per-particle kernels (even, <= 768) */
  int32_t stream_nblk;      /* GB_MODE_STREAM: CTAs per point */
  int32_t n_observers;      /* observer slots (1-8): one per observer in a call of up to GB_MAX_OBSERVERS observers, otherwise
                             * at least the most observers with a frame at the same time */
  int64_t surf_bytes;       /* GB_MODE_STREAM: bytes of the per-(point, slot) surface region */
  int32_t stream_batch;     /* GB_MODE_STREAM: points per batch (<= 65535) */
  int32_t stream_slots;     /* GB_MODE_STREAM: batches in flight (side streams / scratch slots) */
} gb_plan;

/* Border modes of the median high-pass (Tracker.highpass['mode'], scipy.ndimage: d c b a | a b c d | d c b a is 'reflect'). */
#define GB_HP_REFLECT 0
#define GB_HP_CONSTANT 1
#define GB_HP_NEAREST 2
#define GB_HP_MIRROR 3
#define GB_HP_WRAP 4

/* Observers with a frame at the same time: the cameras of one time step travel as kernel launch parameters (operands straight
 * from the constant bank), which bounds their number.  A call may have any number of observers (d.O).  Up to
 * GB_MAX_OBSERVERS observers, every observer has a slot of its own (plan n_observers = O); beyond, each time step gives its
 * observers with a frame (image_index_host >= 0) the slots in ascending observer order, and the plan needs as many slots as
 * the most such observers at one time.  gb_track* return GB_E_RESOURCE when more than GB_MAX_OBSERVERS observers have a frame
 * at one time, GB_E_INVALID for a plan with fewer slots than that.  Templates, masks, obs_flags, window_stats and the
 * gb_stage_io dumps stay indexed by observer. */
#define GB_MAX_OBSERVERS 8

/* Size a launch plan for N particles per point, a w x h template, P points and n_observers observer slots (see GB_MAX_OBSERVERS).
 * `flags`: GB_PLAN_RANKED_FRAMES = some frame is not uint8 (the surface regions are sized for rank histograms of the largest window);
 * GB_PLAN_LARGE_TEMPLATES = admit templates above 1024 pixels, up to 128 pixels a side (without it they return GB_E_RESOURCE;
 * with it a template above 1024 pixels and above 128 pixels a side still does).  The kernels choose their path from the template
 * size, not from the flag; gb_track* accept a template above 1024 pixels only with a plan whose max_template covers it.
 * `mode` must be GB_MODE_STREAM.
 * Plan fields that only that organisation used (cluster, particles_in_smem, n_slabs, slab_bytes, particle_scratch_bytes) are 1 / 0. */
#define GB_PLAN_RANKED_FRAMES 1
#define GB_PLAN_LARGE_TEMPLATES 2
int gb_step_plan(int64_t n_particles, int32_t tile_w, int32_t tile_h, int64_t npoints, int32_t n_observers,
                 int32_t flags, int32_t mode, gb_plan* plan_host);
/* The same with the capacity of the search windows chosen by the caller: in GB_MODE_STREAM every (point, observer) owns a surface
 * region sized for windows up to `window_margin` px larger than the template per axis (gb_step_plan: 191; 4..1023).  A point whose
 * particle cloud outgrows it ends with GB_ST_WINDOW_TOO_LARGE; the Tracker then re-runs that point with the largest margin. */
int gb_step_plan_ex(int64_t n_particles, int32_t tile_w, int32_t tile_h, int64_t npoints, int32_t n_observers,
                    int32_t flags, int32_t mode, int32_t window_margin, gb_plan* plan_host);

/* Everything one Tracker.track call needs (track/tracker.py:225-417).  Shapes use P points,
 * N particles, T times, O observers, S = T - 1 update steps, w x h template. */
typedef struct gb_track_desc {
  int64_t P, N;
  int32_t T, O;
  int32_t tile_w, tile_h;

  /* frames and cameras: images[image_offset_host[o] + i] is image i of observer o */
  const gb_image* images;          /* device array */
  const gb_image* images_host;     /* host copy of the same table (cameras travel to the kernels as launch parameters) */
  void* const* image_events_host;  /* optional [n_images] cudaEvent_t: gb_track makes `stream` wait for event i before the first
                                    * kernel that reads image i (lets the caller overlap frame uploads with tracking); NULL = none */
  const int32_t* image_offset_host; /* [O + 1] */
  const int32_t* image_index_host; /* [T][O] image of observer o matched to time t, -1 = none (tracker.py:466-492) */
  const double* obs_scale_host;    /* [O] 1 / (2 sigma^2) (tracker.py:625) */
  const uint8_t* mask;             /* device [P][O] observer mask (tracker.py:289-290) */
  const int32_t* first;            /* device [P] first / last time index with a masked observer image (tracker.py:321-325) */
  const int32_t* last;
  const uint8_t* mask_host;        /* host copies of the three arrays above (drive the per-time launch decisions) */
  const int32_t* first_host;
  const int32_t* last_host;
  const double* tau_host;          /* [S] dt / time_unit (motion.py:173) */
  const double* tau2_host;         /* [S] tau ** 2 as the host language rounds it */

  /* motion models and surfaces */
  const gb_motion* motion;         /* device [P] */
  const gb_surface* surfaces;      /* device table */
  int32_t n_surfaces;
  int32_t viewshed;                /* index into surfaces, -1 = none (tracker.py:114-117) */

  /* random draws */
  int32_t rng_mode;                /* GB_RNG_* */
  int32_t motion_kinds;            /* bit k set = some point has motion kind k; 0 = unspecified (kernels handle every kind) */
  uint64_t seed;                   /* Philox key */
  int64_t point_offset;            /* global index of point 0 (Philox counters use global indices, so results do not depend on sharding) */
  const double* init_normals;      /* supplied: [P][N][6] = randn(N,2) | randn(N) | randn(N,3) per particle */
  const double* step_normals;      /* supplied: [P][S][N][3] */
  const double* uniforms;          /* supplied: [P][S] one np.random.random() per update (systematic) or [P][S][N] np.random.random(N) (stratified, choice) */

  /* work buffers (caller-allocated) */
  double* state_a;                 /* [P][6][N] */
  double* state_b;                 /* [P][6][N] */
  double* weight_state;            /* [P][N] or NULL; required when an observer's template starts after a point's first frame, or with out_weights */
  double* scratch;                 /* plan.scratch_bytes or NULL */
  /* templates (tracker.py:536-561), filled by the call */
  double* tmpl_tile;               /* [P][O][h*w] high-passed template */
  double* tmpl_values;             /* [P][O][h*w] sorted unique normalised values (helpers.py:433-464) */
  double* tmpl_quantiles;          /* [P][O][h*w] */
  int32_t* tmpl_nvalues;           /* [P][O] */
  int32_t* tmpl_box;               /* [P][O][4] left, top, right, bottom */
  double* tmpl_duv;                /* [P][O][2] */

  /* outputs (caller pre-fills floating outputs with NaN, as tracker.py:306-313 does) */
  double* means;                   /* [P][T][6] */
  double* sigmas;                  /* [P][T][6] or NULL */
  double* covariances;             /* [P][T][36] or NULL */
  double* out_particles;           /* [P][T][N][6] or NULL (return_particles) */
  double* out_weights;             /* [P][T][N] or NULL */
  int32_t* status;                 /* [P] GB_ST_*; must be zero on entry */
  int32_t* status_time;            /* [P] time index at which status was raised */
  uint8_t* obs_flags;              /* [P][T][O] GB_OBS_* */
  int32_t* window_stats;           /* [P][T][O][2] realised search-window (width, height), or NULL */

  int32_t resample_method;         /* GB_RESAMPLE_* (Tracker.resample_method, tracker.py:151-223) */
  int32_t highpass_size;           /* rows | columns << 16 of the median high-pass (Tracker.highpass['size'], tracker.py:59, 530:
                                    * scipy.ndimage.median_filter(tile, size=(rows, columns)), 1..31 each); 0 = the default 5 x 5 */
  int32_t interp_rows, interp_cols; /* Tracker.interpolation (tracker.py:60, observer.py:210): degree of the interpolating spline along the rows
                                    * (kx) and the columns (ky) of the SSE surface, which also sets the minimum surface size (tracker.py:584-594).
                                    * 1 to 5 (3 = cubic not-a-knot and 1 = piecewise linear in Hermite form, 2 / 4 / 5 as B-spline coefficients on
                                    * FITPACK's knots); 0 = the default 3 */
  int32_t highpass_mode;           /* border mode of the median high-pass (scipy.ndimage.median_filter's `mode`): GB_HP_* */
  int32_t highpass_origin;         /* its `origin` as (rows & 0xffff) | (columns & 0xffff) << 16, each a signed 16-bit shift of the window:
                                    * the window of pixel i spans i - size / 2 - origin ... (0 = centred, the default) */
  double highpass_cval;            /* value beyond the border with GB_HP_CONSTANT (`cval`), in the units of the filtered tile */
  const uint32_t* highpass_footprint_host; /* host, or NULL = the full window: `footprint` of the filter, one word per window row (bit b =
                                    * column b takes part); highpass_size is then the footprint's shape and the rank is (cells set) / 2 */
  double* final_weights;           /* [N] or NULL: weights of point P - 1's resampled particles at its last time — what Tracker.weights holds
                                    * after track() in the reference (tracker.py:62-70, 216-223: the state of the last processed track);
                                    * the caller pre-fills it with ones (a point that is never updated keeps its initial weights) */
  gb_plan plan;
} gb_track_desc;

/* Tracker.track for all points, all times (tracker.py:225-417): enqueues the per-time kernels on
 * `stream` and returns without synchronising.  `kernel_launches_host` (optional) receives the
 * number of kernels launched. */
int gb_track(const gb_track_desc* desc_host, void* stream, int64_t* kernel_launches_host);

/* ------------------------------------------------------------------------------------------
 * Teacher-forced stage entry point for parity tests
 * ------------------------------------------------------------------------------------------ */
/* Runs ONE update of the production step kernel for `P` points at time index `t` with any subset
 * of its intermediate values forced to caller-supplied ones and/or dumped:
 *   force_evolved  [P][6][N]   use these particles instead of evolving state_a (a3/a4 skipped)
 *   force_weights  [P][N]      use these weights instead of exp(-ll) (a8..a16 skipped)
 *   dump_evolved   [P][6][N]   particles after the motion step (motion.py:165-179)
 *   dump_uv        [P][O][N][2]  projected particles (camera.py:591-628)
 *   dump_box       [P][O][4]   search window (tracker.py:576-595)
 *   dump_search    [P][O][cap] high-passed, CDF-matched search tile as float32 (tracker.py:605-611)
 *   dump_sse       [P][O][cap] area-normalised SSE surface, float32 (tracker.py:609-614)
 *   dump_sampled   [P][O][N]   spline-sampled SSE (observer.py:178-214)
 *   dump_weights   [P][N]      weights before resampling (tracker.py:145-149)
 *   dump_indices   [P][N]      resampled ancestor indices (tracker.py:168-176)
 *   dump_clocks    [P][16]     clock64() of rank-0 CTA at the phase boundaries of the step (profiling aid)
 * Any pointer may be NULL.  `dump_cap` is the per-(point, observer) capacity of dump_search/dump_sse. */
typedef struct gb_stage_io {
  const double* force_evolved;
  const double* force_weights;
  double* dump_evolved;
  double* dump_uv;
  int32_t* dump_box;
  float* dump_search;
  float* dump_sse;
  double* dump_sampled;
  double* dump_weights;
  int32_t* dump_indices;
  int64_t* dump_clocks;
  int64_t dump_cap;
} gb_stage_io;

int gb_track_step(const gb_track_desc* desc_host, int32_t t, const gb_stage_io* io_host, void* stream);
/* First-frame initialisation (motion.py:149-163, 260-283 + tracker.py:327-330) for points whose
 * first time index is `t`, and template construction (tracker.py:536-561) for templates due at t. */
int gb_track_init(const gb_track_desc* desc_host, int32_t t, void* stream);

/* Motion.evolve_particles as a stand-alone call (motion.py:165-179, 285-311, 392-420, 507-522) on SoA
 * state [P][6][N] in place; normals[P][N][3] supplied (tangent kinds: columns 0-1 = the randn(n,2) draw,
 * column 2 = the randn(n) draw).  `surfaces` is the table motion[].dem indexes (may be NULL when no model is
 * tangent); status[P] (may be NULL) receives GB_ST_DEM_BOUNDS where a tangent model sampled its DEM out of bounds. */
int gb_evolve(const gb_motion* motion, const gb_surface* surfaces, int64_t P, int64_t N, double tau, double tau2,
              const double* normals, double* state, int32_t* status, void* stream);
/* Motion.initialize_particles as a stand-alone call (motion.py:149-163, 260-283, 378-390, 485-505): state [P][6][N] from
 * normals[P][N][6] in the reference's draw order — randn(n,2) -> columns 0-1 (xy), randn(n) -> column 2 (z), randn(n,3) -> columns
 * 3-5 (velocity; tangent kinds: randn(n,2) in columns 3-4, column 5 unused).  status[P] (may be NULL, zero on entry) receives
 * GB_ST_DEM_BOUNDS where the DEM or its sigma was sampled out of bounds (raster.py:961-973). */
int gb_init_particles(const gb_motion* motion, const gb_surface* surfaces, int64_t P, int64_t N, const double* normals, double* state,
                      int32_t* status, void* stream);
/* Motion.compute_log_likelihoods as a stand-alone call (motion.py:181-204): ll[P][N] = (dem(xy) - z)^2 / (2 sigma(xy)^2), 0 where
 * sigma is 0, for SoA state [P][6][N].  (The tangent kinds return None in the reference, motion.py:77-89: the caller does not ask.) */
int gb_motion_log_likelihoods(const gb_motion* motion, const gb_surface* surfaces, int64_t P, int64_t N, const double* state, double* ll,
                              int32_t* status, void* stream);
/* Observer.sample_tile (observer.py:178-214) as a stand-alone call: the interpolating spline RectBivariateSpline(rows, columns, tile,
 * kx, ky, s = 0) of degree 1 to 5 per axis (3 = FITPACK's not-a-knot cubic), evaluated at n points.  tile[rows][cols] f64 (held as
 * float32 on the device, like the SSE surface it is used for); xy[n][2] = (column, row) coordinates measured from the first cell centre
 * in cell units, clamped to the data sites like FITPACK's evaluation; work = rows * (cols | 1) * 16 + (rows + cols) * 88 bytes; out[n]
 * f64.  All device pointers. */
int gb_sample_surface(const double* tile, int32_t rows, int32_t cols, int32_t kx, int32_t ky, const double* xy, int64_t n, void* work,
                      double* out, void* stream);
/* Tracker.particle_mean / compute_particle_sigma / particle_covariance (tracker.py:72-104) on
 * row-major particles[n][6], weights[n]: mean[6], sigma[6] (or NULL), cov[36] (or NULL). */
int gb_moments(const double* particles, const double* weights, int64_t n, double* mean, double* sigma, double* cov,
               void* stream);
/* The draws of rng_mode = GB_RNG_PHILOX as a stand-alone call, computed by the device functions the track kernels call.
 * Philox4x32-10 with key (seed & 0xffffffff, seed >> 32) and counter (particle, time, point & 0xffffffff,
 * (point >> 32) << 8 | rng_stream); streams: 0 and 1 = the six normals of initialisation, 2 = the normals of every later step,
 * 3 = the systematic resampler's uniform (particle word 0xffffffff), 4 = the per-particle uniform of the stratified, choice and
 * residual resamplers.  Element i of `out` (device memory) is particle first_particle + i (GB_DRAW_WORDS, GB_DRAW_NORMALS with
 * `rng_stream`, GB_DRAW_UNIFORM_PARTICLE) or time `time` + i (GB_DRAW_UNIFORM); 1 <= n <= 2^32. */
int gb_philox_draws(uint64_t seed, uint64_t point, uint32_t time, uint32_t first_particle, int64_t n, int32_t kind, int32_t rng_stream,
                    void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GLIMPSE_B200_H */
