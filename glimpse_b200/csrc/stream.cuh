// GB_MODE_STREAM kernels (included by glimpse_b200.cu after StepParams / Moments are defined).
#pragma once
// (already inside namespace gb)

// ---------------------------------------------------------------------------------------------
// GB_MODE_STREAM: one update as kernels over all points of a batch.  Intermediates (evolved particles, projected
// coordinates, weights, spline surfaces) go through global memory / L2; no kernel has a serial stage across CTAs.
// Step-by-step flow (gb_track_step: every intermediate can be forced / dumped; also gb_track with the 'choice' resampler):
//   s0 reset      activity byte, empty cloud boxes and flags                 (per point)
//   s1 propagate  evolve + test + project + integer cloud box                (per particle)
//   s2 surface    search window + tile pipeline -> Hermite surface           (one CTA per point-observer)
//   s3 weights    spline sample + surface likelihood -> weights, block totals (per particle)
//   s4 resample   prefix of the weights, child ranges, child writes, moment partials (per particle; s4c_* for 'choice')
//   s5 finalise   moments, status                                            (per point)
// Pipelined flow (gb_track; further down): s2, s3 as above, s4 of time t fused with s1 of time t + 1.
// ---------------------------------------------------------------------------------------------
#define GB_SBLOCK_THREADS 256

// Per-point byte written by k_s0_reset: bit 0 = the point is updated at this time, bit 1 = its motion
// model has a non-trivial surface likelihood.  One load instead of a chain of dependent ones.
#define GB_ACT_ACTIVE 1
#define GB_ACT_SURFACE_LL 2
#define GB_ACT_NO_MOTION_LL 8 /* the motion model returns no likelihood at all (tangent kinds) */
__device__ __forceinline__ bool stream_point_active(const StepParams& prm, int64_t p) {
  return (prm.s_act[p] & GB_ACT_ACTIVE) != 0;
}

__global__ void k_s0_reset(const __grid_constant__ StepParams prm) {
  // scratch arrays are indexed by the global point number; the host pre-shifts their base pointers so
  // that the batch [p0, p0 + pb) lands in the batch's slot
  const int64_t lo5 = prm.p0 * prm.slot_stride * 5, n = prm.pb * prm.slot_stride * 5;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    prm.s_ibox[lo5 + i] = (i % 5 == 4) ? 0 : 0x7fffffff;
  for (int64_t i = prm.p0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < prm.p0 + prm.pb; i += (int64_t)gridDim.x * blockDim.x) {
    prm.s_pflags[i] = 0;
    const bool active = prm.status[i] == 0 && prm.t > prm.first[i] && prm.t <= prm.last[i];
    const gb_surface& sg = prm.surfaces[prm.motion[i].dem_sigma];
    const bool tangent = prm.motion[i].kind >= GB_MOTION_TANGENT_CARTESIAN;  // compute_log_likelihoods is None (motion.py:77-89)
    const bool sll = !tangent && !(sg.z == nullptr && sg.value == 0.0);
    prm.s_act[i] = (uint8_t)((active ? GB_ACT_ACTIVE : 0) | (sll ? GB_ACT_SURFACE_LL : 0) | (tangent ? GB_ACT_NO_MOTION_LL : 0));
  }
}

// Warp-transposed reduction of K per-lane doubles (K = 16 or 32): recursive halving, 16 (31) shuffles
// instead of 5 K.  On return lane l holds in v[0] the warp total of value index
// transposed_index(l) = lane bits [4..1] (K = 16, both lanes of a pair) or [4..0] (K = 32).
template <int K>
__device__ __forceinline__ void warp_reduce_transpose(double (&v)[K], int lane) {
#pragma unroll
  for (int half = K / 2, bit = 16; half >= 1; half >>= 1, bit >>= 1) {
    const bool upper = (lane & bit) != 0;
#pragma unroll
    for (int k = 0; k < half; ++k) {
      const double send = upper ? v[k] : v[k + half];
      const double keep = upper ? v[k + half] : v[k];
      v[k] = keep + shfl_xor(send, bit);
    }
  }
  if (K == 16) v[0] += shfl_xor(v[0], 1);
}
template <int K>
__device__ __forceinline__ int transposed_index(int lane) {
  return K == 16 ? (lane >> 1) : lane;
}

// s1: two consecutive particles per thread (16-byte loads / stores), one CTA = s_block particles of a point.
__global__ void __launch_bounds__(GB_SBLOCK_THREADS, 4) k_s1_propagate(const __grid_constant__ StepParams prm) {
  __shared__ gb_motion s_motion;
  __shared__ int s_box[GB_MAX_OBS][5];
  const int64_t p = prm.p0 + blockIdx.x / prm.s_nblk;
  const int b = (int)(blockIdx.x % prm.s_nblk);
  if (!stream_point_active(prm, p)) return;
  const int tid = threadIdx.x, lane = tid & 31;
  const int N = (int)prm.N, ns = prm.n_slots, t = prm.t;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(prm.motion + p);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&s_motion);
    for (int k = tid; k < (int)(sizeof(gb_motion) / 4); k += blockDim.x) dst[k] = src[k];
    if (tid < GB_MAX_OBS * 5) s_box[tid / 5][tid % 5] = (tid % 5 == 4) ? 0 : 0x7fffffff;
  }
  __syncthreads();
  const bool forced = prm.io.force_evolved != nullptr;
  const double* sin_ = forced ? prm.io.force_evolved + p * 6 * (int64_t)N : state_buffer(prm, t - 1) + p * 6 * (int64_t)N;
  double* ev = prm.s_ev + p * 6 * (int64_t)N;
  const int s_idx = t - prm.first[p] - 1;
  const double* zn = prm.step_normals ? prm.step_normals + (((int64_t)p * prm.S + s_idx) * N) * 3 : nullptr;
  const bool evolve = !forced && !prm.skip_evolve;
  const bool use_obs = !prm.io.force_weights;
  const double hw = (double)prm.tile_w * 0.5, hh = (double)prm.tile_h * 0.5;
  const bool vec = (N & 1) == 0;  // 16-byte aligned pairs
  uint32_t flags = 0;
  const int blk_end = min(N, (b + 1) * prm.s_block);  // s_block is even: pairs never straddle CTAs
  for (int sub = 0; sub < prm.s_block; sub += 2 * (int)blockDim.x) {
  const int ia = b * prm.s_block + sub + 2 * tid;  // particles ia, ia + 1
  const bool va = ia < blk_end, vb = ia + 1 < blk_end;
  if (va) {
    double s[2][6];
    if (vec) {
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        const double2 x = __ldcs(reinterpret_cast<const double2*>(sin_ + c * (int64_t)N + ia));  // read once: evict first
        s[0][c] = x.x;
        s[1][c] = x.y;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        s[0][c] = sin_[c * (int64_t)N + ia];
        s[1][c] = vb ? sin_[c * (int64_t)N + ia + 1] : s[0][c];
      }
    }
    if (evolve) {
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        double z0, z1, z2;
        const int i = (q == 1 && !vb) ? ia : ia + q;
        if (prm.rng_mode == GB_RNG_SUPPLIED) {
          z0 = zn[3 * (int64_t)i];
          z1 = zn[3 * (int64_t)i + 1];
          z2 = zn[3 * (int64_t)i + 2];
        } else {
          philox_normals3(prm.seed, (uint64_t)(p + prm.point_offset), (uint32_t)t, (uint32_t)i, 2u, z0, z1, z2, evolve_needs(s_motion));
        }
        evolve_particle(s_motion, prm.surfaces, prm.tau, prm.tau2, z0, z1, z2, s[q], flags);
      }
    }
    flags |= test_particle(prm, s[0]);
    if (vb) flags |= test_particle(prm, s[1]);
    if (vec) {
#pragma unroll
      for (int c = 0; c < 6; ++c) *reinterpret_cast<double2*>(ev + c * (int64_t)N + ia) = make_double2(s[0][c], s[1][c]);
    } else {
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        ev[c * (int64_t)N + ia] = s[0][c];
        if (vb) ev[c * (int64_t)N + ia + 1] = s[1][c];
      }
    }
    if (prm.io.dump_evolved) {
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        prm.io.dump_evolved[((int64_t)p * 6 + c) * N + ia] = s[0][c];
        if (vb) prm.io.dump_evolved[((int64_t)p * 6 + c) * N + ia + 1] = s[1][c];
      }
    }
    if (use_obs) {
      for (int sl = 0; sl < ns; ++sl) {
        const int64_t po = p * prm.O + prm.obs[sl];
        if (prm.img[sl] < 0 || !prm.mask[po]) continue;  // block-uniform
        double* uv = prm.s_uv + (p * prm.slot_stride + sl) * 2 * (int64_t)N;
        double u[2], v[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) project_fast(prm.cam[sl], s[q][0], s[q][1], s[q][2], u[q], v[q]);
        if (!vb) {
          u[1] = u[0];
          v[1] = v[0];
        }
        if (vec) {
          *reinterpret_cast<double2*>(uv + ia) = make_double2(u[0], u[1]);
          *reinterpret_cast<double2*>(uv + (int64_t)N + ia) = make_double2(v[0], v[1]);
        } else {
          uv[ia] = u[0];
          uv[(int64_t)N + ia] = v[0];
          if (vb) {
            uv[ia + 1] = u[1];
            uv[(int64_t)N + ia + 1] = v[1];
          }
        }
        int ib[5];
        ib[4] = (isnan(u[0]) | isnan(v[0]) | isnan(u[1]) | isnan(v[1])) ? -1 : 0;
        ib[0] = min(__double2int_rd(u[0] - hw), __double2int_rd(u[1] - hw));
        ib[1] = min(__double2int_rd(v[0] - hh), __double2int_rd(v[1] - hh));
        ib[2] = -max(__double2int_ru(u[0] + hw), __double2int_ru(u[1] + hw));
        ib[3] = -max(__double2int_ru(v[0] + hh), __double2int_ru(v[1] + hh));
        const unsigned mask = __activemask();
        int red[5], mine = 0x7fffffff;
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          red[k] = __reduce_min_sync(mask, ib[k]);
          if (lane == k) mine = red[k];
        }
        // lanes 0..4 of a warp publish one value each; a tail warp without them lets its first lane do all five
        if ((mask & 0x1fu) == 0x1fu) {
          if (lane < 5) atomicMin(&s_box[sl][lane], mine);
        } else if (lane == (__ffs(mask) - 1)) {
#pragma unroll
          for (int k = 0; k < 5; ++k) atomicMin(&s_box[sl][k], red[k]);
        }
        if (prm.io.dump_uv) {
          double* d = prm.io.dump_uv + (po * N + ia) * 2;
          d[0] = u[0];
          d[1] = v[0];
          if (vb) {
            d[2] = u[1];
            d[3] = v[1];
          }
        }
      }
    }
  }
  }
  __shared__ unsigned s_or;
  const int any = (int)block_or(flags, &s_or);
  if (any && tid == 0) atomicOr(&prm.s_pflags[p], any);
  if (use_obs && tid < ns * 5) {
    const int sl = tid / 5, k = tid - sl * 5;
    if (prm.img[sl] >= 0 && prm.mask[p * prm.O + prm.obs[sl]]) atomicMin(&prm.s_ibox[(p * prm.slot_stride + sl) * 5 + k], s_box[sl][k]);
  }
}

#ifndef GB_S2_THREADS
#define GB_S2_THREADS 512
#endif
#ifndef GB_S2_MINB
#define GB_S2_MINB 2
#endif
// LARGE: templates above GB_SMEM_TEMPLATE pixels, read from the window's global region (TileWork::tcol); launched by template
// size, so that smaller templates run the kernel without that path.
template <bool LARGE>
__global__ void __launch_bounds__(GB_S2_THREADS, GB_S2_MINB) k_s2_surface(const __grid_constant__ StepParams prm, const __grid_constant__ FrameMaps fm,
                                                                 int smem_budget) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double s_mm[GB_S2_THREADS / 32][4];
  __shared__ int s_box[4];
  __shared__ __align__(8) uint64_t s_tma_bar;
  const int64_t p = prm.p0 + blockIdx.x / prm.n_slots;
  const int slot = (int)(blockIdx.x % prm.n_slots), o = prm.obs[slot];
  const int64_t ps = p * prm.slot_stride + slot;  // the slot's scratch: cloud box, meta, projections, surface region
  const int64_t po = p * prm.O + o;               // the observer's template, mask and outputs
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, t = prm.t;
  int* meta = prm.s_meta + ps * 8;
  // profiling aid (gb_track_step only): clock64() of thread 0 at the phase boundaries, window size, SM id
  long long* clk = prm.io.dump_clocks ? reinterpret_cast<long long*>(prm.io.dump_clocks) + po * 16 : nullptr;
  if (clk && tid == 0) clk[0] = clock64();
  if (tid == 0) meta[7] = 0;
  // every scalar the CTA branches on is requested before the first branch: one memory round trip instead of five
  int* gib = prm.s_ibox + ps * 5;
  const int act = prm.s_act[p];
  const int seen = prm.mask[po];
  const int failed = prm.s_pflags[p];
  const int n_values = prm.tmpl_nvalues[po];
  const int my_ib = tid < 5 ? gib[tid] : 0;
  if (!(act & GB_ACT_ACTIVE) || prm.io.force_weights) return;
  uint8_t* oflags = prm.obs_flags + ((int64_t)p * prm.T + t) * prm.O;
  if (prm.n_slots < prm.O && slot == 0)  // observers without a slot have no frame at t: the first slot's CTA flags them
    for (int k = tid; k < prm.O; k += blockDim.x) {
      bool slotted = false;
      for (int q = 0; q < prm.n_slots; ++q) slotted |= prm.obs[q] == k;
      if (!slotted) oflags[k] = GB_OBS_NO_IMAGE;
    }
  uint8_t* oflag = oflags + o;
  if (prm.img[slot] < 0 || !seen) {
    if (tid == 0) *oflag = GB_OBS_NO_IMAGE;
    return;
  }
  if (failed != 0) return;  // the point failed its particle tests: reference raises before any observer work
  const int N = (int)prm.N;
  // consume the integer cloud box and leave it empty for the next time
  __shared__ int s_ib[5];
  if (tid < 5) {
    s_ib[tid] = my_ib;
    gib[tid] = (tid == 4) ? 0 : 0x7fffffff;
  }
  if (tid == 32) {
    mbar_init(&s_tma_bar, 1);
    mbar_fence_init();
  }
  __syncthreads();
  const int* ib = s_ib;
  int box_l = ib[0], box_t = ib[1], box_r = -ib[2], box_b = -ib[3];
  const bool nan_any = ib[4] != 0;
  if (!nan_any && ((box_r - box_l) - prm.tile_w < prm.interp_cols + 2 || (box_b - box_t) - prm.tile_h < prm.interp_rows + 2)) {
    // cloud narrower than the spline degree (the integer box is at most 2 px wider than the exact extents): the reference
    // widens the box from the exact extents (tracker.py:584-594)
    const double* uv = prm.s_uv + ps * 2 * (int64_t)N;
    double mm[4] = {CUDART_INF, CUDART_INF, CUDART_INF, CUDART_INF};
    for (int i = tid; i < N; i += blockDim.x) {
      const double u = uv[i], v = uv[(int64_t)N + i];
      mm[0] = fmin(mm[0], u);
      mm[1] = fmin(mm[1], v);
      mm[2] = fmin(mm[2], -u);
      mm[3] = fmin(mm[3], -v);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double x = warp_min(mm[k]);
      if (lane == 0) s_mm[warp][k] = x;
    }
    __syncthreads();
    if (tid == 0) {
      double e[4];
      for (int k = 0; k < 4; ++k) {
        e[k] = s_mm[0][k];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) e[k] = fmin(e[k], s_mm[w][k]);
      }
      const double hw = (double)prm.tile_w * 0.5, hh = (double)prm.tile_h * 0.5;
      const double tw = (double)prm.tile_w, th = (double)prm.tile_h;
      double bl = sub(e[0], hw), bt = sub(e[1], hh), br = add(-e[2], hw), bb = add(-e[3], hh);
      const double ncols = sub((double)prm.interp_cols, sub(sub(br, bl), tw));
      if (ncols > 0.0) {
        bl = add(bl, mul(-ncols, 0.5));
        br = add(br, mul(ncols, 0.5));
      }
      const double nrows = sub((double)prm.interp_rows, sub(sub(bb, bt), th));
      if (nrows > 0.0) {
        bt = add(bt, mul(-nrows, 0.5));
        bb = add(bb, mul(nrows, 0.5));
      }
      s_box[0] = __double2int_rd(bl);
      s_box[1] = __double2int_rd(bt);
      s_box[2] = __double2int_ru(br);
      s_box[3] = __double2int_ru(bb);
    }
    __syncthreads();
    box_l = s_box[0];
    box_t = s_box[1];
    box_r = s_box[2];
    box_b = s_box[3];
  }
  const int W = prm.cam[slot].c.imgsz[0], H = prm.cam[slot].c.imgsz[1];
  const bool inframe = !nan_any && box_l >= 0 && box_l <= W && box_t >= 0 && box_t <= H && box_r >= 0 && box_r <= W &&
                       box_b >= 0 && box_b <= H;
  if (!inframe) {
    if (tid == 0) *oflag = GB_OBS_OUT_OF_FRAME;
    return;
  }
  TileWork w;
  w.Su = box_r - box_l;
  w.Sv = box_b - box_t;
  w.tw = prm.tile_w;
  w.mh = prm.hp_rows;
  w.mw = prm.hp_cols;
  w.hp_mode = prm.hp_mode;
  w.hp_org_r = prm.hp_org_r;
  w.hp_org_c = prm.hp_org_c;
  w.hp_cval = prm.hp_cval;
  w.hp_fp = prm.hp_has_fp ? prm.hp_fp : nullptr;
  w.cub_u = prm.interp_cols != 1;
  w.cub_v = prm.interp_rows != 1;
  w.ku = prm.interp_cols;
  w.kv = prm.interp_rows;
  w.th = prm.tile_h;
  w.Mu = w.Su - w.tw + 1;
  w.Mv = w.Sv - w.th + 1;
  w.dtype = prm.pixdtype[slot];
  w.nbins = w.dtype == GB_PIX_U8 ? 255 * prm.nchan[slot] + 1 : w.Su * w.Sv;  // grey levels, or ranks of the window's pixels
  w.nvals = n_values;
  w.tmap = fm.ok[slot] ? &fm.map[slot] : nullptr;
  w.bar = &s_tma_bar;
  if (tid == 0) {
    *oflag = GB_OBS_USED;
    if (prm.window_stats) {
      int32_t* ws = prm.window_stats + (((int64_t)p * prm.T + t) * prm.O + o) * 2;
      ws[0] = w.Su;
      ws[1] = w.Sv;
    }
    if (prm.io.dump_box) {
      int32_t* d = prm.io.dump_box + po * 4;
      d[0] = box_l;
      d[1] = box_t;
      d[2] = box_r;
      d[3] = box_b;
    }
  }
  char* region = prm.s_surf + ps * prm.surf_bytes;
  const int64_t need = tile_bytes_needed(w.Su, w.Sv, w.tw, w.th, w.nbins, w.nvals);
  const bool gen = !spline_is_hermite(w.ku, w.kv);  // degrees 2 / 4 / 5: coefficients solved with a work area behind the tile's data
  const bool ranked = w.dtype != GB_PIX_U8;          // frames other than uint8: the window's grey values, likewise
  int64_t tail = align16(need);
  if (gen) {
    w.band = reinterpret_cast<double*>(region + tail);
    tail += align16(bspline_band_bytes(w.Mu, w.Mv, w.ku, w.kv));
  }
  if (ranked) {
    w.vals = reinterpret_cast<double*>(region + tail);
    tail += (int64_t)w.Su * w.Sv * 8;
  }
  const int64_t ta = (int64_t)w.tw * w.th;
  if constexpr (LARGE) {
    // large template: its column-major copy goes behind the tile's data and its CDF tables are read where k_template left them
    tail = align16(tail);
    w.tcol = reinterpret_cast<float*>(region + tail);
    tail += ta * 4;
    w.tq = prm.tmpl_quantiles + po * ta;
    w.tv = prm.tmpl_values + po * ta;
  }
  if (tail > prm.surf_bytes || w.Mu > GB_MAX_SURFACE || w.Mv > GB_MAX_SURFACE || (ranked && w.Su * w.Sv > 65535)) {
    if (tid == 0) atomicOr(&prm.s_pflags[p], (int)GB_F_WINDOW);
    return;
  }
  // Where the window is worked on: in shared memory with the surface interleaved (small windows), in shared memory
  // on planes (windows whose 16-byte cells would not fit, up to ~100 px at 110 KB), in shared memory phase by phase
  // with hand-overs through the global region (up to ~128 px), or entirely in its global region.
  // (A negative budget skips the interleaved path: parity tests of the other paths.)
  const int64_t budget = smem_budget < 0 ? -smem_budget : smem_budget;
  const bool in_smem = smem_budget >= 0 && need <= budget;
  const bool planar = !gen && !in_smem && tile_bytes_needed_planar(w.Su, w.Sv, w.tw, w.th, w.nbins, w.nvals) <= budget;
  const bool staged = !gen && !in_smem && !planar && tile_bytes_needed_staged(w.Su, w.Sv, w.tw, w.th, w.nbins, w.nvals) <= budget;
  // (TMA staging is used by the interleaved organisation only — windows up to ~82 px, 96 % of them on the bench scene; the
  //  planar / staged organisations of the largest windows read their pixels with ordinary loads)
  if (!in_smem) w.tmap = nullptr;
  if (clk && tid == 0) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    clk[1] = clock64();
    clk[7] = w.Su;
    clk[8] = w.Sv;
    clk[9] = smid;
    clk[10] = in_smem ? 1 : planar ? 2 : staged ? 3 : 0;
  }
  const int boxv[4] = {box_l, box_t, box_r, box_b};
  float* dump_search = prm.io.dump_search ? prm.io.dump_search + po * prm.io.dump_cap : nullptr;
  float* dump_sse = prm.io.dump_sse ? prm.io.dump_sse + po * prm.io.dump_cap : nullptr;
  if (planar) {
    TilePlanes pl;
    tile_carve_planar(reinterpret_cast<char*>(smem_raw), w, pl);
    tile_prepare(prm.pixels[slot], prm.pitch[slot], prm.nchan[slot], boxv, prm.tmpl_tile + po * ta, prm.tmpl_quantiles + po * ta,
                 prm.tmpl_values + po * ta, w, dump_search, prm.io.dump_cap, clk ? clk + 2 : nullptr);
    tile_finish_planar(w, pl, reinterpret_cast<float4*>(region), dump_sse, prm.io.dump_cap, clk ? clk + 2 : nullptr);
    if (clk && tid == 0) clk[5] = clock64();
  } else if (staged) {
    tile_build_surface_staged(reinterpret_cast<char*>(smem_raw), region, prm.pixels[slot], prm.pitch[slot], prm.nchan[slot], boxv,
                              prm.tmpl_tile + po * ta, prm.tmpl_quantiles + po * ta, prm.tmpl_values + po * ta, w, dump_search, dump_sse,
                              prm.io.dump_cap, clk ? clk + 2 : nullptr);
    if (clk && tid == 0) clk[5] = clock64();
  } else {
    tile_carve(in_smem ? reinterpret_cast<char*>(smem_raw) : region, w);
    tile_build_surface(prm.pixels[slot], prm.pitch[slot], prm.nchan[slot], boxv, prm.tmpl_tile + po * ta, prm.tmpl_quantiles + po * ta,
                       prm.tmpl_values + po * ta, w, dump_search, dump_sse, prm.io.dump_cap, clk ? clk + 2 : nullptr);
    if (clk && tid == 0) clk[5] = clock64();
    if (in_smem) {
      float4* dst = reinterpret_cast<float4*>(region);
      for (int i = tid; i < w.Mv * w.Mp; i += blockDim.x) dst[i] = w.herm[i];
    }
  }
  if (tid == 0) {
    meta[0] = box_l;
    meta[1] = box_t;
    meta[2] = box_r;
    meta[3] = box_b;
    meta[4] = w.Mu;
    meta[5] = w.Mv;
    meta[6] = w.Mp;
    meta[7] = 1;
    if (clk) clk[6] = clock64();
  }
}

// Exclusive offsets of one value per thread across the CTA (warp shuffles + one pass over the
// warp totals).  Returns the offset of the calling thread.
template <int NWARPS = GB_SBLOCK_THREADS / 32>
__device__ __forceinline__ double block_exclusive_offset(double v, double* s_warp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double incl = warp_inclusive_scan(v, lane);
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  double off = 0.0;
#pragma unroll
  for (int k = 0; k < NWARPS; ++k) off += k < warp ? s_warp[k] : 0.0;
  double excl = shfl_up(incl, 1);
  if (lane == 0) excl = 0.0;
  return off + excl;
}


// ---------------------------------------------------------------------------------------------
// Cheaper forms of three per-particle operations (same results within the stated bounds)
// ---------------------------------------------------------------------------------------------
// exp(-l) as 2^(n + f): the integer part goes into the exponent field, the fraction through MUFU.EX2.
// Relative error < 3e-7 — below the float32 rounding of the SSE surface the exponent is sampled from (the reference's
// own cv2.matchTemplate differs from an exact sum by 4e-6, DESIGN.md §6).  Underflows to 0 like exp(); NaN stays NaN.
__device__ __forceinline__ double exp_neg_fast(double l) {
  const double t = l * -1.4426950408889634074;
  if (!(t > -1074.0)) return (t != t) ? t : 0.0;
  const int n = min(__double2int_rd(t), 1023);
  const float f = (float)(t - (double)n);
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(f));
  const double rd = (double)r;  // [1, 2]
  if (n >= -1020) return __hiloint2double(__double2hiint(rd) + (n << 20), __double2loint(rd));
  return __hiloint2double(__double2hiint(rd) + ((n + 1000) << 20), __double2loint(rd)) * 9.33263618503218878990e-302;  // 2^-1000
}

// Bicubic Hermite patch at (x, y) measured from the first cell centre in cell units, NOT yet clamped: the clamp of
// FITPACK's evaluation (argument limited to the first / last data site) is the saturation of the in-cell offset.
__device__ __forceinline__ float hermite_eval_sat(const float4* __restrict__ herm, int Mp, int Mu, int Mv, double x, double y, bool lin_u,
                                                  bool lin_v) {
  const int j = max(min(__double2int_rz(x), Mu - 2), 0), i = max(min(__double2int_rz(y), Mv - 2), 0);
  const float tx = __saturatef((float)(x - (double)j)), ty = __saturatef((float)(y - (double)i));
  const float tx2 = tx * tx, tx3 = tx2 * tx, ty2 = ty * ty, ty3 = ty2 * ty;
  const float a2 = lin_u ? tx : 3.0f * tx2 - 2.0f * tx3, a0 = 1.0f - a2, a3 = lin_u ? 0.0f : tx3 - tx2, a1 = lin_u ? 0.0f : a3 - tx2 + tx;
  const float b2 = lin_v ? ty : 3.0f * ty2 - 2.0f * ty3, b0 = 1.0f - b2, b3 = lin_v ? 0.0f : ty3 - ty2, b1 = lin_v ? 0.0f : b3 - ty2 + ty;
  const float4* row0 = herm + i * Mp + j;
  const float4 h00 = row0[0], h01 = row0[1], h10 = row0[Mp], h11 = row0[Mp + 1];
  const float top_f = a0 * h00.x + a2 * h01.x + a1 * h00.y + a3 * h01.y;
  const float bot_f = a0 * h10.x + a2 * h11.x + a1 * h10.y + a3 * h11.y;
  const float top_v = a0 * h00.z + a2 * h01.z + a1 * h00.w + a3 * h01.w;
  const float bot_v = a0 * h10.z + a2 * h11.z + a1 * h10.w + a3 * h11.w;
  return b0 * top_f + b2 * bot_f + b1 * top_v + b3 * bot_v;
}

// Child range end with the verification only where it can matter: floor(c N - u) + 1 is the answer unless c N - u lies
// within 1e-6 of an integer (its rounding error is ~1e-12), where the reference's own position formula decides.
__device__ __forceinline__ int count_positions_le_fast(double c, double u, double inv_n, int N, double dN) {
  const double x = fma(c, dN, -u);
  const double fl = floor(x);
  if (x - fl > 1e-6 && x - fl < 1.0 - 1e-6) return min(max((int)fl + 1, 0), N);
  return count_positions_le(c, u, inv_n, N);
}

// Per-(CTA, observer) constants of the spline surface: geo-reference (tracker.py:615-620) and cell
// centres (observer.py:203-208).
struct SurfaceRef {
  double sl, st, sr, sb, cu0, cv0, cu1, cv1, scale;
  const float4* herm;
  double* sampled;  // gb_stage_io.dump_sampled row of the slot's observer
  int Mu, Mv, Mp, ok;
};

// s3: spline sample + surface likelihood -> weight; two consecutive particles per thread.  Grid: blocks of a
// point x points; launched with s3_threads(s_block) threads so that full trips cover the CTA's particle pairs.
#ifndef GB_S3_MAX_THREADS
#define GB_S3_MAX_THREADS 64
#endif
#ifndef GB_S3_MINB
#define GB_S3_MINB 16
#endif
__host__ __device__ inline int s3_threads(int s_block) {
  const int pairs = (s_block + 1) / 2;
  const int trips = (pairs + GB_S3_MAX_THREADS - 1) / GB_S3_MAX_THREADS;
  return ((pairs + trips - 1) / trips + 31) / 32 * 32;
}

// One warp per point (k_s3b_publish): turns the CTA totals of k_s3 into what k_s4p needs — the prefix
// of the totals (CTA b owns cumulative weights (pre[b], pre[b + 1]]), 1 / total, the uniform draw of this update
// and 1 / N.  Every k_s4p CTA of the point reads the same record, so child ranges meet exactly at CTA boundaries.
__device__ __forceinline__ void s3_publish_prefix(const StepParams& prm, int64_t p, int lane) {
  const int nblk = prm.s_nblk;
  const double* bs = prm.s_bsum + p * nblk;
  double* pre = prm.s_pre + p * (nblk + 4);
  double run = 0.0;
  for (int c0 = 0; c0 < nblk; c0 += 32) {
    const double x = c0 + lane < nblk ? bs[c0 + lane] : 0.0;
    const double incl = run + warp_inclusive_scan(x, lane);
    if (c0 + lane < nblk) pre[c0 + lane + 1] = incl;
    run = __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) {
    pre[0] = 0.0;
    pre[nblk + 1] = quo(1.0, run);
    pre[nblk + 2] = prm.resample_method != GB_RESAMPLE_SYSTEMATIC ? 0.0
                    : prm.rng_mode == GB_RNG_SUPPLIED ? prm.uniforms[(int64_t)p * prm.S + (prm.t - prm.first[p] - 1)]
                                                      : philox_uniform(prm.seed, (uint64_t)(p + prm.point_offset), (uint32_t)prm.t);
    pre[nblk + 3] = quo(1.0, (double)prm.N);
  }
}
// GEN: spline degrees other than 1 / 3 (B-spline coefficients; its own instantiation keeps the default kernel's registers)
template <bool GEN>
__global__ void __launch_bounds__(GB_S3_MAX_THREADS, GB_S3_MINB) k_s3_weights(const __grid_constant__ StepParams prm) {
  __shared__ gb_motion s_motion;
  __shared__ SurfaceRef s_ref[GB_MAX_OBS];
  __shared__ double s_warp[GB_S3_MAX_THREADS / 32];
  const int64_t p = prm.p0 + blockIdx.y;
  const int b = (int)blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = (int)prm.N, ns = prm.n_slots;
  const int act = prm.s_act[p];
  const int failed_at_t = prm.s_pflags[p];
  // every scalar of the prologue is requested before the first branch: one memory round trip instead of two
  int meta[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  double du_t = 0.0, dv_t = 0.0, obs_scale = 0.0;
  if (tid < ns) {
    const int64_t ps = p * prm.slot_stride + tid, po = p * prm.O + prm.obs[tid];
    const int4 m0 = *reinterpret_cast<const int4*>(prm.s_meta + ps * 8), m1 = *reinterpret_cast<const int4*>(prm.s_meta + ps * 8 + 4);
    meta[0] = m0.x; meta[1] = m0.y; meta[2] = m0.z; meta[3] = m0.w;
    meta[4] = m1.x; meta[5] = m1.y; meta[6] = m1.z; meta[7] = m1.w;
    du_t = prm.tmpl_duv[po * 2];
    dv_t = prm.tmpl_duv[po * 2 + 1];
    obs_scale = prm.obs_scale[tid];
  }
  if (!(act & GB_ACT_ACTIVE) || failed_at_t != 0) return;
  const bool surface_ll = (act & GB_ACT_SURFACE_LL) != 0;
  {
    if (surface_ll) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(prm.motion + p);
      uint32_t* dst = reinterpret_cast<uint32_t*>(&s_motion);
      for (int k = tid; k < (int)(sizeof(gb_motion) / 4); k += blockDim.x) dst[k] = src[k];
    }
    if (tid < ns) {
      const int sl = tid;
      SurfaceRef r;
      r.ok = meta[7];
      r.Mu = meta[4];
      r.Mv = meta[5];
      r.Mp = meta[6];
      const double eu = sub(mul((double)prm.tile_w, 0.5), 0.5), evv = sub(mul((double)prm.tile_h, 0.5), 0.5);
      r.sl = add(add((double)meta[0], eu), du_t);
      r.st = add(add((double)meta[1], evv), dv_t);
      r.sr = add(add((double)meta[2], -eu), du_t);
      r.sb = add(add((double)meta[3], -evv), dv_t);
      r.cu0 = add(r.sl, mul(quo(sub(r.sr, r.sl), (double)max(r.Mu, 1)), 0.5));
      r.cv0 = add(r.st, mul(quo(sub(r.sb, r.st), (double)max(r.Mv, 1)), 0.5));
      r.cu1 = add(r.cu0, (double)(r.Mu - 1));
      r.cv1 = add(r.cv0, (double)(r.Mv - 1));
      r.scale = obs_scale;
      r.herm = reinterpret_cast<const float4*>(prm.s_surf + (p * prm.slot_stride + sl) * prm.surf_bytes);
      r.sampled = prm.io.dump_sampled ? prm.io.dump_sampled + (p * prm.O + prm.obs[sl]) * N : nullptr;
      s_ref[sl] = r;
    }
  }
  __syncthreads();
  const double* ev = prm.s_ev + p * 6 * (int64_t)N;
  const double* fw = prm.io.force_weights ? prm.io.force_weights + (int64_t)p * N : nullptr;
  if (!fw && (act & GB_ACT_NO_MOTION_LL)) {
    // no image likelihood at this time and a motion model without one: the reference leaves the weights of the last
    // resampling in place (tracker.py:146-149); they live in weight_state (ones after initialisation)
    bool any_ok = false;
    for (int sl = 0; sl < ns; ++sl) any_ok |= s_ref[sl].ok != 0;
    if (!any_ok && prm.weight_state) fw = prm.weight_state + (int64_t)p * N;
  }
  const bool vec = (N & 1) == 0;
  const bool lin_u = prm.interp_cols == 1, lin_v = prm.interp_rows == 1;  // Tracker.interpolation: degree 1 along an axis
  constexpr bool gen = GEN;
  uint32_t flags = 0;
  double wacc = 0.0;
  const int blk_end = min(N, (b + 1) * prm.s_block);  // s_block is even: pairs never straddle CTAs
  for (int sub = 0; sub < prm.s_block; sub += 2 * (int)blockDim.x) {
  const int ia = b * prm.s_block + sub + 2 * tid;
  const bool va = ia < blk_end, vb = ia + 1 < blk_end;
  double w[2] = {0.0, 0.0};
  if (va) {
    if (fw) {
      w[0] = fw[ia];
      w[1] = vb ? fw[ia + 1] : 0.0;
    } else {
      double ll[2] = {0.0, 0.0};
      // observers in slot order, which is ascending observer order: the reference's order of the sum
      for (int sl = 0; sl < ns; ++sl) {
        const SurfaceRef& r = s_ref[sl];
        if (!r.ok) continue;
        const double* uv = prm.s_uv + (p * prm.slot_stride + sl) * 2 * (int64_t)N;
        double u[2], v[2];
        if (vec) {
          const double2 a = *reinterpret_cast<const double2*>(uv + ia), c = *reinterpret_cast<const double2*>(uv + (int64_t)N + ia);
          u[0] = a.x;
          u[1] = a.y;
          v[0] = c.x;
          v[1] = c.y;
        } else {
          u[0] = uv[ia];
          v[0] = uv[(int64_t)N + ia];
          u[1] = vb ? uv[ia + 1] : u[0];
          v[1] = vb ? uv[(int64_t)N + ia + 1] : v[0];
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          if (!((u[q] >= r.sl) & (u[q] <= r.sr) & (v[q] >= r.st) & (v[q] <= r.sb))) flags |= GB_F_SAMPLE_OUTSIDE;
          // FITPACK evaluates at the argument clamped to the first/last data site: the saturation inside hermite_eval_sat
          const double val = gen ? (double)bspline_eval(r.herm, r.Mp, r.Mu, r.Mv, u[q] - r.cu0, v[q] - r.cv0, prm.interp_cols, prm.interp_rows)
                                 : (double)hermite_eval_sat(r.herm, r.Mp, r.Mu, r.Mv, u[q] - r.cu0, v[q] - r.cv0, lin_u, lin_v);
          ll[q] = add(ll[q], mul(val, r.scale));
          if (prm.io.dump_sampled && (q == 0 || vb)) r.sampled[ia + q] = val;
        }
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (q == 1 && !vb) break;
        const int i = ia + q;
        double l = ll[q];
        if (surface_ll) l = add(l, surface_log_likelihood(s_motion, prm.surfaces, ev[i], ev[(int64_t)N + i], ev[2 * (int64_t)N + i], flags));
        else l = add(l, 0.0);
        w[q] = add(exp_neg_fast(l), 1e-300);
      }
    }
    double* wd = prm.s_w + (int64_t)p * N;
    if (vec) {
      *reinterpret_cast<double2*>(wd + ia) = make_double2(w[0], w[1]);
    } else {
      wd[ia] = w[0];
      if (vb) wd[ia + 1] = w[1];
    }
    if (prm.io.dump_weights) {
      prm.io.dump_weights[(int64_t)p * N + ia] = w[0];
      if (vb) prm.io.dump_weights[(int64_t)p * N + ia + 1] = w[1];
    }
  }
  wacc += w[0] + w[1];
  }
  // CTA total of the weights (fixed association: per thread, warp butterfly, warps in order)
  const double tsum = warp_sum(wacc);
  if (lane == 0) s_warp[warp] = tsum;
  __shared__ unsigned s_or;
  const int any = (int)block_or(flags, &s_or);
  if (tid == 0) {
    double tot = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) tot += s_warp[k];
    prm.s_bsum[p * prm.s_nblk + b] = tot;
    if (any) atomicOr(&prm.s_pflags[p], any);
  }
}

// s3b (pipelined flow): one warp per point turns the CTA totals of k_s3 into the record k_s4p reads.
__global__ void k_s3b_publish(const __grid_constant__ StepParams prm) {
  const int64_t p = prm.p0 + ((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
  if (p >= prm.p0 + prm.pb) return;
  if (!(prm.s_act[p] & GB_ACT_ACTIVE) || prm.s_pflags[p] != 0) return;
  s3_publish_prefix(prm, p, threadIdx.x & 31);
}

// s4: prefix of the weights and child ranges (GB_S4_PPT consecutive parents per thread), then one thread
// per CHILD: find the parent in the CTA's sorted range ends, gather its state, write coalesced, and add it
// to the moment partials (sum over children == sum over parents weighted by their child counts).
#define GB_S4_PPT 8
template <bool COV>
__global__ void __launch_bounds__(GB_SBLOCK_THREADS, 4) k_s4_resample(const __grid_constant__ StepParams prm) {
  constexpr int NM = Moments<COV>::NM, KP = COV ? 32 : 16, PPT = GB_S4_PPT, CAP = PPT * GB_SBLOCK_THREADS;
  __shared__ double s_warp[GB_SBLOCK_THREADS / 32];
  __shared__ double s_pref[6];
  __shared__ double s_red[GB_SBLOCK_THREADS / 32][KP];
  __shared__ double s_w[CAP];
  __shared__ int s_end[CAP];
  __shared__ int s_j0;
  const int64_t p = prm.p0 + blockIdx.x / prm.s_nblk;
  const int b = (int)(blockIdx.x % prm.s_nblk);
  if (!stream_point_active(prm, p) || prm.s_pflags[p] != 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, t = prm.t;
  const int N = (int)prm.N;
  // prefix of the preceding CTAs and the point total, summed in CTA order by one thread (every CTA of the
  // point computes the same chain, so child ranges meet exactly at CTA boundaries)
  if (tid == 0) {
    const double* bs = prm.s_bsum + p * prm.s_nblk;
    double run = 0.0, pre = 0.0, nxt = 0.0;
    for (int k = 0; k < prm.s_nblk; ++k) {
      if (k == b) pre = run;
      run += bs[k];
      if (k == b) nxt = run;
    }
    s_pref[0] = pre;
    s_pref[1] = run;
    s_pref[2] = nxt;
    s_pref[3] = prm.resample_method != GB_RESAMPLE_SYSTEMATIC ? 0.0
                : prm.rng_mode == GB_RNG_SUPPLIED ? prm.uniforms[(int64_t)p * prm.S + (t - prm.first[p] - 1)]
                                                  : philox_uniform(prm.seed, (uint64_t)(p + prm.point_offset), (uint32_t)t);
    s_pref[4] = quo(1.0, (double)N);
    s_pref[5] = quo(1.0, run);
  }
  const double* wsrc = prm.s_w + (int64_t)p * N;
  const int base = b * prm.s_block;
  const int n_here = max(0, min(N, base + prm.s_block) - base);  // parents of this CTA (<= CAP)
  const int k0 = PPT * tid;                                      // first local parent of this thread
  double w[PPT];
  if ((N & 1) == 0 && k0 + PPT <= n_here) {
#pragma unroll
    for (int q = 0; q < PPT; q += 2) {
      const double2 x = *reinterpret_cast<const double2*>(wsrc + base + k0 + q);
      w[q] = x.x;
      w[q + 1] = x.y;
    }
  } else {
#pragma unroll
    for (int q = 0; q < PPT; ++q) w[q] = (k0 + q < n_here) ? wsrc[base + k0 + q] : 0.0;
  }
  double tsum = 0.0;
#pragma unroll
  for (int q = 0; q < PPT; ++q) {
    if (k0 + q < CAP) s_w[k0 + q] = w[q];
    tsum += w[q];
    w[q] = tsum;  // inclusive prefix inside the thread
  }
  const double off = block_exclusive_offset(tsum, s_warp);  // contains a __syncthreads(): s_pref is visible
  const double prefix = s_pref[0], total = s_pref[1], next_prefix = s_pref[2], u01 = s_pref[3], inv_n = s_pref[4], inv_total = s_pref[5];
  const bool stratified = prm.resample_method == GB_RESAMPLE_STRATIFIED;
  // The last parent of the CTA takes the next CTA's prefix as its cumulative weight, so that child ranges
  // are seamless across CTAs whatever the association of the in-CTA sums.
#pragma unroll
  for (int q = 0; q < PPT; ++q) {
    const int k = k0 + q;
    if (k < n_here) {
      const double c = (k == n_here - 1) ? next_prefix : prefix + (off + w[q]);
      s_end[k] = stratified ? count_positions_le_stratified(quo(c, total), stratified_draws(prm, p, t), inv_n, N)
                            : count_positions_le(quo(c, total), u01, inv_n, N);
    }
  }
  if (tid == 0) {
    const double c0 = prefix >= total ? 1.0 : prefix * inv_total;
    s_j0 = b == 0 ? 0 : stratified ? count_positions_le_stratified(c0, stratified_draws(prm, p, t), inv_n, N) : count_positions_le(c0, u01, inv_n, N);
  }
  __syncthreads();
  const int J0 = s_j0, J1 = n_here > 0 ? s_end[n_here - 1] : J0;
  const double* ev = prm.s_ev + p * 6 * (int64_t)N + base;
  const double* sin0 = prm.io.force_evolved ? prm.io.force_evolved + p * 6 * (int64_t)N : state_buffer(prm, t - 1) + p * 6 * (int64_t)N;
  double ref[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) ref[c] = sin0[c * (int64_t)N];
  double* sout = state_buffer(prm, t) + p * 6 * (int64_t)N;
  double* wst = prm.weight_state ? prm.weight_state + (int64_t)p * N : nullptr;
  double* outp = prm.out_particles ? prm.out_particles + ((int64_t)p * prm.T + t) * N * 6 : nullptr;
  double* outw = prm.out_weights ? prm.out_weights + ((int64_t)p * prm.T + t) * N : nullptr;
  int* outi = prm.io.dump_indices ? prm.io.dump_indices + (int64_t)p * N : nullptr;
  double* fin = (prm.final_weights && p == prm.P - 1 && t == prm.last[p]) ? prm.final_weights : nullptr;
  Moments<COV> mom;
  mom.clear();
  for (int j = J0 + tid; j < J1; j += GB_SBLOCK_THREADS) {
    int lo = 0, hi = n_here - 1;  // smallest parent whose range end exceeds j
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (s_end[mid] > j) hi = mid; else lo = mid + 1;
    }
    double s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) s[c] = ev[c * (int64_t)N + lo];
    const double wj = s_w[lo];
#pragma unroll
    for (int c = 0; c < 6; ++c) __stcs(&sout[c * (int64_t)N + j], s[c]);  // next read is a whole update away
    mom.accumulate(wj, s, ref);
    if (wst) wst[j] = wj;
    if (fin) fin[j] = wj;
    if (outp) {
#pragma unroll
      for (int c = 0; c < 6; ++c) outp[(int64_t)j * 6 + c] = s[c];
    }
    if (outw) outw[j] = wj;
    if (outi) outi[j] = base + lo;
  }
  // per-CTA moment partials, combined in CTA order by s5 (bit-reproducible)
  double r[KP];
#pragma unroll
  for (int k = 0; k < KP; ++k) r[k] = k < NM ? mom.a[k] : 0.0;
  warp_reduce_transpose<KP>(r, lane);
  if (KP == 32 || (lane & 1) == 0) s_red[warp][transposed_index<KP>(lane)] = r[0];
  __syncthreads();
  if (tid < NM) {
    double x = s_red[0][tid];
    for (int wv = 1; wv < (int)(blockDim.x >> 5); ++wv) x += s_red[wv][tid];
    prm.s_pm[(p * prm.s_nblk + b) * 28 + tid] = x;
  }
}

// Random choice with replacement (Tracker(resample_method='choice'), tracker.py:205-209 = the legacy generator's inverse-CDF
// sampling).  Children are not sorted by parent, so every child searches the point's whole cumulative distribution:
// k_s4c_scan writes it (normalised cumulative weights, last entry exactly 1) into the point's projected-coordinate scratch,
// which is dead after k_s3; k_s4c_gather draws one uniform per child, finds #{i : cdf[i] <= u} and copies that parent.
// Used by the step-by-step flow only (gb_track falls back to it for this method).
__global__ void __launch_bounds__(GB_SBLOCK_THREADS, 4) k_s4c_scan(const __grid_constant__ StepParams prm) {
  constexpr int PPT = GB_S4_PPT;
  __shared__ double s_warp[GB_SBLOCK_THREADS / 32];
  __shared__ double s_pref[2];
  const int64_t p = prm.p0 + blockIdx.x / prm.s_nblk;
  const int b = (int)(blockIdx.x % prm.s_nblk);
  if (!stream_point_active(prm, p) || prm.s_pflags[p] != 0) return;
  const int tid = threadIdx.x;
  const int N = (int)prm.N;
  if (tid == 0) {
    const double* bs = prm.s_bsum + p * prm.s_nblk;
    double run = 0.0, pre = 0.0;
    for (int k = 0; k < prm.s_nblk; ++k) {
      if (k == b) pre = run;
      run += bs[k];
    }
    s_pref[0] = pre;
    s_pref[1] = run;
  }
  const double* wsrc = prm.s_w + (int64_t)p * N;
  const int base = b * prm.s_block;
  const int n_here = max(0, min(N, base + prm.s_block) - base);
  const int k0 = PPT * tid;
  double w[PPT], tsum = 0.0;
#pragma unroll
  for (int q = 0; q < PPT; ++q) {
    tsum += (k0 + q < n_here) ? wsrc[base + k0 + q] : 0.0;
    w[q] = tsum;
  }
  const double off = block_exclusive_offset(tsum, s_warp);
  const double prefix = s_pref[0], total = s_pref[1];
  double* cdf = prm.s_uv + p * prm.slot_stride * 2 * (int64_t)N;
#pragma unroll
  for (int q = 0; q < PPT; ++q) {
    const int k = k0 + q;
    if (k < n_here) cdf[base + k] = (base + k == N - 1) ? 1.0 : quo(prefix + (off + w[q]), total);
  }
}

// np.add.reduce over a contiguous float64 vector = NumPy's pairwise summation (numpy/core/src/umath/loops_utils.h:
// fewer than 8 elements in order; up to 128 with eight strided accumulators combined as ((r0 + r1) + (r2 + r3)) + ((r4 + r5) +
// (r6 + r7)) and the remainder added in order; longer vectors split at n / 2 rounded down to a multiple of 8).  One thread.
// `scale`, `shift`: the summand is a[i] * scale - shift[i] (shift may be null) — the residual resampler sums derived vectors.
template <class F>
__device__ __forceinline__ double numpy_pairwise_block(F a, int64_t lo, int64_t n) {  // n <= 128
  if (n < 8) {
    double res = 0.0;
    for (int64_t i = 0; i < n; ++i) res += a(lo + i);
    return res;
  }
  double r[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = a(lo + k);
  int64_t i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] += a(lo + i + k);
  }
  double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) res += a(lo + i);
  return res;
}
template <class F>
__device__ double numpy_pairwise_sum(F a, int64_t lo0, int64_t n0) {
  // the recursion, unrolled on an explicit stack (post-order: left subtree, right subtree, add)
  int64_t lo[40], n[40];
  double left[40];
  int phase[40];
  int sp = 0;
  lo[0] = lo0;
  n[0] = n0;
  phase[0] = 0;
  double ret = 0.0;
  while (sp >= 0) {
    if (n[sp] <= 128) {
      ret = numpy_pairwise_block(a, lo[sp], n[sp]);
      --sp;
      continue;
    }
    int64_t n2 = n[sp] / 2;
    n2 -= n2 % 8;
    if (phase[sp] == 0) {
      phase[sp] = 1;
      lo[sp + 1] = lo[sp];
      n[sp + 1] = n2;
      phase[sp + 1] = 0;
      ++sp;
    } else if (phase[sp] == 1) {
      left[sp] = ret;
      phase[sp] = 2;
      lo[sp + 1] = lo[sp] + n2;
      n[sp + 1] = n[sp] - n2;
      phase[sp + 1] = 0;
      ++sp;
    } else {
      ret = left[sp] + ret;
      --sp;
    }
  }
  return ret;
}

// Residual resampling exactly as the reference does it (tracker.py:188-203), including what a textbook version would not:
// the residuals are taken of the NORMALISED weights minus the integer repetitions (not of n w), so their cumulative sum is not
// monotone, and np.searchsorted's answers on it depend on NumPy's search, which keeps one bound from the previous key
// (numpy/core/src/npysort/binsearch.cpp) — restated here operation by operation.  One CTA per point: the sums, the cumulative
// sum and the search run on one thread in NumPy's order (this method is a compatibility path, not a fast one); repetitions and
// their offsets on all threads.  Output: the parent of every child, int32 [N], behind the cumulative sums in the point's
// projected-coordinate scratch (dead after k_s3) — k_s4c_gather copies the parents.
__global__ void __launch_bounds__(GB_SBLOCK_THREADS) k_s4r_residual(const __grid_constant__ StepParams prm) {
  __shared__ double s_tot[2];
  __shared__ int s_scan[GB_SBLOCK_THREADS];
  __shared__ int s_K;
  const int64_t p = prm.p0 + blockIdx.x;
  if (!stream_point_active(prm, p) || prm.s_pflags[p] != 0) return;
  const int tid = threadIdx.x, N = (int)prm.N, t = prm.t;
  const double* w = prm.s_w + (int64_t)p * N;
  double* cs = prm.s_uv + p * prm.slot_stride * 2 * (int64_t)N;    // [N] normalised weights, then residuals, then their cumulative sum
  int* ridx = reinterpret_cast<int*>(cs + N);           // [N] parent of every child
  int* cum = ridx + N;                                  // [N] inclusive prefix of the repetitions
  if (tid == 0) s_tot[0] = numpy_pairwise_sum([w](int64_t i) { return w[i]; }, 0, N);
  __syncthreads();
  const double total = s_tot[0], dn = (double)N;
  // repetitions = (n * weights).astype(int); blocked layout so that one scan over the threads orders them
  const int per = (N + GB_SBLOCK_THREADS - 1) / GB_SBLOCK_THREADS, i0 = tid * per, i1 = min(N, i0 + per);
  int mine = 0;
  for (int i = i0; i < i1; ++i) {
    const double wn = quo(w[i], total);
    const int reps = (int)mul(dn, wn);
    cs[i] = sub(wn, (double)reps);  // residuals = weights - repetitions
    mine += reps;
    cum[i] = mine;
  }
  s_scan[tid] = mine;
  __syncthreads();
  if (tid == 0) {
    int run = 0;
    for (int k = 0; k < GB_SBLOCK_THREADS; ++k) {
      const int x = s_scan[k];
      s_scan[k] = run;
      run += x;
    }
    s_K = run;
  }
  __syncthreads();
  for (int i = i0; i < i1; ++i) cum[i] += s_scan[tid];
  __syncthreads();
  const int K = min(s_K, N);
  // initial_indexes = np.repeat(np.arange(n), repetitions): child j belongs to the first parent whose inclusive prefix exceeds j
  for (int j = tid; j < K; j += GB_SBLOCK_THREADS) {
    int lo = 0, hi = N - 1;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (cum[mid] > j) hi = mid; else lo = mid + 1;
    }
    ridx[j] = lo;
  }
  if (tid == 0) {
    // residuals *= 1 / residuals.sum(); cumulative_sum = np.cumsum(residuals); cumulative_sum[-1] = 1.0
    const double inv = quo(1.0, numpy_pairwise_sum([cs](int64_t i) { return cs[i]; }, 0, N));
    double run = 0.0;
    for (int i = 0; i < N; ++i) {
      run = add(run, mul(cs[i], inv));
      cs[i] = run;
    }
    cs[N - 1] = 1.0;
    // additional_indexes = np.searchsorted(cumulative_sum, np.random.random(n - len(initial_indexes)))
    const StratifiedDraws draws = stratified_draws(prm, p, t);  // one uniform per additional child, in order
    int64_t lo = 0, hi = N;
    double last = K < N ? draws.u(0) : 0.0;
    for (int k = 0; k < N - K; ++k) {
      const double key = draws.u(k);
      if (last < key) {
        hi = N;
      } else {
        lo = 0;
        hi = hi < N ? hi + 1 : N;
      }
      last = key;
      while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (cs[mid] < key) lo = mid + 1; else hi = mid;
      }
      ridx[K + k] = (int)lo;
    }
  }
}

template <bool COV>
__global__ void __launch_bounds__(GB_SBLOCK_THREADS, 4) k_s4c_gather(const __grid_constant__ StepParams prm) {
  constexpr int NM = Moments<COV>::NM, KP = COV ? 32 : 16;
  __shared__ double s_red[GB_SBLOCK_THREADS / 32][KP];
  const int64_t p = prm.p0 + blockIdx.x / prm.s_nblk;
  const int b = (int)(blockIdx.x % prm.s_nblk);
  if (!stream_point_active(prm, p) || prm.s_pflags[p] != 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, t = prm.t;
  const int N = (int)prm.N;
  const int base = b * prm.s_block, end = min(N, base + prm.s_block);
  const double* cdf = prm.s_uv + p * prm.slot_stride * 2 * (int64_t)N;
  const double* ev = prm.s_ev + p * 6 * (int64_t)N;
  const double* wsrc = prm.s_w + (int64_t)p * N;
  const StratifiedDraws draws = stratified_draws(prm, p, t);  // one uniform per child, like the stratified resampler
  const double* sin0 = prm.io.force_evolved ? prm.io.force_evolved + p * 6 * (int64_t)N : state_buffer(prm, t - 1) + p * 6 * (int64_t)N;
  double ref[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) ref[c] = sin0[c * (int64_t)N];
  double* sout = state_buffer(prm, t) + p * 6 * (int64_t)N;
  double* wst = prm.weight_state ? prm.weight_state + (int64_t)p * N : nullptr;
  double* outp = prm.out_particles ? prm.out_particles + ((int64_t)p * prm.T + t) * N * 6 : nullptr;
  double* outw = prm.out_weights ? prm.out_weights + ((int64_t)p * prm.T + t) * N : nullptr;
  int* outi = prm.io.dump_indices ? prm.io.dump_indices + (int64_t)p * N : nullptr;
  double* fin = (prm.final_weights && p == prm.P - 1 && t == prm.last[p]) ? prm.final_weights : nullptr;
  Moments<COV> mom;
  mom.clear();
  const bool given = prm.resample_method == GB_RESAMPLE_RESIDUAL;  // k_s4r_residual has written every child's parent
  const int* ridx = reinterpret_cast<const int*>(cdf + N);
  for (int j = base + tid; j < end; j += GB_SBLOCK_THREADS) {
    int idx;
    if (given) {
      idx = min(max(ridx[j], 0), N - 1);
    } else {
      const double u = draws.u(j);
      int lo = 0, hi = N;  // number of entries <= u (np.searchsorted side='right')
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cdf[mid] <= u) lo = mid + 1; else hi = mid;
      }
      idx = min(lo, N - 1);
    }
    double s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) s[c] = ev[c * (int64_t)N + idx];
    const double wj = wsrc[idx];
#pragma unroll
    for (int c = 0; c < 6; ++c) sout[c * (int64_t)N + j] = s[c];
    mom.accumulate(wj, s, ref);
    if (wst) wst[j] = wj;
    if (fin) fin[j] = wj;
    if (outp) {
#pragma unroll
      for (int c = 0; c < 6; ++c) outp[(int64_t)j * 6 + c] = s[c];
    }
    if (outw) outw[j] = wj;
    if (outi) outi[j] = idx;
  }
  double r[KP];
#pragma unroll
  for (int k = 0; k < KP; ++k) r[k] = k < NM ? mom.a[k] : 0.0;
  warp_reduce_transpose<KP>(r, lane);
  if (KP == 32 || (lane & 1) == 0) s_red[warp][transposed_index<KP>(lane)] = r[0];
  __syncthreads();
  if (tid < NM) {
    double x = s_red[0][tid];
    for (int wv = 1; wv < (int)(blockDim.x >> 5); ++wv) x += s_red[wv][tid];
    prm.s_pm[(p * prm.s_nblk + b) * 28 + tid] = x;
  }
}

// s5: one warp per point: lane k sums moment k over the CTAs in order, lane 0 finalises.
template <bool COV>
__global__ void k_s5_finalize(const __grid_constant__ StepParams prm) {
  const int64_t p = prm.p0 + ((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (p >= prm.p0 + prm.pb || !stream_point_active(prm, p)) return;
  const int t = prm.t;
  const int f = prm.s_pflags[p];
  if (f) {
    if (lane == 0) {
      prm.status[p] = status_from_flags((uint32_t)f);
      prm.status_time[p] = t;
    }
    return;
  }
  constexpr int NM = Moments<COV>::NM;
  double x = 0.0;
  if (lane < NM)
    for (int b = 0; b < prm.s_nblk; ++b) x += prm.s_pm[(p * prm.s_nblk + b) * 28 + lane];
  double a[NM];
#pragma unroll
  for (int k = 0; k < NM; ++k) a[k] = __shfl_sync(0xffffffffu, x, k);
  if (lane != 0) return;
  const int64_t N = prm.N;
  const double* sin_ = prm.io.force_evolved ? prm.io.force_evolved + p * 6 * N : state_buffer(prm, t - 1) + p * 6 * N;
  double ref[6];
  for (int c = 0; c < 6; ++c) ref[c] = sin_[c * N];
  double mean[6], sg[6], cv[36];
  finalize_moments<COV>(a, ref, mean, sg, cv);
  double* mo = prm.means + ((int64_t)p * prm.T + t) * 6;
  for (int c = 0; c < 6; ++c) mo[c] = mean[c];
  if (COV) {
    double* co = prm.covariances + ((int64_t)p * prm.T + t) * 36;
    for (int c = 0; c < 36; ++c) co[c] = cv[c];
  } else {
    double* so = prm.sigmas + ((int64_t)p * prm.T + t) * 6;
    for (int c = 0; c < 6; ++c) so[c] = sg[c];
  }
}

// ---------------------------------------------------------------------------------------------
// Pipelined flow used by gb_track: the resampling of time t and the motion step to time t + 1 are
// one kernel (k_s4p), so the resampled state is never written to / read back from HBM between
// updates: a child thread gathers its parent's evolved particle, and immediately evolves, tests and
// projects it for the next time.  Per time t and batch:  [k_s0p ->] k_s2 -> k_s3 -> k_s3b -> k_s4p -> k_s5p
// (k_s0p only at a track's first time and after initialisation / template kernels).
//   activity bits of (point, t):  ACTIVE    = an update happens at t        (first < t <= last, alive)
//                                 PROPAGATE = particles are advanced to t+1 (first <= t < last, alive)
// Evolved particles and the per-point failure flags are double-buffered by time parity
// (s_ev / s_ev_next, s_pflags / s_pflags_next); the integer cloud box is consumed and reset by k_s2.
// ---------------------------------------------------------------------------------------------
#define GB_ACT_PROPAGATE 4

__device__ __forceinline__ uint8_t activity_bits(const StepParams& prm, int64_t i, int t, bool alive) {
  const int f = prm.first[i], l = prm.last[i];
  const gb_surface& sg = prm.surfaces[prm.motion[i].dem_sigma];
  const bool tangent = prm.motion[i].kind >= GB_MOTION_TANGENT_CARTESIAN;  // compute_log_likelihoods is None (motion.py:77-89)
  const bool sll = !tangent && !(sg.z == nullptr && sg.value == 0.0);
  return (uint8_t)(((alive && f < t && t <= l) ? GB_ACT_ACTIVE : 0) | (sll ? GB_ACT_SURFACE_LL : 0) | (tangent ? GB_ACT_NO_MOTION_LL : 0) |
                   ((alive && f <= t && t < l) ? GB_ACT_PROPAGATE : 0));
}

// Activity of time prm.t.  Launched at a track's first time and after the kernels that can change a point's status
// outside the update (initialisation, templates); otherwise k_s5p_finalize of time t - 1 has already written it.
__global__ void k_s0p_activity(const __grid_constant__ StepParams prm) {
  for (int64_t i = prm.p0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < prm.p0 + prm.pb; i += (int64_t)gridDim.x * blockDim.x)
    prm.s_act[i] = activity_bits(prm, i, prm.t, prm.status[i] == 0);
}

// Start of a gb_track: empty cloud boxes, no failure flags in either parity.
__global__ void k_s0p_reset(const __grid_constant__ StepParams prm) {
  const int64_t lo5 = prm.p0 * prm.slot_stride * 5, n = prm.pb * prm.slot_stride * 5;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    prm.s_ibox[lo5 + i] = (i % 5 == 4) ? 0 : 0x7fffffff;
  for (int64_t i = prm.p0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < prm.p0 + prm.pb; i += (int64_t)gridDim.x * blockDim.x) {
    prm.s_pflags[i] = 0;
    prm.s_pflags_next[i] = 0;
  }
}

// Capacity of one k_s4p CTA: the parents' evolved state (48 B), weight (8 B), child range end (4 B) and the
// children's parent index (4 B) live in shared memory — 64 B per parent, 48 KB per CTA, four CTAs per SM.
#ifndef GB_S4P_THREADS
#define GB_S4P_THREADS 192
#endif
#ifndef GB_S4P_CAP
#define GB_S4P_CAP 768
#endif
#ifndef GB_S4P_MINB
#define GB_S4P_MINB 4
#endif
#define GB_S4P_PPT ((GB_S4P_CAP + GB_S4P_THREADS - 1) / GB_S4P_THREADS)
constexpr int kS4pSmem = GB_S4P_CAP * 64;
static_assert(GB_S4P_THREADS >= 134, "k_s4p's prologue spreads its scalar loads over the first 134 threads");

// One projected child: image coordinates of time t + 1 and its contribution to the integer cloud box.
__device__ __forceinline__ void s4p_project_child(const CamK& cam, const double (&s)[6], double* uv, int64_t N, int j, double hw,
                                                  double hh, int (&e)[5]) {
  double u, v;
  project_fast(cam, s[0], s[1], s[2], u, v);
  uv[j] = u;
  uv[N + j] = v;
  e[0] = __double2int_rd(u - hw);
  e[1] = __double2int_rd(v - hh);
  e[2] = -__double2int_ru(u + hw);
  e[3] = -__double2int_ru(v + hh);
  e[4] = (isnan(u) | isnan(v)) ? -1 : 0;
}

template <bool COV, bool TAN>
__global__ void __launch_bounds__(GB_S4P_THREADS, GB_S4P_MINB) k_s4p_resample_propagate(const __grid_constant__ StepParams prm,
                                                                                   const __grid_constant__ NextParams nxt) {
  constexpr int NM = Moments<COV>::NM, KP = COV ? 32 : 16, PPT = GB_S4P_PPT, CAP = GB_S4P_CAP, NW = GB_S4P_THREADS / 32, TH = GB_S4P_THREADS;
  extern __shared__ __align__(128) unsigned char s4p_raw[];
  double* s_st = reinterpret_cast<double*>(s4p_raw);  // [6][CAP] parents' state: bulk-copy destination
  double* s_w = s_st + 6 * CAP;                       // [CAP] parents' weights
  int* s_end = reinterpret_cast<int*>(s_w + CAP);     // [CAP] child range ends
  int* s_par = s_end + CAP;                           // [CAP] parent of each child of the current chunk
  __shared__ __align__(8) uint64_t s_bar[2];
  __shared__ double s_warp[NW];
  __shared__ double s_red[NW][KP];
  __shared__ int s_wmax[NW];
  __shared__ int s_j0;
  __shared__ gb_motion s_motion;
  __shared__ int s_box[GB_MAX_OBS][5];
  __shared__ unsigned s_or;
  __shared__ double s_pre6[6];            // the point's published prefix record, as far as this CTA needs it
  __shared__ double s_refv[6];            // moment origin of the point (read in the prologue, used after the parents arrive)
  __shared__ uint8_t s_mask[GB_MAX_OBS];  // observers that see the point
  const int64_t p = prm.p0 + blockIdx.y;  // grid: (blocks of a point, points of the batch)
  const int b = (int)blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, t = prm.t;
  const int N = (int)prm.N, ns = nxt.n_slots;  // slots of t + 1, where the children are projected
  const int base = b * prm.s_block;
  const int n_here = max(0, min(N, base + prm.s_block) - base);  // parents of this CTA (<= CAP)
  const double* wsrc = prm.s_w + (int64_t)p * N + base;
  // When no point starts at this time every point that is processed is resampled from its evolved particles: the bulk
  // copies of the CTA's parents are requested before the point's activity byte is even read (one memory round trip less
  // in the prologue).  A point that turns out inactive or failed waits for the copies to land and leaves.
  const double* spec6 = prm.s_ev + p * 6 * (int64_t)N + base;
  const bool spec = nxt.spec_update && n_here > 0 && ((N | n_here) & 1) == 0 &&
                    ((reinterpret_cast<uintptr_t>(spec6) | reinterpret_cast<uintptr_t>(wsrc)) & 15) == 0;
  if (tid == 0) {
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    mbar_fence_init();
    if (spec) {
      const uint32_t row = (uint32_t)n_here * 8u;
      mbar_expect_tx(&s_bar[0], row);
      bulk_load(s_w, wsrc, row, &s_bar[0]);
      mbar_expect_tx(&s_bar[1], 6u * row);
#pragma unroll
      for (int c = 0; c < 6; ++c) bulk_load(s_st + c * CAP, spec6 + c * (int64_t)N, row, &s_bar[1]);
    }
  }
  const int act = prm.s_act[p];
  const int failed_at_t = prm.s_pflags[p];
  // the point's motion model, moment origin and observer mask are requested in the same breath (one word per thread):
  // they are needed by everybody who stays, and asking before the activity is known costs nothing
  static_assert(sizeof(gb_motion) / 4 <= 64, "one motion word per thread of the first two warps");
  uint32_t motion_word = 0;
  double ref_word = 0.0;
  uint8_t mask_byte = 0;
  if (tid < (int)(sizeof(gb_motion) / 4)) motion_word = reinterpret_cast<const uint32_t*>(prm.motion + p)[tid];
  if (tid >= 64 && tid < 70) ref_word = prm.s_ref[p * 6 + (tid - 64)];
  if (tid >= 96 && tid < 96 + ns) mask_byte = prm.mask[p * prm.O + nxt.obs[tid - 96]];
  if (tid >= 128 && tid < 134) {
    // written by k_s3b_publish: prefix of this and the next CTA, total, 1 / total, the uniform draw, 1 / N
    const int k = tid - 128;
    ref_word = prm.s_pre[p * (prm.s_nblk + 4) + (k < 2 ? b + k : prm.s_nblk + (k - 2))];
  }
  const bool update = (act & GB_ACT_ACTIVE) != 0, propagate = (act & GB_ACT_PROPAGATE) != 0;
  if ((!update && !propagate) || failed_at_t != 0) {  // a point that failed at t is neither resampled nor advanced
    if (spec && tid == 0) {
      mbar_wait(&s_bar[0], 0);
      mbar_wait(&s_bar[1], 0);
    }
    return;
  }
  // source of the particles that are resampled: the evolved particles of time t, or — at a point's first
  // time — the initial particles, taken one to one
  const double* src6 = (update ? prm.s_ev : state_buffer(prm, t)) + p * 6 * (int64_t)N + base;
  const bool bulk = n_here > 0 && ((N | n_here) & 1) == 0 && ((reinterpret_cast<uintptr_t>(src6) | reinterpret_cast<uintptr_t>(wsrc)) & 15) == 0;
  if (tid < (int)(sizeof(gb_motion) / 4)) reinterpret_cast<uint32_t*>(&s_motion)[tid] = motion_word;
  if (propagate && tid < GB_MAX_OBS * 5) s_box[tid / 5][tid % 5] = (tid % 5 == 4) ? 0 : 0x7fffffff;
  if (tid >= 64 && tid < 70) s_refv[tid - 64] = ref_word;
  if (tid >= 96 && tid < 96 + ns) s_mask[tid - 96] = mask_byte;
  if (tid >= 128 && tid < 134) s_pre6[tid - 128] = ref_word;
  __syncthreads();
  if (bulk) {
    // weights first (the prefix needs them), then the six state rows: all in flight while the prefix is computed
    if (tid == 0 && !spec) {
      const uint32_t row = (uint32_t)n_here * 8u;
      if (update) {
        mbar_expect_tx(&s_bar[0], row);
        bulk_load(s_w, wsrc, row, &s_bar[0]);
      }
      mbar_expect_tx(&s_bar[1], 6u * row);
#pragma unroll
      for (int c = 0; c < 6; ++c) bulk_load(s_st + c * CAP, src6 + c * (int64_t)N, row, &s_bar[1]);
    }
  } else {
    for (int i = tid; i < n_here; i += TH) {
      if (update) s_w[i] = wsrc[i];
#pragma unroll
      for (int c = 0; c < 6; ++c) s_st[c * CAP + i] = src6[c * (int64_t)N + i];
    }
  }
  // ---- child ranges of the CTA's parents ----
  int J0, J1;
  if (update) {
    const double prefix = s_pre6[0], next_prefix = s_pre6[1], total = s_pre6[2], inv_total = s_pre6[3], u01 = s_pre6[4],
                 inv_n = s_pre6[5];
    const bool stratified = prm.resample_method == GB_RESAMPLE_STRATIFIED;
    const double dN = (double)N;
    if (bulk) mbar_wait(&s_bar[0], 0);
    else __syncthreads();
    const int k0 = PPT * tid;  // first local parent of this thread (consecutive parents: in-thread prefix)
    double w[PPT];
    double tsum = 0.0;
#pragma unroll
    for (int q = 0; q < PPT; ++q) {
      tsum += (k0 + q < n_here) ? s_w[k0 + q] : 0.0;
      w[q] = tsum;  // inclusive prefix inside the thread
    }
    const double off = block_exclusive_offset<NW>(tsum, s_warp);
#pragma unroll
    for (int q = 0; q < PPT; ++q) {
      const int k = k0 + q;
      if (k < n_here) {
        // The last parent of the CTA takes the next CTA's prefix as its cumulative weight: child ranges are seamless
        // across CTAs whatever the association of the in-CTA sums.
        const double c = (k == n_here - 1) ? next_prefix : prefix + (off + w[q]);
        // normalised cumulative weight: one reciprocal per CTA instead of a division per particle (the total maps to exactly 1)
        const double cn = c >= total ? 1.0 : c * inv_total;
        s_end[k] = stratified ? count_positions_le_stratified(cn, stratified_draws(prm, p, t), inv_n, N) : count_positions_le_fast(cn, u01, inv_n, N, dN);
      }
    }
    if (tid == 0) {
      const double c0 = prefix >= total ? 1.0 : prefix * inv_total;
      s_j0 = b == 0 ? 0 : stratified ? count_positions_le_stratified(c0, stratified_draws(prm, p, t), inv_n, N) : count_positions_le_fast(c0, u01, inv_n, N, dN);
    }
    __syncthreads();
    J0 = s_j0;
    J1 = n_here > 0 ? s_end[n_here - 1] : J0;
  } else {
    J0 = base;
    J1 = base + n_here;
  }
  if (bulk) mbar_wait(&s_bar[1], 0);
  else if (!update) __syncthreads();
  // ---- moments of the resampled set: parents weighted by (children x weight), from shared memory ----
  if (update) {
    double ref[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) ref[c] = s_refv[c];
    Moments<COV> mom;
    mom.clear();
#pragma unroll
    for (int q = 0; q < PPT; ++q) {
      const int k = tid + q * TH;
      if (k < n_here) {
        const int cnt = s_end[k] - (k > 0 ? s_end[k - 1] : J0);
        if (cnt > 0) {
          double s[6];
#pragma unroll
          for (int c = 0; c < 6; ++c) s[c] = s_st[c * CAP + k];
          mom.accumulate((double)cnt * s_w[k], s, ref);
        }
      }
    }
    double r[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) r[k] = k < NM ? mom.a[k] : 0.0;
    warp_reduce_transpose<KP>(r, lane);
    if (KP == 32 || (lane & 1) == 0) s_red[warp][transposed_index<KP>(lane)] = r[0];
    __syncthreads();
    if (tid < NM) {
      double x = s_red[0][tid];
      for (int wv = 1; wv < NW; ++wv) x += s_red[wv][tid];
      prm.s_pm[(p * prm.s_nblk + b) * 28 + tid] = x;
    }
  }
  // ---- children: gather from shared memory, report, and advance to t + 1 ----
  const bool last_time = !propagate;  // t == last: the resampled particles are the final state
  double* sout = state_buffer(prm, t) + p * 6 * (int64_t)N;
  double* evn = prm.s_ev_next + p * 6 * (int64_t)N;
  double* wst = prm.weight_state ? prm.weight_state + (int64_t)p * N : nullptr;
  double* outp = (update && prm.out_particles) ? prm.out_particles + ((int64_t)p * prm.T + t) * N * 6 : nullptr;
  double* outw = (update && prm.out_weights) ? prm.out_weights + ((int64_t)p * prm.T + t) * N : nullptr;
  const int s_idx = (t + 1) - prm.first[p] - 1;
  const double* zn = (propagate && prm.step_normals) ? prm.step_normals + (((int64_t)p * prm.S + s_idx) * N) * 3 : nullptr;
  const double hw = (double)prm.tile_w * 0.5, hh = (double)prm.tile_h * 0.5;
  uint32_t flags = 0;
  const int need = propagate ? evolve_needs(s_motion) : 0;
  int ibx[2][5];  // register boxes for the first two observers; others go straight to shared memory
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    ibx[o][0] = ibx[o][1] = ibx[o][2] = ibx[o][3] = 0x7fffffff;
    ibx[o][4] = 0;
  }
  unsigned obs_on = 0;  // slots of t + 1 whose observer sees this point (block-uniform)
  if (propagate)
    for (int o = 0; o < ns; ++o)
      if (nxt.img[o] >= 0 && s_mask[o]) obs_on |= 1u << o;
  int carry = 0;  // parent of the last child of the previous chunk
  for (int Jc = J0; Jc < J1; Jc += CAP) {
    const int nch = min(CAP, J1 - Jc);
    if (update) {
      // parent of every child of the chunk: each parent marks its first child, a running maximum fills the rest
      for (int i = tid; i < nch; i += TH) s_par[i] = 0;
      __syncthreads();
#pragma unroll
      for (int q = 0; q < PPT; ++q) {
        const int k = tid + q * TH;
        if (k < n_here) {
          const int st = k > 0 ? s_end[k - 1] : J0, en = s_end[k];
          if (en > st && st >= Jc && st - Jc < nch) s_par[st - Jc] = k;
        }
      }
      __syncthreads();
      int v[PPT], run = 0;
#pragma unroll
      for (int q = 0; q < PPT; ++q) {
        const int i = PPT * tid + q;
        run = max(run, i < nch ? s_par[i] : 0);
        v[q] = run;
      }
      int incl = run;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl = max(incl, x);
      }
      if (lane == 31) s_wmax[warp] = incl;
      __syncthreads();
      int pre = carry, all = carry;
#pragma unroll
      for (int k = 0; k < NW; ++k) {
        const int x = s_wmax[k];
        if (k < warp) pre = max(pre, x);
        all = max(all, x);
      }
      int excl = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) excl = 0;
      pre = max(pre, excl);
#pragma unroll
      for (int q = 0; q < PPT; ++q) {
        const int i = PPT * tid + q;
        if (i < nch) s_par[i] = max(pre, v[q]);
      }
      carry = all;
      __syncthreads();
    }
    for (int j = Jc + tid; j < Jc + nch; j += TH) {
      const int lo = update ? s_par[j - Jc] : j - base;
      double s[6];
#pragma unroll
      for (int c = 0; c < 6; ++c) s[c] = s_st[c * CAP + lo];
      if (update) {
        const double wj = s_w[lo];
        if (last_time) {
#pragma unroll
          for (int c = 0; c < 6; ++c) __stcs(&sout[c * (int64_t)N + j], s[c]);
          if (prm.final_weights && p == prm.P - 1) prm.final_weights[j] = wj;
        }
        if (wst) wst[j] = wj;
        if (outp) {
#pragma unroll
          for (int c = 0; c < 6; ++c) outp[(int64_t)j * 6 + c] = s[c];
        }
        if (outw) outw[j] = wj;
      }
      if (propagate) {
        double z0, z1, z2;
        if (prm.rng_mode == GB_RNG_SUPPLIED) {
          z0 = zn[3 * (int64_t)j];
          z1 = zn[3 * (int64_t)j + 1];
          z2 = zn[3 * (int64_t)j + 2];
        } else {
          philox_normals3(prm.seed, (uint64_t)(p + prm.point_offset), (uint32_t)(t + 1), (uint32_t)j, 2u, z0, z1, z2, need);
        }
        evolve_particle<TAN>(s_motion, prm.surfaces, nxt.tau, nxt.tau2, z0, z1, z2, s, flags);
        flags |= test_particle(prm, s);
#pragma unroll
        for (int c = 0; c < 6; ++c) evn[c * (int64_t)N + j] = s[c];
        // the first two observers are unrolled: their camera operands come straight from the constant bank
#pragma unroll
        for (int o = 0; o < 2; ++o) {
          if (o >= ns) break;
          if (!(obs_on >> o & 1)) continue;
          const int64_t po = p * prm.slot_stride + o;
          int e[5];
          s4p_project_child(nxt.cam[o], s, prm.s_uv + po * 2 * (int64_t)N, N, j, hw, hh, e);
#pragma unroll
          for (int k = 0; k < 5; ++k) ibx[o][k] = min(ibx[o][k], e[k]);
        }
        for (int o = 2; o < ns; ++o) {
          if (!(obs_on >> o & 1)) continue;
          const int64_t po = p * prm.slot_stride + o;
          int e[5];
          s4p_project_child(nxt.cam[o], s, prm.s_uv + po * 2 * (int64_t)N, N, j, hw, hh, e);
#pragma unroll
          for (int k = 0; k < 5; ++k) atomicMin(&s_box[o][k], e[k]);
        }
      }
    }
    if (update && Jc + CAP < J1) __syncthreads();  // the next chunk rewrites s_par
  }
  if (propagate) {
    // cloud boxes of time t + 1: registers -> warp -> shared -> global
#pragma unroll
    for (int o = 0; o < 2; ++o) {
      if (o >= ns) break;
      int mine = 0x7fffffff;
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const int x = __reduce_min_sync(0xffffffffu, ibx[o][k]);
        if (lane == k) mine = x;
      }
      if (lane < 5) atomicMin(&s_box[o][lane], mine);
    }
    const int any = (int)block_or(flags, &s_or);  // also orders the shared-memory atomics above
    if (any && tid == 0) atomicOr(&prm.s_pflags_next[p], any);
    if (tid < ns * 5) {
      const int o = tid / 5, k = tid - o * 5;
      const int64_t po = p * prm.slot_stride + o;
      if (obs_on >> o & 1) atomicMin(&prm.s_ibox[po * 5 + k], s_box[o][k]);
    }
  }
}

// s5 of the pipelined flow: moments and status of time t, then the failure flags of this parity are cleared
// for time t + 2.  Also stores the moment origin of the next time (the first resampled particle).
template <bool COV>
__global__ void k_s5p_finalize(const __grid_constant__ StepParams prm) {
  const int64_t p = prm.p0 + ((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (p >= prm.p0 + prm.pb) return;
  const int act = prm.s_act[p];
  const int t = prm.t;
  const int f = prm.s_pflags[p];
  if (lane == 0) prm.s_pflags[p] = 0;
  // (every exit also writes the activity of time t + 1: the next update needs no launch of its own for it)
  if (!(act & GB_ACT_ACTIVE)) {
    if (lane == 0) {
      bool alive = prm.status[p] == 0;
      // a point can fail while being advanced from its first time: the failure belongs to time t
      if (f && alive && t > prm.first[p] && t <= prm.last[p]) {
        prm.status[p] = status_from_flags((uint32_t)f);
        prm.status_time[p] = t;
        alive = false;
      }
      prm.s_act[p] = activity_bits(prm, p, t + 1, alive);
    }
    return;
  }
  if (f) {
    if (lane == 0) {
      prm.status[p] = status_from_flags((uint32_t)f);
      prm.status_time[p] = t;
      prm.s_act[p] = activity_bits(prm, p, t + 1, false);
    }
    return;
  }
  constexpr int NM = Moments<COV>::NM;
  double x = 0.0;
  if (lane < NM)
    for (int b = 0; b < prm.s_nblk; ++b) x += prm.s_pm[(p * prm.s_nblk + b) * 28 + lane];
  double a[NM];
#pragma unroll
  for (int k = 0; k < NM; ++k) a[k] = __shfl_sync(0xffffffffu, x, k);
  if (lane != 0) return;
  prm.s_act[p] = activity_bits(prm, p, t + 1, true);
  double ref[6];
  for (int c = 0; c < 6; ++c) ref[c] = prm.s_ref[p * 6 + c];
  double mean[6], sg[6], cv[36];
  finalize_moments<COV>(a, ref, mean, sg, cv);
  double* mo = prm.means + ((int64_t)p * prm.T + t) * 6;
  for (int c = 0; c < 6; ++c) mo[c] = mean[c];
  if (COV) {
    double* co = prm.covariances + ((int64_t)p * prm.T + t) * 36;
    for (int c = 0; c < 36; ++c) co[c] = cv[c];
  } else {
    double* so = prm.sigmas + ((int64_t)p * prm.T + t) * 6;
    for (int c = 0; c < 6; ++c) so[c] = sg[c];
  }
}
