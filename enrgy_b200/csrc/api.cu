// C ABI of enrgy_b200 (include/enrgy_b200.h): context, device memory, launches.  No CPU fallback:
// every entry point that computes needs a CUDA device and fails with ENRGY_ERR_NODEVICE /
// ENRGY_ERR_CUDA otherwise.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "../../include/enrgy_b200.h"
#include "common.cuh"
#include "kernels.cuh"
#include "prepass.cuh"

using namespace enrgy;

namespace {

thread_local std::string g_err;

// largest raster side (rows or columns) accepted, include/enrgy_b200.h:enrgy_create and DESIGN.md §3
constexpr int kMaxSide = 1 << 20;

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CU_TRY(expr)                                                                      \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess)                                                                \
      return fail(ENRGY_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                  __FILE__, __LINE__);                                                    \
  } while (0)

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  cudaError_t alloc(size_t count) {
    if (count <= n && p) return cudaSuccess;
    release();
    cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
};

// ---- CUDA event pairs around the kernels of the last run (several chunks -> several pairs) ---------
struct EventPairs {
  std::vector<cudaEvent_t> ev;   // begin, end, begin, end, ...
  int used = 0;
  bool pending = false;
  double last_ms = 0.0;
  void reset() { used = 0; pending = false; }
  cudaError_t begin(cudaStream_t s) {
    while ((int)ev.size() < used + 2) {
      cudaEvent_t e;
      cudaError_t rc = cudaEventCreate(&e);
      if (rc != cudaSuccess) return rc;
      ev.push_back(e);
    }
    return cudaEventRecord(ev[used], s);
  }
  cudaError_t end(cudaStream_t s) {
    cudaError_t rc = cudaEventRecord(ev[used + 1], s);
    used += 2;
    pending = true;
    return rc;
  }
  double collect() {
    if (pending) {
      double tot = 0.0;
      for (int i = 0; i + 1 < used; i += 2) {
        float ms = 0.f;
        if (cudaEventSynchronize(ev[i + 1]) == cudaSuccess && cudaEventElapsedTime(&ms, ev[i], ev[i + 1]) == cudaSuccess) tot += ms;
      }
      last_ms = tot;
      pending = false;
    }
    return last_ms;
  }
  EventPairs() = default;
  EventPairs(const EventPairs&) = delete;
  EventPairs& operator=(const EventPairs&) = delete;
  ~EventPairs() {
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
};

}  // namespace

struct enrgy_ctx {
  int device = 0, rows = 0, cols = 0, precision = ENRGY_F32;
  int sm_count = 148;
  int l2_persist_max = 0, l2_window_max = 0;   // persisting-L2 carve-out and largest access-policy window [bytes]
  enrgy_params p{};
  double albedo_offset = 0.0;     // ensemble member
  double base_albedo_ice = 0.0, base_albedo_snow = 0.0;
  bool have_params = false, have_dem = false, have_forcing = false, prepass_done = false;
  bool state_advanced = false;
  // geometry
  int pitch = 0, rows_pad_full = 0, band_row0 = 0, band_rows = 0, band_rows_pad = 0;
  int tile_h = 8, tile_w = kTileW, tiles_r = 0, tiles_c = 0, n_tiles = 0;
  double n_valid = 0.0;
  double mom[5] = {0, 0, 0, 0, 0};   // moments of (dem - elev_aws) over the band's glacier cells
  size_t band_elems = 0;  // band_rows_pad * pitch
  // host copies
  std::vector<float> h_dem;       // full host copy, kept only when the AWS-cell shading ray needs it
  std::vector<float> h_terrain;   // ... and the uncropped terrain, when one was set (enrgy_set_terrain)
  float aws_nbhd[9] = {};         // terrain at the AWS cell and its 8 neighbours
  std::vector<double> forcing;
  int n_steps = 0;
  std::vector<double> pot_aws;
  PrepassOutput pre;
  // device rasters
  DevBuf<float> d_dem, d_terrain, d_albedo, d_pot, d_tmp32, d_scan, d_scan_t;
  bool have_terrain = false;
  int dem_pitch = 0;
  float* dem0 = nullptr;          // cell (0, 0) of the DEM buffer
  // shading: sunlit masks of a range of sub-steps, kept between runs (they depend on the terrain and
  // the sub-step directions only -- ensemble members and repeated passes reuse them)
  DevBuf<unsigned> d_maskbuf, d_masktmp;
  DevBuf<SweepSub> d_sweepsubs;
  int mask_sub0 = 0, mask_sub1 = 0;   // cached range [sub0, sub1) of d_maskbuf
  size_t mask_budget = (size_t)16 << 30;
  // a run cut into several launches: SWE at its start (total_snow = start - end is added by the last)
  DevBuf<unsigned char> d_swe_ref;
  int defer = 0;                  // 0 off, 1 deferring (launches leave total_snow alone), 2 the next launch applies
  DevBuf<unsigned char> d_nx, d_ny, d_nz, d_swe, d_ts, d_ti, d_dump, d_stage, d_snap, d_layer_t;
  bool have_msm = false;
  std::vector<double> alb_aws, layer_t_aws;
  double swe_aws = 0.0;
  bool snap_valid = false, snap_advanced = false;
  int n_maps = 0;
  int pot_t0 = 0, pot_n = 0;
  // tables
  DevBuf<unsigned char> d_steps, d_subs;
  DevBuf<StepRec<double>> d_steps64;
  DevBuf<TimeBlock> d_blocks;
  DevBuf<int2> d_tiles;
  DevBuf<int> d_counts;
  // host pre-pass started ahead of enrgy_prepass (see start_early_prepass)
  std::thread pre_thread;
  PrepassOutput pre_early;
  int pre_early_rc = 0;
  std::string pre_early_err;
  DevBuf<double> d_stats, d_small;
  // fused ensemble members (enrgy_run_members): state rasters [slots][3][band_elems], per-step member
  // scalars [T][nm] of the group in flight, float64 master records per member [slots][T]
  DevBuf<unsigned char> d_mstate, d_mrecs;
  DevBuf<StepRec<double>> d_msteps64;
  int member_slots = 0, members_last = 0;
  // station blend (enrgy_set_stations): extra weather stations and the cloud attenuation of the shortwave
  bool stations_on = false;
  int n_extra = 0;
  double st_row[kMaxStations] = {}, st_col[kMaxStations] = {}, st_elev[kMaxStations] = {};
  std::vector<double> st_series;   // [n_extra][n_steps][ENRGY_ST_COUNT]
  double cloud_k = NAN;
  DevBuf<unsigned char> d_strecs;  // StationRec<R> [n_steps][kMaxStations]
  DevBuf<unsigned char> d_partials;
  DevBuf<unsigned long long> d_counters;
  std::vector<ShadeRec> mask_shades;   // directions the cached masks were swept for
  EventPairs ev_fused, ev_sweep;   // around the fused kernels / the shading sweeps of the last run
  // SWE statistics of the initial raster (first CSV row)
  double swe0_sum = 0.0, swe0_nsnow = 0.0, swe0_nvalid = 0.0;
  // runtime
  cudaStream_t stream = nullptr;
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int64_t launches = 0;
  LaunchInfo info{};
};

namespace {

size_t rsize(const enrgy_ctx* c) { return c->precision == ENRGY_F32 ? 4 : 8; }

// f(float{}) or f(double{}): the handle's precision as a type
template <typename F>
auto with_precision(const enrgy_ctx* c, F&& f) {
  return c->precision == ENRGY_F32 ? f(float{}) : f(double{});
}

// terrain normals of the band for the in-kernel insolation; terrain: full raster laid out like the DEM buffer
cudaError_t launch_normals(enrgy_ctx* c, const float* terrain) {
  return with_precision(c, [&](auto r) {
    using R = decltype(r);
    return launch_terrain<R>(c->dem0, terrain, c->dem_pitch, c->rows, c->cols, c->pitch, c->band_row0, c->band_rows_pad,
                             c->p.cell_size, (R*)c->d_nx.p, (R*)c->d_ny.p, (R*)c->d_nz.p, c->stream);
  });
}

// the band's cells of three padded device state rasters src[q] (in the handle's precision) into the host
// buffers dst[q] (skipped when null) as float32 (dtype 32) or float64 (64)
int download_state(enrgy_ctx* c, int dtype, const unsigned char* const src[3], void* const dst[3]) {
  if (dtype != 32 && dtype != 64) return fail(ENRGY_ERR_ARG, "dtype must be 32 or 64");
  const size_t n = (size_t)c->band_rows * c->cols;
  const size_t osz = dtype == 32 ? 4 : 8;
  CU_TRY(c->d_stage.alloc(n * osz));
  for (int q = 0; q < 3; ++q) {
    if (!dst[q]) continue;
    CU_TRY(with_precision(c, [&](auto r) {
      using R = decltype(r);
      return launch_unpad_state<R>((const R*)src[q], c->pitch, c->band_rows, c->cols, dtype, c->d_stage.p, c->stream);
    }));
    c->launches++;
    CU_TRY(cudaMemcpyAsync(dst[q], c->d_stage.p, n * osz, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
  }
  return ENRGY_OK;
}

int use_device(enrgy_ctx* c) {
  if (!c) return fail(ENRGY_ERR_ARG, "null context");
  CU_TRY(cudaSetDevice(c->device));
  return ENRGY_OK;
}

// host [rows][cols] float -> device padded [rows_pad][pitch] float (padding = NaN)
int upload_padded(enrgy_ctx* c, const float* src, int rows, float* dst, int rows_pad) {
  CU_TRY(cudaMemsetAsync(dst, 0xFF, (size_t)rows_pad * c->pitch * sizeof(float), c->stream));
  CU_TRY(cudaMemcpy2DAsync(dst, (size_t)c->pitch * sizeof(float), src, (size_t)c->cols * sizeof(float),
                           (size_t)c->cols * sizeof(float), rows, cudaMemcpyHostToDevice, c->stream));
  return ENRGY_OK;
}

constexpr const char* kNanWhereDemValid = "%s is NaN at %llu cells where the DEM is valid; the reference would propagate NaN "
                                          "into only some of its area means there -- not supported";

// fails with ENRGY_ERR_MASK (nan_fmt, what, count) when d_other is NaN where the DEM of the band is valid
int check_mask(enrgy_ctx* c, const float* d_other, const char* what, const char* nan_fmt = kNanWhereDemValid) {
  CU_TRY(c->d_counters.alloc(2));
  CU_TRY(cudaMemsetAsync(c->d_counters.p, 0, 2 * sizeof(unsigned long long), c->stream));
  CU_TRY(launch_mask_check(c->dem0, c->dem_pitch, d_other, c->pitch, c->band_row0, c->band_rows, c->cols,
                           c->d_counters.p, c->stream));
  c->launches++;
  unsigned long long h[2];
  CU_TRY(cudaMemcpyAsync(h, c->d_counters.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  if (h[0] != 0) return fail(ENRGY_ERR_MASK, nan_fmt, what, h[0]);
  return ENRGY_OK;
}

template <typename R>
int upload_tables(enrgy_ctx* c) {
  const PrepassOutput& o = c->pre;
  const int T = c->n_steps;
  std::vector<StepRec<R>> st(T);
  for (int i = 0; i < T; ++i) {
    const StepRec<double>& s = o.steps[i];
    StepRec<R>& d = st[i];
    d.t_air = (R)s.t_air; d.lapse = (R)s.lapse; d.p_hpa = (R)s.p_hpa; d.e_aws = (R)s.e_aws;
    d.c_sens = (R)s.c_sens; d.c_lat = (R)s.c_lat; d.c_lwd = (R)s.c_lwd; d.c_lwu = (R)s.c_lwu;
    d.c_sw = (R)s.c_sw; d.c_melt = (R)s.c_melt; d.alb_w = (R)s.alb_w; d.snow_alb = (R)s.snow_alb;
    d.dsum = (R)s.dsum; d.dt = (R)s.dt; d.inv_dt = (R)s.inv_dt; d.c_lw0 = (R)s.c_lw0; d.c_lw1 = (R)s.c_lw1;
    d.dir_u = (R)s.dir_u; d.dir_e = (R)s.dir_e; d.dir_n = (R)s.dir_n;
    // (rounded DOWN into the kernel's precision: the test it feeds must stay conservative)
    d.tan2_min = (R)s.tan2_min;
    if ((double)d.tan2_min > s.tan2_min) d.tan2_min = std::nextafter(d.tan2_min, (R)-1);
    // the two integer codes travel as int32 bit patterns in the low word of their slots (no float -> int
    // conversion at the head of every step)
    const int32_t pair_code = (int32_t)s.alb_pair, sub_code = (int32_t)s.sub;
    d.alb_pair = (R)0; d.sub = (R)0;
    std::memcpy(&d.alb_pair, &pair_code, sizeof(int32_t));
    std::memcpy(&d.sub, &sub_code, sizeof(int32_t));
  }
  const size_t ns = o.subs.size();
  std::vector<SubRec<R>> sb(std::max<size_t>(ns, 1));
  for (size_t i = 0; i < ns; ++i) {
    sb[i].e = (R)o.subs[i].e; sb[i].n = (R)o.subs[i].n; sb[i].u = (R)o.subs[i].u; sb[i].b = (R)o.subs[i].b;
  }
  CU_TRY(c->d_steps.alloc(std::max<size_t>(T, 1) * sizeof(StepRec<R>)));
  CU_TRY(c->d_steps64.alloc(std::max<size_t>(T, 1)));
  CU_TRY(c->d_subs.alloc(sb.size() * sizeof(SubRec<R>)));
  CU_TRY(c->d_blocks.alloc(std::max<size_t>(o.blocks.size(), 1)));
  if (T) {
    CU_TRY(cudaMemcpyAsync(c->d_steps.p, st.data(), (size_t)T * sizeof(StepRec<R>), cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaMemcpyAsync(c->d_steps64.p, o.steps.data(), (size_t)T * sizeof(StepRec<double>), cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaMemcpyAsync(c->d_blocks.p, o.blocks.data(), o.blocks.size() * sizeof(TimeBlock), cudaMemcpyHostToDevice, c->stream));
  }
  if (ns) {
    CU_TRY(cudaMemcpyAsync(c->d_subs.p, sb.data(), ns * sizeof(SubRec<R>), cudaMemcpyHostToDevice, c->stream));
  }
  CU_TRY(cudaStreamSynchronize(c->stream));   // host vectors go out of scope
  return ENRGY_OK;
}

// per-step values of the stations (station blend): k = 0 the primary AWS, unused stations zero
template <typename R>
int upload_stations(enrgy_ctx* c) {
  const int T = c->n_steps;
  std::vector<StationRec<R>> recs((size_t)std::max(T, 1) * kMaxStations);
  for (int i = 0; i < T; ++i) {
    const StepRec<double>& s = c->pre.steps[i];
    StationRec<R>* r = &recs[(size_t)i * kMaxStations];
    r[0].t = (R)s.t_air; r[0].p = (R)s.p_hpa; r[0].e = (R)s.e_aws; r[0].cn = (R)0;
    const double n0 = c->forcing[(size_t)i * ENRGY_F_COUNT + ENRGY_F_CLOUD];
    for (int k = 1; k < kMaxStations; ++k) {
      if (k <= c->n_extra) {
        const double* v = &c->st_series[((size_t)(k - 1) * T + i) * ENRGY_ST_COUNT];
        const double tk = v[ENRGY_ST_T_AIR], pk = v[ENRGY_ST_PRESSURE];
        r[k].t = (R)tk;
        r[k].p = (R)pk;
        r[k].e = (R)(v[ENRGY_ST_RH] * sat_vapour_pressure(tk + 273.15, pk * 100));      // var_classes.py:83-85
        r[k].cn = (R)(v[ENRGY_ST_CLOUD] - n0);
      } else {
        r[k].t = r[k].p = r[k].e = r[k].cn = (R)0;
      }
    }
  }
  CU_TRY(c->d_strecs.alloc(recs.size() * sizeof(StationRec<R>)));
  CU_TRY(cudaMemcpyAsync(c->d_strecs.p, recs.data(), recs.size() * sizeof(StationRec<R>), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  return ENRGY_OK;
}
template <typename R>
void fill_station_args(const enrgy_ctx* c, KernelArgs<R>& a) {
  a.n_stations = 1 + c->n_extra;
  a.st_row[0] = (R)c->p.aws_row; a.st_col[0] = (R)c->p.aws_col; a.st_elev[0] = (R)c->p.elev_aws;
  for (int k = 1; k < kMaxStations; ++k) {
    a.st_row[k] = (R)c->st_row[k]; a.st_col[k] = (R)c->st_col[k]; a.st_elev[k] = (R)c->st_elev[k];
  }
  a.station_recs = (const StationRec<R>*)c->d_strecs.p;
  a.cloud_on = std::isnan(c->cloud_k) ? 0 : 1;
  a.cloud_neg_k = a.cloud_on ? (R)(-c->cloud_k) : (R)0;
}

// NaN fields of enrgy_params -> the reference's defaults
void resolve_defaults(enrgy_params& p) {
  auto dflt = [](double& v, double d) { if (std::isnan(v)) v = d; };
  dflt(p.zm, 0.001);                 // turbo.py:273-274
  dflt(p.z_h_or_e, p.zm / 10);       // turbo.py:275-277
  dflt(p.emissivity, 0.98);          // model.py:541-542
  dflt(p.max_ice_albedo, 0.45);      // model.py:325-326
  dflt(p.snow_density, 387.0);       // var_classes.py:9
  dflt(p.ice_density, 900.0);
  dflt(p.solar_const, 1367.0);       // saga_lighting.py:42
  dflt(p.transmittance, 0.70);       // saga_lighting.py:44
  dflt(p.hour_step, 0.25);           // saga_lighting.py:43
  dflt(p.sensible_corr, 1.0);
  dflt(p.latent_corr, 1.0);
}

// terrain at the AWS cell and its 8 neighbours (NaN outside the raster)
void aws_neighbourhood(const float* dem, int rows, int cols, int aws_row, int aws_col, float* nbhd /*[9]*/) {
  for (int dr = -1; dr <= 1; ++dr)
    for (int dc = -1; dc <= 1; ++dc) {
      const int r = aws_row + dr, x = aws_col + dc;
      nbhd[(dr + 1) * 3 + (dc + 1)] = (r >= 0 && r < rows && x >= 0 && x < cols) ? dem[(size_t)r * cols + x]
                                                                            : std::numeric_limits<float>::quiet_NaN();
    }
}

int check_forcing(int n_steps, const double* forcing) {
  for (int i = 0; i < n_steps; ++i) {
    const double* f = forcing + (size_t)i * ENRGY_F_COUNT;
    if (!(f[ENRGY_F_RH] <= 1.0)) return fail(ENRGY_ERR_RANGE, "row %d: HUMID must be a 0..1 fraction here (helpers.py:74-87)", i);
    if (!(f[ENRGY_F_DT] > 0)) return fail(ENRGY_ERR_RANGE, "row %d: time step must be > 0", i);
  }
  return ENRGY_OK;
}

// ---- early host pre-pass ----------------------------------------------------------------------
// The per-step scalars depend on the forcing table, the parameters and the DEM around the AWS cell
// only (not on the albedo / SWE rasters, unless the sub-surface model integrates the AWS cell).  So
// when the forcing arrives after the DEM, the pre-pass starts on a host thread right away and runs
// while the caller is still uploading rasters; enrgy_prepass() joins it.  Any call that changes an
// input of the pre-pass drops the early result first.
void fill_prepass_input(enrgy_ctx* c, PrepassInput& in) {
  in.p = c->p; in.precision = c->precision; in.rows = c->rows; in.cols = c->cols;
  in.albedo_offset = c->albedo_offset;
  in.dem = c->have_terrain ? (c->h_terrain.empty() ? nullptr : c->h_terrain.data()) : (c->h_dem.empty() ? nullptr : c->h_dem.data());
  in.n_steps = c->n_steps; in.forcing = c->forcing.data();
  std::memcpy(in.nbhd, c->aws_nbhd, sizeof(in.nbhd));
  in.pot_aws = c->pot_aws.data();
  in.alb_aws = c->alb_aws; in.swe_aws = c->swe_aws; in.layer_t_aws = c->layer_t_aws;
  if (c->stations_on) {
    in.n_extra = c->n_extra;
    std::memcpy(in.st_row, c->st_row, sizeof(in.st_row));
    std::memcpy(in.st_col, c->st_col, sizeof(in.st_col));
    std::memcpy(in.st_elev, c->st_elev, sizeof(in.st_elev));
    in.st_series = c->st_series.data();
    in.cloud_k = c->cloud_k;
  }
}
void drop_early_prepass(enrgy_ctx* c) {
  if (c->pre_thread.joinable()) c->pre_thread.join();
  c->pre_early = PrepassOutput{};
  c->pre_early_rc = -1000;   // "no early result"
}
void start_early_prepass(enrgy_ctx* c) {
  drop_early_prepass(c);
  if (!c->have_dem || !c->have_forcing || c->p.msm_layers > 0 || c->p.insol_mode != ENRGY_INSOL_COMPUTED) return;
  c->pre_early_rc = 0;
  PrepassInput in;                 // snapshot taken on the calling thread
  fill_prepass_input(c, in);
  c->pre_thread = std::thread([c, in]() { c->pre_early_rc = run_prepass(in, c->pre_early, c->pre_early_err); });
}

// the fused-kernel instance of this handle's mode
FusedVariant fused_variant(const enrgy_ctx* c, bool dump, int nm = 1, bool stats = true) {
  FusedVariant v;
  v.insol = c->p.insol_mode == ENRGY_INSOL_STREAMED ? kInsolStreamed : c->p.shadow ? kInsolMasked : kInsolComputed;
  v.msm = c->p.msm_layers > 0;
  v.dump = dump;
  v.nm = nm;
  v.stats = stats;
  v.ns = c->stations_on ? kMaxStations : 1;
  return v;
}

// arguments of a fused pass over the steps [t0, t1) of the handle's own state; masks: sunlit masks of this
// band from the run's sunlit sub-step sub0 (the first of step t0) on
template <typename R>
void fill_args(enrgy_ctx* c, int t0, int t1, const unsigned* masks, int sub0, KernelArgs<R>& a) {
  a = KernelArgs<R>{};
  a.rows_full = c->rows; a.cols = c->cols; a.pitch = c->pitch;
  a.band_row0 = c->band_row0; a.band_rows = c->band_rows; a.rows_pad_full = c->rows_pad_full;
  a.dem = c->dem0; a.dem_pitch = c->dem_pitch;
  a.mask_words = c->pitch / 32;
  a.mask_sub_stride = (size_t)c->band_rows_pad * a.mask_words;   // (rows_pad / 8) x words x 8
  a.nx = (const R*)c->d_nx.p; a.ny = (const R*)c->d_ny.p; a.nz = (const R*)c->d_nz.p;
  a.albedo = c->d_albedo.p;
  a.map_stride = c->band_elems;
  a.albedo_const = c->p.albedo_const;
  a.albedo_ice = (R)c->p.albedo_ice; a.albedo_snow = (R)c->p.albedo_snow;
  a.albedo_offset = (R)c->albedo_offset;
  a.max_ice_albedo = c->p.albedo_const ? (R)INFINITY : (R)c->p.max_ice_albedo;
  a.elev_aws = (R)c->p.elev_aws;
  a.swe = (R*)c->d_swe.p; a.total_snow = (R*)c->d_ts.p; a.total_ice = (R*)c->d_ti.p;
  a.swe_ref = c->defer ? (const R*)c->d_swe_ref.p : nullptr;
  a.update_total_snow = c->defer == 1 ? 0 : 1;
  a.pot = c->d_pot.p; a.pot_stride = c->band_elems; a.pot_t0 = c->pot_t0;
  a.layer_t = (R*)c->d_layer_t.p;
  a.layer_stride = c->band_elems;
  a.msm.layers = c->p.msm_layers;
  for (int l = 0; l < kMaxLayers; ++l) {
    const double d = l < c->p.msm_layers ? c->p.msm_depths[l] : 1.0;
    a.msm.d[l] = (R)d;
    a.msm.inv_d[l] = (R)(1.0 / d);
  }
  a.msm.c_ice = (R)kCice; a.msm.k_ice = (R)kKappaIce; a.msm.k_snow = (R)kKappaSnow;
  a.msm.rho_ice = (R)c->p.ice_density; a.msm.rho_snow = (R)c->p.snow_density;
  a.msm.inv_snow_density = (R)(1.0 / c->p.snow_density);
  a.msm.g0_ice = a.msm.k_ice * a.msm.c_ice * a.msm.rho_ice;
  a.msm.crd_ice = a.msm.c_ice * a.msm.rho_ice * a.msm.d[0];
  a.steps = (const StepRec<R>*)c->d_steps.p;
  a.subs = (const SubRec<R>*)c->d_subs.p;
  a.blocks = c->d_blocks.p;
  a.cap_steps = c->pre.cap_steps; a.cap_subs = c->pre.cap_subs;
  int b0 = 0;
  const auto& bl = c->pre.blocks;
  while (b0 < (int)bl.size() && bl[b0].t_end <= t0) ++b0;
  int b1 = b0;
  while (b1 < (int)bl.size() && bl[b1].t_begin < t1) ++b1;
  a.block_begin = b0; a.block_end = b1;
  a.t0 = t0; a.t1 = t1;
  a.tiles = c->d_tiles.p; a.n_tiles = c->n_tiles;
  a.masks = masks; a.mask_sub0 = sub0;
  // (prefetches stop at the last sub-step of the range; at sub0 when it has none)
  a.mask_sub_last = t1 > t0 ? std::max(c->pre.sub_first[t1 - 1] + c->pre.sub_count[t1 - 1] - 1, sub0) : sub0;
  if (c->stations_on) fill_station_args<R>(c, a);
}

int check_run_ready(enrgy_ctx* c, int t0, int t1) {
  if (!c->have_dem || !c->prepass_done) return fail(ENRGY_ERR_ARG, "set_dem / set_forcing / prepass must precede run");
  if (t0 < 0 || t1 > c->n_steps || t0 > t1) return fail(ENRGY_ERR_ARG, "step range [%d, %d) outside [0, %d)", t0, t1, c->n_steps);
  if (!c->p.albedo_const && c->n_maps == 0) return fail(ENRGY_ERR_ARG, "albedo maps not set");
  if (c->p.msm_layers > 0 && !c->have_msm) return fail(ENRGY_ERR_ARG, "enrgy_set_msm must precede run when msm_layers > 0");
  if (c->p.insol_mode == ENRGY_INSOL_STREAMED && t1 > t0 &&
      (t0 < c->pot_t0 || t1 > c->pot_t0 + c->pot_n)) {
    return fail(ENRGY_ERR_ARG, "insolation rasters resident for steps [%d, %d), run asks [%d, %d)",
                c->pot_t0, c->pot_t0 + c->pot_n, t0, t1);
  }
  return ENRGY_OK;
}

// ---- shading: sunlit masks by the line sweep (shade.cu) -------------------------------------------
// uint32 words of one sub-step's mask for a band of `rows` rows: [rows_pad / 8][pitch / 32][8]
size_t mask_words_per_sub(const enrgy_ctx* c, int rows) { return (size_t)round_up(std::max(rows, 1), 16) * (c->pitch / 32); }

// sweeps the sunlit sub-steps [sub0, sub1) of the run into the given destination segments
int sweep_range(enrgy_ctx* c, int sub0, int sub1, int n_seg, const SweepSeg* segs, cudaStream_t stream) {
  if (sub1 <= sub0) return ENRGY_OK;
  if (!c->d_scan.p) return fail(ENRGY_ERR_ARG, "shading is off for this handle (params.shadow = 0)");
  std::vector<SweepSub> row_subs, col_subs;
  std::vector<int> zenith;
  for (int i = sub0; i < sub1; ++i) {
    const ShadeRec& sr = c->pre.subs[i].shade;
    if (!std::isfinite(sr.dz) || (sr.dc_fix == 0 && sr.dr_fix == 0)) {   // sun at the zenith: nothing can shade
      zenith.push_back(i - sub0);
      continue;
    }
    bool row_type; int sigma, dfix;
    line_geometry(sr.dc_fix, sr.dr_fix, &row_type, &sigma, &dfix);
    SweepSub sw{};
    sw.dfix = dfix; sw.sigma = sigma; sw.dz = (double)sr.dz; sw.out = i - sub0; sw.out2 = i - sub0;
    (row_type ? row_subs : col_subs).push_back(sw);
  }
  // neighbours in the lists have similar directions: the Q warps of a CTA then sweep nearly the same
  // cells and share the terrain rows through L1 (the same hour of consecutive days)
  auto by_direction = [](const SweepSub& x, const SweepSub& y) { return x.sigma != y.sigma ? x.sigma < y.sigma : x.dfix < y.dfix; };
  std::stable_sort(row_subs.begin(), row_subs.end(), by_direction);
  std::stable_sort(col_subs.begin(), col_subs.end(), by_direction);
  // the sub-steps go to launch_sweep in slices of at most kSweepMaxRowSubs / kSweepMaxColSubs (CUDA grid
  // limits; a long run on a small raster holds millions of sub-steps in one chunk); the column-type ones
  // of a slice share one transposed temporary
  for (size_t i = 0; i < col_subs.size(); ++i) col_subs[i].out = (int)(i % kSweepMaxColSubs);   // slot in it
  const size_t n_slices = std::max((row_subs.size() + kSweepMaxRowSubs - 1) / kSweepMaxRowSubs,
                                   (col_subs.size() + kSweepMaxColSubs - 1) / kSweepMaxColSubs);
  SweepArgs a{};
  a.rows = c->rows; a.cols = c->cols;
  a.scan = c->d_scan.p + (size_t)kScanRowApron * scan_pitch(c->cols) + kScanColApron;
  a.scan_t = c->d_scan_t.p + (size_t)kScanRowApron * scan_pitch(c->rows) + kScanColApron;
  a.n_seg = n_seg;
  for (int q = 0; q < n_seg; ++q) a.seg[q] = segs[q];
  a.tmp_words = sweep_tmp_words(c->rows);
  CU_TRY(c->d_sweepsubs.alloc(row_subs.size() + col_subs.size() + 1));
  // (pageable source: the copy is staged before the call returns, the vectors may go out of scope)
  if (!row_subs.empty()) CU_TRY(cudaMemcpyAsync(c->d_sweepsubs.p, row_subs.data(), row_subs.size() * sizeof(SweepSub), cudaMemcpyHostToDevice, stream));
  if (!col_subs.empty()) CU_TRY(cudaMemcpyAsync(c->d_sweepsubs.p + row_subs.size(), col_subs.data(), col_subs.size() * sizeof(SweepSub), cudaMemcpyHostToDevice, stream));
  if (!col_subs.empty()) {
    CU_TRY(c->d_masktmp.alloc(std::min(col_subs.size(), (size_t)kSweepMaxColSubs) * (size_t)c->cols * a.tmp_words));
    a.tmp = c->d_masktmp.p;
  }
  for (int z : zenith) {
    for (int q = 0; q < n_seg; ++q) {
      const size_t words = (size_t)segs[q].rg * segs[q].words * 8;
      CU_TRY(cudaMemsetAsync(segs[q].ptr + (size_t)z * words, 0xFF, words * sizeof(unsigned), stream));
    }
  }
  CU_TRY(c->ev_sweep.begin(stream));
  for (size_t k = 0; k < n_slices; ++k) {
    // (stream order: the transpose of slice k has read the temporary before slice k + 1 sweeps into it)
    const size_t r0 = std::min(row_subs.size(), k * kSweepMaxRowSubs), r1 = std::min(row_subs.size(), r0 + kSweepMaxRowSubs);
    const size_t c0 = std::min(col_subs.size(), k * kSweepMaxColSubs), c1 = std::min(col_subs.size(), c0 + kSweepMaxColSubs);
    a.row_subs = c->d_sweepsubs.p + r0; a.n_row_subs = (int)(r1 - r0);
    a.col_subs = c->d_sweepsubs.p + row_subs.size() + c0; a.n_col_subs = (int)(c1 - c0);
    int n = 0;
    CU_TRY(launch_sweep(a, c->sm_count, stream, &n));
    c->launches += n;
  }
  CU_TRY(c->ev_sweep.end(stream));
  return ENRGY_OK;
}

// sunlit sub-steps of the steps [t0, t1) (0 for an empty range and for rows where the sun stays down)
int sunlit_subs(const enrgy_ctx* c, int t0, int t1) {
  return t1 > t0 ? c->pre.sub_first[t1 - 1] + c->pre.sub_count[t1 - 1] - c->pre.sub_first[t0] : 0;
}

// masks of [sub0, sub1) for this handle's own band in c->d_maskbuf (kept: they depend only on the
// terrain and the sub-step directions, so later runs, ensemble members and debug views reuse them);
// *masks = the mask of sub0, or null for an empty range (the kernel reads no mask in a row without a
// sunlit sub-step)
int ensure_masks(enrgy_ctx* c, int sub0, int sub1, cudaStream_t stream, const unsigned** masks) {
  if (sub1 <= sub0) {
    *masks = nullptr;
    return ENRGY_OK;
  }
  const size_t per = mask_words_per_sub(c, c->band_rows);
  bool hit = sub0 >= c->mask_sub0 && sub1 <= c->mask_sub1;
  for (int i = sub0; i < sub1 && hit; ++i) {
    hit = std::memcmp(&c->mask_shades[i - c->mask_sub0], &c->pre.subs[i].shade, sizeof(ShadeRec)) == 0;
  }
  if (!hit) {
    c->mask_sub0 = c->mask_sub1 = 0;
    CU_TRY(c->d_maskbuf.alloc((size_t)(sub1 - sub0) * per));
    SweepSeg sg{};
    sg.row0 = c->band_row0; sg.rows = c->band_rows; sg.rg = c->band_rows_pad / 8; sg.words = c->pitch / 32;
    sg.ptr = c->d_maskbuf.p;
    if (int e = sweep_range(c, sub0, sub1, 1, &sg, stream)) return e;
    c->mask_shades.resize(sub1 - sub0);
    for (int i = sub0; i < sub1; ++i) c->mask_shades[i - sub0] = c->pre.subs[i].shade;
    c->mask_sub0 = sub0; c->mask_sub1 = sub1;
  }
  *masks = c->d_maskbuf.p + (size_t)(sub0 - c->mask_sub0) * per;
  return ENRGY_OK;
}

struct Chunk { int t0, t1, s0, s1; };
// steps [t0, t1) cut so that the masks (and the transposed temporaries, worst case all of them) of a
// chunk fit the budget; one chunk when everything fits
std::vector<Chunk> plan_chunks(const enrgy_ctx* c, int t0, int t1) {
  const size_t per_sub = (mask_words_per_sub(c, c->band_rows) + (size_t)c->cols * sweep_tmp_words(c->rows)) * sizeof(unsigned);
  size_t budget = c->mask_budget;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
    // what is already held for masks counts as available
    const size_t held = (c->d_maskbuf.n + c->d_masktmp.n) * sizeof(unsigned);
    budget = std::min(budget, (free_b + held) / 2);
  }
  const int max_subs = (int)std::max<size_t>(budget / per_sub, 1);
  std::vector<Chunk> out;
  int t = t0;
  while (t < t1) {
    Chunk ch{t, t, c->pre.sub_first[t], c->pre.sub_first[t]};
    while (ch.t1 < t1 && (ch.t1 == ch.t0 || ch.s1 - ch.s0 + c->pre.sub_count[ch.t1] <= max_subs)) {
      ch.s1 += c->pre.sub_count[ch.t1];
      ++ch.t1;
    }
    out.push_back(ch);
    t = ch.t1;
  }
  return out;
}

// A run cut into several launches: defer_begin copies the SWE rasters at its start (stream-ordered; the
// handle's own, or one per fused member slot), the launches that follow leave total_snow alone, and after
// defer_last the next chunk adds swe(start of the run) - swe(end) -- exactly what a single launch over the
// whole range does.
int defer_begin(enrgy_ctx* c, const void* swe, size_t bytes, cudaStream_t stream) {
  CU_TRY(c->d_swe_ref.alloc(bytes));
  CU_TRY(cudaMemcpyAsync(c->d_swe_ref.p, swe, bytes, cudaMemcpyDeviceToDevice, stream));
  c->defer = 1;
  return ENRGY_OK;
}
void defer_last(enrgy_ctx* c) { if (c->defer == 1) c->defer = 2; }
void defer_done(enrgy_ctx* c) { if (c->defer == 2) c->defer = 0; }

// Runs the steps [t0, t1) as run_chunk(chunk, masks): with shading in chunks whose sunlit masks fit the
// budget (plan_chunks), each one's masks swept or found in the cache first; else as one chunk without
// masks.  A run of several chunks defers total_snow to its last chunk; swe: the run's SWE rasters (bytes).
template <typename F>
int run_chunks(enrgy_ctx* c, int t0, int t1, const void* swe, size_t bytes, cudaStream_t stream, F&& run_chunk) {
  const bool shaded = fused_variant(c, false).insol == kInsolMasked && t1 > t0;
  const std::vector<Chunk> chunks = shaded ? plan_chunks(c, t0, t1) : std::vector<Chunk>{Chunk{t0, t1, 0, 0}};
  if (chunks.size() > 1 && c->defer == 0) {
    if (int e = defer_begin(c, swe, bytes, stream)) return e;
  }
  for (size_t q = 0; q < chunks.size(); ++q) {
    const Chunk& ch = chunks[q];
    if (q + 1 == chunks.size() && chunks.size() > 1) defer_last(c);
    const unsigned* masks = nullptr;
    if (shaded) {
      if (int e = ensure_masks(c, ch.s0, ch.s1, stream, &masks)) return e;
    }
    if (int e = run_chunk(ch, masks)) return e;
    defer_done(c);
  }
  return ENRGY_OK;
}

// the first run on new state rasters turns their off-glacier cells into NaN (model.py:258)
template <typename R>
int nan_offglacier(enrgy_ctx* c, cudaStream_t stream) {
  if (c->state_advanced) return ENRGY_OK;
  CU_TRY(launch_nan_offglacier<R>(c->dem0, c->dem_pitch, c->pitch, c->band_row0, c->band_rows, c->cols, (R*)c->d_swe.p,
                                  (R*)c->d_ts.p, (R*)c->d_ti.p, stream));
  c->launches++;
  return ENRGY_OK;
}

// where the per-step statistics of one member of a fused pass go: its float64 step records, its rows
struct StatsOut { const StepRec<double>* steps64; double* stats; };

// one launch of the fused kernel variant v over a's steps; the statistics of the pass's members
// 0 .. n_out - 1 are finalized into out[]
template <typename R>
int fused_pass(enrgy_ctx* c, KernelArgs<R>& a, const FusedVariant& v, const StatsOut* out, int n_out, cudaStream_t stream) {
  LaunchInfo li;
  CU_TRY(configure_energy_balance<R>(v, c->sm_count, a.cap_steps, a.cap_subs, &li));
  const int grid = std::min(li.grid, std::max(c->n_tiles, 1));
  const int n = a.t1 - a.t0;
  const size_t partial_bytes = v.stats ? (size_t)grid * std::max(n, 1) * v.nm * (v.msm ? kStatsP : kStatsK) * sizeof(R) : 0;
  if (v.stats) {
    // (the launches are stream-ordered and finalize runs right behind its kernel: one buffer serves all)
    CU_TRY(c->d_partials.alloc(partial_bytes));
    CU_TRY(cudaMemsetAsync(c->d_partials.p, 0, partial_bytes, stream));
    a.partials = (R*)c->d_partials.p;
  }
  // The per-CTA statistic rows are read-modify-written once per tile and time block.  In float32 mode they
  // (42 MB for a season) stay in L2 by themselves; the float64 rows (twice the size) were evicted by the
  // raster traffic and came back from DRAM every time (ncu: 1.06 GB per season launch against 0.4 GB
  // algorithmic).  An L2 access-policy window pins them for the launch.
  const bool pin_rows = sizeof(R) == 8 && partial_bytes > 0 && c->l2_persist_max > 0;
  if (pin_rows) {
    cudaStreamAttrValue av{};
    av.accessPolicyWindow.base_ptr = c->d_partials.p;
    av.accessPolicyWindow.num_bytes = std::min(partial_bytes, (size_t)c->l2_window_max);
    av.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)c->l2_persist_max / (double)av.accessPolicyWindow.num_bytes);
    av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    CU_TRY(cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &av));
  }
  CU_TRY(c->ev_fused.begin(stream));
  CU_TRY(launch_energy_balance<R>(a, v, c->sm_count, grid, &c->info, stream));
  CU_TRY(c->ev_fused.end(stream));
  if (pin_rows) {
    cudaStreamAttrValue av{};
    av.accessPolicyWindow.num_bytes = 0;                 // window off for whatever follows on this stream
    CU_TRY(cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &av));
  }
  c->launches++;
  for (int k = 0; k < n_out && n > 0; ++k) {
    FinalizeArgs f{};
    f.partials = c->d_partials.p; f.n_ctas = grid; f.n_steps = n; f.t0 = a.t0;
    f.nm = v.nm; f.member = k;
    f.n_valid = c->n_valid; f.f32_mode = c->precision == ENRGY_F32; f.msm = v.msm ? 1 : 0;
    f.lwd_summed = v.ns > 1 ? 1 : 0;
    for (int q = 0; q < 5; ++q) f.mom[q] = c->mom[q];
    f.steps64 = out[k].steps64; f.stats = out[k].stats;
    f.override_first = (a.t0 == 0 && !c->state_advanced) ? 1 : 0;
    f.swe0_sum = c->swe0_sum; f.swe0_nsnow = c->swe0_nsnow; f.swe0_nvalid = c->swe0_nvalid;
    CU_TRY(launch_finalize(f, stream));
    c->launches++;
  }
  return ENRGY_OK;
}

// one fused pass of the handle's own state over [t0, t1) (+ statistics into d_stats); masks: sunlit masks
// of this band from the run's sunlit sub-step sub0 on (may be null when the range has no sunlit sub-step:
// the kernel reads a mask only inside a sub-step)
template <typename R>
int launch_range(enrgy_ctx* c, int t0, int t1, double* d_stats, cudaStream_t stream, const unsigned* masks, int sub0) {
  const FusedVariant v = fused_variant(c, false);
  if (v.insol == kInsolMasked && masks == nullptr && sunlit_subs(c, t0, t1) > 0)
    return fail(ENRGY_ERR_ARG, "no sunlit masks for a run with shading");
  KernelArgs<R> a;
  fill_args<R>(c, t0, t1, masks, sub0, a);
  if (t1 > t0) {
    if (int e = nan_offglacier<R>(c, stream)) return e;
  }
  const StatsOut out{c->d_steps64.p, d_stats};
  if (int e = fused_pass<R>(c, a, v, &out, d_stats ? 1 : 0, stream)) return e;
  if (t1 > t0) c->state_advanced = true;
  return ENRGY_OK;
}

template <typename R>
int run_typed(enrgy_ctx* c, int t0, int t1, double* d_stats, cudaStream_t stream) {
  c->ev_fused.reset();
  c->ev_sweep.reset();
  return run_chunks(c, t0, t1, c->d_swe.p, c->band_elems * sizeof(R), stream, [&](const Chunk& ch, const unsigned* masks) {
    return launch_range<R>(c, ch.t0, ch.t1, d_stats ? d_stats + (size_t)(ch.t0 - t0) * ENRGY_S_COUNT : nullptr, stream,
                           masks, ch.s0);
  });
}

template <typename R>
int dump_typed(enrgy_ctx* c, int t0, int t1, double* out) {
  const FusedVariant v = fused_variant(c, true);
  const int s0 = c->pre.sub_first[t0], s1 = c->pre.sub_first[t1 - 1] + c->pre.sub_count[t1 - 1];
  const unsigned* masks = nullptr;
  if (v.insol == kInsolMasked) {
    if (int e = ensure_masks(c, s0, s1, c->stream, &masks)) return e;
  }
  KernelArgs<R> a;
  fill_args<R>(c, t0, t1, masks, s0, a);
  const int n = t1 - t0;
  const size_t per_step = (size_t)ENRGY_D_COUNT * c->band_elems;
  CU_TRY(c->d_dump.alloc((size_t)n * per_step * sizeof(R)));
  CU_TRY(cudaMemsetAsync(c->d_dump.p, 0xFF, (size_t)n * per_step * sizeof(R), c->stream));
  a.dump = (R*)c->d_dump.p;
  a.dump_field_stride = c->band_elems;
  CU_TRY(launch_energy_balance<R>(a, v, c->sm_count, 0, nullptr, c->stream));
  c->launches++;
  std::vector<R> h((size_t)n * per_step);
  CU_TRY(cudaMemcpyAsync(h.data(), c->d_dump.p, h.size() * sizeof(R), cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  for (int s = 0; s < n; ++s)
    for (int fld = 0; fld < ENRGY_D_COUNT; ++fld)
      for (int r = 0; r < c->band_rows; ++r) {
        const R* src = h.data() + ((size_t)s * ENRGY_D_COUNT + fld) * c->band_elems + (size_t)r * c->pitch;
        double* dst = out + (((size_t)s * ENRGY_D_COUNT + fld) * c->band_rows + r) * c->cols;
        for (int x = 0; x < c->cols; ++x) dst[x] = (double)src[x];
      }
  return ENRGY_OK;
}

// ---- fused ensemble members (BASELINE config C5) ---------------------------------------------------
struct MemberSpec { double offset, zm, zhe, alb_ice, alb_snow; };

template <typename R>
int run_members_typed(enrgy_ctx* c, const std::vector<MemberSpec>& mem, const std::vector<PrepassOutput>& pres,
                      int t0, int t1, double* d_stats /* [n][t1 - t0][S_COUNT] or null */, double* totals_out /* host [n][4] or null */,
                      cudaStream_t stream) {
  const int n_members = (int)mem.size(), n = t1 - t0, T = c->n_steps;
  const int slots = (n_members + 1) / 2 * 2;                  // an odd count is padded by a copy of the last member
  const size_t be = c->band_elems, bytes = be * sizeof(R);
  // state of every member = the handle's current state
  CU_TRY(c->d_mstate.alloc((size_t)slots * 3 * bytes));
  R* const ms_swe = (R*)c->d_mstate.p;
  R* const ms_ts = ms_swe + (size_t)slots * be;
  R* const ms_ti = ms_ts + (size_t)slots * be;
  if (n > 0) {
    if (int e = nan_offglacier<R>(c, stream)) return e;
  }
  for (int m = 0; m < slots; ++m) {
    CU_TRY(cudaMemcpyAsync(ms_swe + (size_t)m * be, c->d_swe.p, bytes, cudaMemcpyDeviceToDevice, stream));
    CU_TRY(cudaMemcpyAsync(ms_ts + (size_t)m * be, c->d_ts.p, bytes, cudaMemcpyDeviceToDevice, stream));
    CU_TRY(cudaMemcpyAsync(ms_ti + (size_t)m * be, c->d_ti.p, bytes, cudaMemcpyDeviceToDevice, stream));
  }
  c->member_slots = slots;
  c->members_last = n_members;
  // groups of 4 members, then one of 2
  struct Group { int first, nm; };
  std::vector<Group> groups;
  for (int m = 0; m < slots;) {
    const int nm = slots - m >= 4 ? 4 : 2;
    groups.push_back({m, nm});
    m += nm;
  }
  auto member_of = [&](int slot) { return std::min(slot, n_members - 1); };
  // per-step member scalars [group][T][nm] and the float64 master records per member (finalize)
  std::vector<MemberRec<R>> recs((size_t)slots * std::max(T, 1));
  {
    size_t o = 0;
    for (const Group& g : groups)
      for (int t = 0; t < T; ++t)
        for (int k = 0; k < g.nm; ++k, ++o) {
          const StepRec<double>& sr = pres[member_of(g.first + k)].steps[t];
          recs[o].c_sens = (R)sr.c_sens;
          recs[o].c_lat = (R)sr.c_lat;
        }
  }
  CU_TRY(c->d_mrecs.alloc(recs.size() * sizeof(MemberRec<R>)));
  CU_TRY(c->d_msteps64.alloc((size_t)n_members * std::max(T, 1)));
  if (T) {
    CU_TRY(cudaMemcpyAsync(c->d_mrecs.p, recs.data(), recs.size() * sizeof(MemberRec<R>), cudaMemcpyHostToDevice, stream));
    for (int m = 0; m < n_members; ++m)
      CU_TRY(cudaMemcpyAsync(c->d_msteps64.p + (size_t)m * T, pres[m].steps.data(), (size_t)T * sizeof(StepRec<double>),
                             cudaMemcpyHostToDevice, stream));
  }
  c->ev_fused.reset();
  c->ev_sweep.reset();
  // with shading the sunlit masks of a chunk of steps are swept once and serve every group
  const int rc = run_chunks(c, t0, t1, ms_swe, (size_t)slots * bytes, stream, [&](const Chunk& ch, const unsigned* masks) {
    for (const Group& g : groups) {
      KernelArgs<R> a;
      fill_args<R>(c, ch.t0, ch.t1, masks, ch.s0, a);
      a.swe = ms_swe + (size_t)g.first * be;
      a.total_snow = ms_ts + (size_t)g.first * be;
      a.total_ice = ms_ti + (size_t)g.first * be;
      if (a.swe_ref) a.swe_ref += (size_t)g.first * be;
      a.member_stride = be;
      a.member_recs = (const MemberRec<R>*)c->d_mrecs.p + (size_t)g.first * T;     // groups are stored one after the other
      for (int k = 0; k < g.nm; ++k) {
        const MemberSpec& ms = mem[member_of(g.first + k)];
        a.member_offset[k] = (R)ms.offset;
        a.member_albedo_ice[k] = (R)ms.alb_ice;
        a.member_albedo_snow[k] = (R)ms.alb_snow;
      }
      std::vector<StatsOut> out;                        // (not for the padding copy)
      for (int m = g.first; d_stats && m < g.first + g.nm && m < n_members; ++m)
        out.push_back({c->d_msteps64.p + (size_t)m * T, d_stats + ((size_t)m * n + (ch.t0 - t0)) * ENRGY_S_COUNT});
      if (int e = fused_pass<R>(c, a, fused_variant(c, false, g.nm, d_stats != nullptr), out.data(), (int)out.size(), stream))
        return e;
    }
    return ENRGY_OK;
  });
  if (rc != ENRGY_OK) return rc;
  if (totals_out) {
    // glacier-wide means of the final rasters of every member (no per-step statistics needed)
    constexpr int kBlocks = 128;
    CU_TRY(c->d_small.alloc((size_t)n_members * kBlocks * 4));
    CU_TRY(launch_member_totals<R>(c->dem0, c->dem_pitch, c->pitch, c->band_row0, c->band_rows, c->cols, ms_swe, ms_ts, ms_ti, be,
                                   n_members, c->d_small.p, kBlocks, stream));
    c->launches++;
    std::vector<double> hb((size_t)n_members * kBlocks * 4);
    CU_TRY(cudaMemcpyAsync(hb.data(), c->d_small.p, hb.size() * sizeof(double), cudaMemcpyDeviceToHost, stream));
    CU_TRY(cudaStreamSynchronize(stream));
    for (int m = 0; m < n_members; ++m) {
      double acc[4] = {0, 0, 0, 0};
      for (int b = 0; b < kBlocks; ++b)
        for (int q = 0; q < 4; ++q) acc[q] += hb[((size_t)m * kBlocks + b) * 4 + q];
      for (int q = 0; q < 3; ++q) totals_out[m * 4 + q] = acc[3] > 0 ? acc[q] / acc[3] : NAN;
      totals_out[m * 4 + 3] = acc[3];
    }
  }
  CU_TRY(cudaStreamSynchronize(stream));                // `recs` goes out of scope
  return ENRGY_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int enrgy_abi_version(void) { return ENRGY_ABI_VERSION; }
const char* enrgy_last_error(void) { return g_err.c_str(); }

int enrgy_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int enrgy_create(int device, int rows, int cols, int precision, enrgy_ctx** out) {
  if (!out) return fail(ENRGY_ERR_ARG, "out is null");
  *out = nullptr;
  if (rows <= 0 || cols <= 0 || rows > kMaxSide || cols > kMaxSide)
    return fail(ENRGY_ERR_ARG, "raster %d x %d outside 1..%d", rows, cols, kMaxSide);
  if (precision != ENRGY_F32 && precision != ENRGY_F64) return fail(ENRGY_ERR_ARG, "precision must be 32 or 64");
  const int n = enrgy_device_count();
  if (n <= 0) return fail(ENRGY_ERR_NODEVICE, "no CUDA device visible; enrgy_b200 has no CPU fallback");
  if (device < 0 || device >= n) return fail(ENRGY_ERR_ARG, "device %d outside 0..%d", device, n - 1);
  CU_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    return fail(ENRGY_ERR_NODEVICE, "device %d is sm_%d%d; this library carries sm_100a code only", device,
                prop.major, prop.minor);
  }
  enrgy_ctx* c = new enrgy_ctx();
  c->device = device; c->rows = rows; c->cols = cols; c->precision = precision;
  c->sm_count = prop.multiProcessorCount;
  if (precision == ENRGY_F64 && prop.persistingL2CacheMaxSize > 0) {
    // room for the float64 statistic rows of a season (launch_range pins them); a hint, so failure is not fatal
    const size_t want = std::min<size_t>((size_t)prop.persistingL2CacheMaxSize, (size_t)80 << 20);
    if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
      c->l2_persist_max = (int)want;
      c->l2_window_max = prop.accessPolicyMaxWindowSize;
    } else {
      cudaGetLastError();
    }
  }
  c->pitch = round_up(cols, kTileW);
  c->rows_pad_full = round_up(rows, 16);
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
    delete c;
    return fail(ENRGY_ERR_CUDA, "stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
  }
  c->stream = c->own_stream;
  *out = c;
  return ENRGY_OK;
}

int enrgy_destroy(enrgy_ctx* c) {
  if (!c) return ENRGY_OK;
  drop_early_prepass(c);
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
  return ENRGY_OK;
}

int enrgy_set_params(enrgy_ctx* c, const enrgy_params* pin) {
  if (int e = use_device(c)) return e;
  if (!pin) return fail(ENRGY_ERR_ARG, "params is null");
  if (c->have_dem) return fail(ENRGY_ERR_ARG, "set_params must precede set_dem");
  drop_early_prepass(c);
  enrgy_params p = *pin;
  resolve_defaults(p);
  if (!(p.cell_size > 0)) return fail(ENRGY_ERR_ARG, "cell_size must be > 0");
  if (!(p.sensor_z > 0) || !(p.zm > 0) || !(p.z_h_or_e > 0)) return fail(ENRGY_ERR_ARG, "sensor_z, zm, z_h_or_e must be > 0");
  if (p.msm_layers < 0 || p.msm_layers > ENRGY_MAX_LAYERS - 1) return fail(ENRGY_ERR_ARG, "msm_layers outside 0..%d", ENRGY_MAX_LAYERS - 1);
  if (p.msm_layers > kMaxLayers) return fail(ENRGY_ERR_ARG, "msm_layers > %d", kMaxLayers);
  for (int l = 0; l < p.msm_layers; ++l) {
    if (!(p.msm_depths[l] > 0)) return fail(ENRGY_ERR_ARG, "msm layer %d: thickness must be > 0 (zero-thickness layers never occur in the reference's model path: update_layers is not called, msm.py:300)", l);
  }
  if (p.insol_mode != ENRGY_INSOL_STREAMED && p.insol_mode != ENRGY_INSOL_COMPUTED) return fail(ENRGY_ERR_ARG, "bad insol_mode");
  if (p.band_rows == 0) { p.band_row0 = 0; p.band_rows = c->rows; }
  if (p.band_row0 < 0 || p.band_rows < 0 || p.band_row0 + p.band_rows > c->rows) return fail(ENRGY_ERR_ARG, "row band outside the raster");
  // the sweep writes the sunlit masks in groups of 8 raster rows (shade.cu)
  if (p.shadow && (p.band_row0 & 7)) return fail(ENRGY_ERR_ARG, "with shading the row band must start on a multiple of 8 rows (band_row0 = %d)", p.band_row0);
  c->p = p;
  c->albedo_offset = 0.0;
  c->base_albedo_ice = p.albedo_ice; c->base_albedo_snow = p.albedo_snow;
  c->band_row0 = p.band_row0;
  c->band_rows = p.band_rows;
  with_precision(c, [&](auto r) { energy_balance_tile<decltype(r)>(p.msm_layers > 0, &c->tile_h, &c->tile_w); });
  c->have_msm = false;
  c->band_rows_pad = round_up(std::max(c->band_rows, 1), 16);
  c->band_elems = (size_t)c->band_rows_pad * c->pitch;
  c->have_params = true;
  return ENRGY_OK;
}

int enrgy_set_dem(enrgy_ctx* c, const float* dem) {
  if (int e = use_device(c)) return e;
  if (!c->have_params) return fail(ENRGY_ERR_ARG, "set_params must precede set_dem");
  if (!dem) return fail(ENRGY_ERR_ARG, "dem is null");
  drop_early_prepass(c);
  if (c->p.aws_row < 0 || c->p.aws_row >= c->rows || c->p.aws_col < 0 || c->p.aws_col >= c->cols)
    return fail(ENRGY_ERR_ARG, "AWS cell (%d, %d) outside the %d x %d raster", c->p.aws_row, c->p.aws_col, c->rows, c->cols);
  aws_neighbourhood(dem, c->rows, c->cols, c->p.aws_row, c->p.aws_col, c->aws_nbhd);
  if (c->p.insol_mode == ENRGY_INSOL_COMPUTED && c->p.shadow) {
    c->h_dem.assign(dem, dem + (size_t)c->rows * c->cols);
  } else {
    c->h_dem.clear();
    c->h_dem.shrink_to_fit();
  }
  c->have_terrain = false;
  c->h_terrain.clear();
  c->h_terrain.shrink_to_fit();
  c->d_terrain.release();
  c->mask_sub0 = c->mask_sub1 = 0;
  // DEM buffer [rows_pad_full][pitch], padding cells NaN
  c->dem_pitch = c->pitch;
  const size_t dem_elems = (size_t)c->rows_pad_full * c->dem_pitch;
  CU_TRY(c->d_dem.alloc(dem_elems));
  c->dem0 = c->d_dem.p;
  CU_TRY(cudaMemsetAsync(c->d_dem.p, 0xFF, dem_elems * sizeof(float), c->stream));
  {
    // Only the shading rays read the DEM outside the band; without them the band plus one row on
    // either side (terrain normals) is all the device needs -- on a multi-GPU run every rank then
    // uploads its share instead of the whole raster.  The rest of the buffer stays NaN.
    const bool need_all = c->p.insol_mode == ENRGY_INSOL_COMPUTED && c->p.shadow;
    const int r_a = need_all ? 0 : std::max(0, c->band_row0 - 1);
    const int r_b = need_all ? c->rows : std::min(c->rows, c->band_row0 + c->band_rows + 1);
    if (r_b > r_a) {
      CU_TRY(cudaMemcpy2DAsync(c->dem0 + (size_t)r_a * c->dem_pitch, (size_t)c->dem_pitch * sizeof(float),
                               dem + (size_t)r_a * c->cols, (size_t)c->cols * sizeof(float),
                               (size_t)c->cols * sizeof(float), r_b - r_a, cudaMemcpyHostToDevice, c->stream));
    }
  }
  // shading: scan copies of the terrain for the line sweep (shade.cu)
  if (c->p.insol_mode == ENRGY_INSOL_COMPUTED && c->p.shadow) {
    CU_TRY(c->d_scan.alloc(scan_elems(c->rows, c->cols)));
    CU_TRY(c->d_scan_t.alloc(scan_elems(c->cols, c->rows)));
    CU_TRY(launch_scan_prepare(c->dem0, c->dem_pitch, c->rows, c->cols, c->d_scan.p, c->d_scan_t.p, c->stream));
    c->launches += 3;
  } else {
    c->d_scan.release();
    c->d_scan_t.release();
  }
  // active tiles of the band
  c->tiles_r = (c->band_rows + c->tile_h - 1) / c->tile_h;
  c->tiles_c = c->pitch / c->tile_w;
  const int nt = c->tiles_r * c->tiles_c;
  CU_TRY(c->d_counts.alloc(std::max(nt, 1)));
  std::vector<int> counts(std::max(nt, 1), 0);
  if (nt > 0) {
    CU_TRY(launch_tile_scan(c->dem0, c->dem_pitch, c->band_row0, c->band_rows, c->cols, c->tile_h, c->tile_w,
                            c->tiles_r, c->tiles_c, c->d_counts.p, c->stream));
    c->launches++;
    CU_TRY(cudaMemcpyAsync(counts.data(), c->d_counts.p, (size_t)nt * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
  }
  std::vector<int2> tiles;
  double nv = 0.0;
  for (int tr = 0; tr < c->tiles_r; ++tr)
    for (int tc = 0; tc < c->tiles_c; ++tc) {
      const int n = counts[tr * c->tiles_c + tc];
      if (n > 0) {
        tiles.push_back(make_int2(tr, tc));
        nv += n;
      }
    }
  c->n_tiles = (int)tiles.size();
  c->n_valid = nv;
  CU_TRY(c->d_tiles.alloc(std::max<size_t>(tiles.size(), 1)));
  if (!tiles.empty()) CU_TRY(cudaMemcpyAsync(c->d_tiles.p, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, c->stream));
  // moments of the elevation difference (area sum of the downward longwave flux)
  {
    const int blocks = 296;
    CU_TRY(c->d_small.alloc((size_t)blocks * 5));
    CU_TRY(with_precision(c, [&](auto r) {
      return launch_moments<decltype(r)>(c->dem0, c->dem_pitch, c->band_row0, c->band_rows, c->cols, c->p.elev_aws,
                                         c->d_small.p, blocks, c->stream);
    }));
    c->launches++;
    std::vector<double> h((size_t)blocks * 5);
    CU_TRY(cudaMemcpyAsync(h.data(), c->d_small.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    for (int q = 0; q < 5; ++q) {
      c->mom[q] = 0.0;
      for (int b = 0; b < blocks; ++b) c->mom[q] += h[(size_t)b * 5 + q];
    }
  }
  // state rasters: zeros (model.py:76-80)
  const size_t rs = rsize(c);
  CU_TRY(c->d_swe.alloc(c->band_elems * rs));
  CU_TRY(c->d_ts.alloc(c->band_elems * rs));
  CU_TRY(c->d_ti.alloc(c->band_elems * rs));
  CU_TRY(cudaMemsetAsync(c->d_swe.p, 0, c->band_elems * rs, c->stream));
  CU_TRY(cudaMemsetAsync(c->d_ts.p, 0, c->band_elems * rs, c->stream));
  CU_TRY(cudaMemsetAsync(c->d_ti.p, 0, c->band_elems * rs, c->stream));
  c->swe0_sum = 0.0; c->swe0_nsnow = 0.0; c->swe0_nvalid = (double)c->band_rows * c->cols;
  c->state_advanced = false;
  // terrain normals for the in-kernel insolation
  if (c->p.insol_mode == ENRGY_INSOL_COMPUTED) {
    CU_TRY(c->d_nx.alloc(c->band_elems * rs));
    CU_TRY(c->d_ny.alloc(c->band_elems * rs));
    CU_TRY(c->d_nz.alloc(c->band_elems * rs));
    CU_TRY(launch_normals(c, c->dem0));
    c->launches++;
  }
  CU_TRY(cudaStreamSynchronize(c->stream));
  c->have_dem = true;
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_set_terrain(enrgy_ctx* c, const float* terrain) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "set_dem must precede set_terrain");
  if (!terrain) return fail(ENRGY_ERR_ARG, "terrain is null");
  if (c->p.insol_mode != ENRGY_INSOL_COMPUTED) return fail(ENRGY_ERR_ARG, "the terrain only matters with insol_mode = COMPUTED");
  drop_early_prepass(c);
  const size_t n = (size_t)c->rows * c->cols;
  {
    // every glacier cell needs terrain under it
    const int ar = c->p.aws_row, ac = c->p.aws_col;
    if (!(terrain[(size_t)ar * c->cols + ac] == terrain[(size_t)ar * c->cols + ac]))
      return fail(ENRGY_ERR_MASK, "the terrain raster is NaN at the AWS cell");
  }
  const size_t elems = (size_t)c->rows_pad_full * c->dem_pitch;
  CU_TRY(c->d_terrain.alloc(elems));
  CU_TRY(cudaMemsetAsync(c->d_terrain.p, 0xFF, elems * sizeof(float), c->stream));
  CU_TRY(cudaMemcpy2DAsync(c->d_terrain.p, (size_t)c->dem_pitch * sizeof(float), terrain, (size_t)c->cols * sizeof(float),
                           (size_t)c->cols * sizeof(float), c->rows, cudaMemcpyHostToDevice, c->stream));
  // (the band's rows of the DEM are on the device in every mode; the mask check needs no more)
  if (int e = check_mask(c, c->d_terrain.p + (size_t)c->band_row0 * c->dem_pitch, "the terrain raster",
                         "%s is NaN at %llu glacier cells"))
    return e;
  aws_neighbourhood(terrain, c->rows, c->cols, c->p.aws_row, c->p.aws_col, c->aws_nbhd);
  CU_TRY(launch_normals(c, c->d_terrain.p));
  c->launches++;
  if (c->p.shadow) {
    c->h_terrain.assign(terrain, terrain + n);
    CU_TRY(launch_scan_prepare(c->d_terrain.p, c->dem_pitch, c->rows, c->cols, c->d_scan.p, c->d_scan_t.p, c->stream));
    c->launches += 3;
  }
  CU_TRY(cudaStreamSynchronize(c->stream));
  c->have_terrain = true;
  c->mask_sub0 = c->mask_sub1 = 0;
  c->prepass_done = false;
  if (c->have_forcing) start_early_prepass(c);
  return ENRGY_OK;
}

int enrgy_set_albedo_maps(enrgy_ctx* c, int n_maps, const float* const* maps) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "set_dem must precede set_albedo_maps");
  if (n_maps < 1 || n_maps > 255 || !maps) return fail(ENRGY_ERR_ARG, "n_maps outside 1..255");
  CU_TRY(c->d_albedo.alloc((size_t)n_maps * c->band_elems));
  for (int m = 0; m < n_maps; ++m) {
    if (!maps[m]) return fail(ENRGY_ERR_ARG, "albedo map %d is null", m);
    float* dst = c->d_albedo.p + (size_t)m * c->band_elems;
    if (int e = upload_padded(c, maps[m], c->band_rows, dst, c->band_rows_pad)) return e;
    if (int e = check_mask(c, dst, "albedo map")) return e;
  }
  c->n_maps = n_maps;
  {
    const int ar = c->p.aws_row - c->band_row0;
    c->alb_aws.clear();
    if (ar >= 0 && ar < c->band_rows) {
      for (int m = 0; m < n_maps; ++m) c->alb_aws.push_back((double)maps[m][(size_t)ar * c->cols + c->p.aws_col]);
    }
  }
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_set_swe(enrgy_ctx* c, const float* swe) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "set_dem must precede set_swe");
  const size_t rs = rsize(c);
  if (!swe) {
    CU_TRY(cudaMemsetAsync(c->d_swe.p, 0, c->band_elems * rs, c->stream));
    c->swe0_sum = 0.0; c->swe0_nsnow = 0.0; c->swe0_nvalid = (double)c->band_rows * c->cols;
    c->swe_aws = 0.0;
    c->prepass_done = false;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return ENRGY_OK;
  }
  {
    const int ar = c->p.aws_row - c->band_row0;
    if (ar >= 0 && ar < c->band_rows) c->swe_aws = (double)swe[(size_t)ar * c->cols + c->p.aws_col];
  }
  c->prepass_done = false;
  CU_TRY(c->d_tmp32.alloc(c->band_elems));
  if (int e = upload_padded(c, swe, c->band_rows, c->d_tmp32.p, c->band_rows_pad)) return e;
  if (int e = check_mask(c, c->d_tmp32.p, "SWE raster")) return e;
  const int blocks = 296;
  CU_TRY(c->d_small.alloc((size_t)blocks * 3));
  CU_TRY(launch_swe0_stats(c->d_tmp32.p, c->pitch, c->band_rows, c->cols, c->d_small.p, blocks, c->stream));
  c->launches++;
  std::vector<double> h((size_t)blocks * 3);
  CU_TRY(cudaMemcpyAsync(h.data(), c->d_small.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(with_precision(c, [&](auto r) {
    using R = decltype(r);
    return launch_pad_convert<R>(c->d_tmp32.p, (R*)c->d_swe.p, c->band_elems, c->stream);
  }));
  c->launches++;
  CU_TRY(cudaStreamSynchronize(c->stream));
  c->swe0_sum = c->swe0_nsnow = c->swe0_nvalid = 0.0;
  for (int b = 0; b < blocks; ++b) {
    c->swe0_sum += h[b * 3 + 0]; c->swe0_nsnow += h[b * 3 + 1]; c->swe0_nvalid += h[b * 3 + 2];
  }
  c->state_advanced = false;
  return ENRGY_OK;
}

int enrgy_set_msm(enrgy_ctx* c, const double* temps, double elev) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "set_dem must precede set_msm");
  const int nl = c->p.msm_layers;
  if (nl <= 0) return fail(ENRGY_ERR_ARG, "msm_layers is 0 in the parameters");
  if (!temps) return fail(ENRGY_ERR_ARG, "temps is null");
  const size_t rs = rsize(c);
  CU_TRY(c->d_layer_t.alloc((size_t)(nl + 1) * c->band_elems * rs));
  c->layer_t_aws.assign(nl + 1, 0.0);
  CU_TRY(with_precision(c, [&](auto r) {
    using R = decltype(r);
    // the AWS cell's own boundary temperatures for the serial pre-pass, model.py:133-143, rounded like the kernel's
    const R d = (R)c->aws_nbhd[4] - (R)elev;
    for (int l = 0; l <= nl; ++l) {
      volatile R prod = d * (R)-0.006;
      const double t = (double)((R)temps[l] + prod);
      c->layer_t_aws[l] = t > 0 ? 0.0 : t;
    }
    return launch_msm_init<R>(c->dem0, c->dem_pitch, c->pitch, c->band_row0, c->band_rows_pad, nl + 1, temps, elev,
                              (R*)c->d_layer_t.p, c->band_elems, c->stream);
  }));
  c->launches++;
  c->have_msm = true;
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_set_member(enrgy_ctx* c, double albedo_offset, double zm, double z_h_or_e) {
  if (int e = use_device(c)) return e;
  if (!c->have_params) return fail(ENRGY_ERR_ARG, "set_params must precede set_member");
  drop_early_prepass(c);
  if (std::isnan(albedo_offset)) albedo_offset = 0.0;
  if (!std::isnan(zm)) {
    if (!(zm > 0)) return fail(ENRGY_ERR_ARG, "zm must be > 0");
    c->p.zm = zm;
  }
  if (!std::isnan(z_h_or_e)) {
    if (!(z_h_or_e > 0)) return fail(ENRGY_ERR_ARG, "z_h_or_e must be > 0");
    c->p.z_h_or_e = z_h_or_e;
  }
  c->albedo_offset = albedo_offset;
  auto clip = [](double a) { return std::min(std::max(a, 0.001), 1.0); };
  if (c->p.albedo_const) {
    c->p.albedo_ice = albedo_offset != 0.0 ? clip(c->base_albedo_ice + albedo_offset) : c->base_albedo_ice;
    c->p.albedo_snow = albedo_offset != 0.0 ? clip(c->base_albedo_snow + albedo_offset) : c->base_albedo_snow;
  }
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_set_stations(enrgy_ctx* c, int n_extra, const double* row, const double* col, const double* elev,
                       const double* series, double cloud_k) {
  if (int e = use_device(c)) return e;
  if (n_extra < 0) {                      // back to the reference's single AWS
    c->stations_on = false; c->n_extra = 0; c->st_series.clear(); c->cloud_k = NAN;
    c->prepass_done = false;
    return ENRGY_OK;
  }
  if (n_extra > kMaxStations - 1) return fail(ENRGY_ERR_ARG, "at most %d extra stations", kMaxStations - 1);
  if (!c->have_forcing) return fail(ENRGY_ERR_ARG, "set_forcing must precede set_stations (the series share its time base)");
  if (n_extra > 0 && (!row || !col || !elev || !series)) return fail(ENRGY_ERR_ARG, "set_stations: null arrays");
  if (!std::isnan(cloud_k) && cloud_k < 0) return fail(ENRGY_ERR_ARG, "cloud_k must be >= 0 (NaN = no cloud attenuation)");
  for (int k = 0; k < n_extra; ++k) {
    if (!std::isfinite(row[k]) || !std::isfinite(col[k]) || !std::isfinite(elev[k])) return fail(ENRGY_ERR_ARG, "station %d: position not finite", k + 1);
    c->st_row[k + 1] = row[k]; c->st_col[k + 1] = col[k]; c->st_elev[k + 1] = elev[k];
  }
  const size_t n = (size_t)n_extra * c->n_steps * ENRGY_ST_COUNT;
  for (size_t i = 0; i < n; ++i)
    if (!std::isfinite(series[i])) return fail(ENRGY_ERR_ARG, "station series: value %zu is not finite", i);
  c->st_series.assign(series, series + n);
  c->n_extra = n_extra;
  c->cloud_k = cloud_k;
  c->stations_on = true;
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_set_forcing(enrgy_ctx* c, int n_steps, const double* forcing) {
  if (int e = use_device(c)) return e;
  if (n_steps < 0 || (n_steps > 0 && !forcing)) return fail(ENRGY_ERR_ARG, "bad forcing table");
  if (int e = check_forcing(n_steps, forcing)) return e;
  drop_early_prepass(c);
  c->forcing.assign(forcing, forcing + (size_t)n_steps * ENRGY_F_COUNT);
  c->n_steps = n_steps;
  c->pot_aws.assign(n_steps, std::numeric_limits<double>::quiet_NaN());
  c->have_forcing = true;
  c->prepass_done = false;
  start_early_prepass(c);      // runs while the caller uploads the remaining rasters
  return ENRGY_OK;
}

int enrgy_set_insolation(enrgy_ctx* c, int t0, int n, const float* pot) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem || !c->have_forcing) return fail(ENRGY_ERR_ARG, "set_dem and set_forcing must precede set_insolation");
  if (c->p.insol_mode != ENRGY_INSOL_STREAMED) return fail(ENRGY_ERR_ARG, "insol_mode is not STREAMED");
  if (t0 < 0 || n < 0 || t0 + n > c->n_steps || (n > 0 && !pot)) return fail(ENRGY_ERR_ARG, "bad insolation window");
  CU_TRY(c->d_pot.alloc((size_t)std::max(n, 1) * c->band_elems));
  const size_t per = (size_t)c->band_rows * c->cols;
  const int ar = c->p.aws_row - c->band_row0;
  for (int i = 0; i < n; ++i) {
    float* dst = c->d_pot.p + (size_t)i * c->band_elems;
    if (int e = upload_padded(c, pot + (size_t)i * per, c->band_rows, dst, c->band_rows_pad)) return e;
    if (ar >= 0 && ar < c->band_rows) c->pot_aws[t0 + i] = (double)pot[(size_t)i * per + (size_t)ar * c->cols + c->p.aws_col];
  }
  // NaN masks: checked on the first raster of the window (the reference writes them all with one cutline)
  if (n > 0) {
    if (int e = check_mask(c, c->d_pot.p, "insolation raster")) return e;
  }
  CU_TRY(cudaStreamSynchronize(c->stream));
  c->pot_t0 = t0;
  c->pot_n = n;
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_set_insolation_aws(enrgy_ctx* c, int t0, int n, const double* pot_aws) {
  if (!c) return fail(ENRGY_ERR_ARG, "null context");
  if (!c->have_forcing) return fail(ENRGY_ERR_ARG, "set_forcing must precede set_insolation_aws");
  if (t0 < 0 || n < 0 || t0 + n > c->n_steps || (n > 0 && !pot_aws)) return fail(ENRGY_ERR_ARG, "bad insolation window");
  for (int i = 0; i < n; ++i) c->pot_aws[t0 + i] = pot_aws[i];
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_prepass(enrgy_ctx* c) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem || !c->have_forcing) return fail(ENRGY_ERR_ARG, "set_dem and set_forcing must precede prepass");
  if (c->p.insol_mode == ENRGY_INSOL_STREAMED) {
    for (int i = c->pot_t0; i < c->pot_t0 + c->pot_n; ++i)
      if (std::isnan(c->pot_aws[i]))
        return fail(ENRGY_ERR_ARG, "step %d: no potential insolation at the AWS cell -- it lies outside this handle's row band "
                                   "(hand its values in with enrgy_set_insolation_aws) or on a NaN cell of the rasters", i);
  }
  if (c->p.msm_layers > 0 && !c->have_msm) return fail(ENRGY_ERR_ARG, "enrgy_set_msm must precede prepass when msm_layers > 0");
  if (c->p.msm_layers > 0 && !c->p.albedo_const && (int)c->alb_aws.size() != c->n_maps)
    return fail(ENRGY_ERR_ARG, "the AWS cell lies outside this handle's row band: its albedo/SWE are needed for the sub-surface pre-pass");
  // (before the pre-pass: with the sub-surface model it reads the series)
  if (c->stations_on && (int)c->st_series.size() != c->n_extra * c->n_steps * ENRGY_ST_COUNT)
    return fail(ENRGY_ERR_ARG, "station series were set for another forcing table: call enrgy_set_stations after enrgy_set_forcing");
  int rc;
  std::string err;
  if (c->pre_thread.joinable()) {          // started by enrgy_set_forcing, inputs unchanged since
    c->pre_thread.join();
    rc = c->pre_early_rc;
    err = c->pre_early_err;
    c->pre = std::move(c->pre_early);
    c->pre_early = PrepassOutput{};
    c->pre_early_rc = -1000;
  } else {
    PrepassInput in;
    fill_prepass_input(c, in);
    rc = run_prepass(in, c->pre, err);
  }
  if (rc != ENRGY_OK) return fail(rc, "%s", err.c_str());
  if (int e = with_precision(c, [&](auto r) {
        using R = decltype(r);
        if (int e2 = upload_tables<R>(c)) return e2;
        return c->stations_on ? upload_stations<R>(c) : (int)ENRGY_OK;
      }))
    return e;
  c->prepass_done = true;
  return ENRGY_OK;
}

int enrgy_host_prepass(const enrgy_params* pin, int precision, int rows, int cols, const float* dem, int n_steps,
                       const double* forcing, const double* pot_aws, double* point_out) {
  if (!pin || !dem || (n_steps > 0 && (!forcing || !point_out))) return fail(ENRGY_ERR_ARG, "null argument");
  if (precision != ENRGY_F32 && precision != ENRGY_F64) return fail(ENRGY_ERR_ARG, "precision must be 32 or 64");
  if (rows <= 0 || cols <= 0 || rows > kMaxSide || cols > kMaxSide || n_steps < 0)
    return fail(ENRGY_ERR_ARG, "bad sizes: raster %d x %d (1..%d a side), %d steps", rows, cols, kMaxSide, n_steps);
  PrepassInput in;
  in.p = *pin;
  resolve_defaults(in.p);
  if (in.p.msm_layers > 0) return fail(ENRGY_ERR_ARG, "enrgy_host_prepass: the sub-surface model needs the cell state of a loaded handle");
  if (in.p.insol_mode == ENRGY_INSOL_STREAMED && n_steps > 0 && !pot_aws) return fail(ENRGY_ERR_ARG, "pot_aws is needed in streamed mode");
  if (in.p.aws_row < 0 || in.p.aws_row >= rows || in.p.aws_col < 0 || in.p.aws_col >= cols)
    return fail(ENRGY_ERR_ARG, "AWS cell (%d, %d) outside the %d x %d raster", in.p.aws_row, in.p.aws_col, rows, cols);
  in.precision = precision; in.rows = rows; in.cols = cols; in.dem = dem;
  aws_neighbourhood(dem, rows, cols, in.p.aws_row, in.p.aws_col, in.nbhd);
  in.n_steps = n_steps; in.forcing = forcing;
  std::vector<double> nan_pot(std::max(n_steps, 1), std::numeric_limits<double>::quiet_NaN());
  in.pot_aws = pot_aws ? pot_aws : nan_pot.data();
  if (int e = check_forcing(n_steps, forcing)) return e;
  PrepassOutput out;
  std::string err;
  const int rc = run_prepass(in, out, err);
  if (rc != ENRGY_OK) return fail(rc, "%s", err.c_str());
  if (n_steps > 0) std::memcpy(point_out, out.point.data(), out.point.size() * sizeof(double));
  return ENRGY_OK;
}

int enrgy_get_point_scalars(enrgy_ctx* c, double* out) {
  if (!c || !out) return fail(ENRGY_ERR_ARG, "null argument");
  if (!c->prepass_done) return fail(ENRGY_ERR_ARG, "prepass has not run");
  std::memcpy(out, c->pre.point.data(), c->pre.point.size() * sizeof(double));
  return ENRGY_OK;
}

int enrgy_get_point_layers(enrgy_ctx* c, double* out) {
  if (!c || !out) return fail(ENRGY_ERR_ARG, "null argument");
  if (!c->prepass_done) return fail(ENRGY_ERR_ARG, "prepass has not run");
  if (c->p.msm_layers <= 0) return fail(ENRGY_ERR_ARG, "the sub-surface model is off");
  const int nb = c->p.msm_layers + 1;
  for (int i = 0; i < c->n_steps; ++i)
    for (int l = 0; l < nb; ++l) out[(size_t)i * nb + l] = c->pre.point_layers[(size_t)i * (kMaxLayers + 1) + l];
  return ENRGY_OK;
}

int enrgy_set_aws_cell(enrgy_ctx* c, int n_maps, const double* albedo_at_aws, double swe_at_aws) {
  if (!c) return fail(ENRGY_ERR_ARG, "null context");
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "set_dem must precede set_aws_cell");
  if (n_maps < 0 || (n_maps > 0 && !albedo_at_aws)) return fail(ENRGY_ERR_ARG, "bad albedo list");
  if (n_maps > 0 && c->n_maps > 0 && n_maps != c->n_maps) return fail(ENRGY_ERR_ARG, "%d albedo values for %d maps", n_maps, c->n_maps);
  drop_early_prepass(c);
  c->alb_aws.assign(albedo_at_aws, albedo_at_aws + n_maps);
  c->swe_aws = swe_at_aws;
  c->prepass_done = false;
  return ENRGY_OK;
}

int enrgy_get_substeps(enrgy_ctx* c, int step, int max_sub, double* out, int* n_out) {
  if (!c || !out || !n_out) return fail(ENRGY_ERR_ARG, "null argument");
  if (!c->prepass_done) return fail(ENRGY_ERR_ARG, "prepass has not run");
  if (step < 0 || step >= c->n_steps) return fail(ENRGY_ERR_ARG, "step outside the forcing table");
  const int n = c->pre.sub_count[step], first = c->pre.sub_first[step];
  if (n > max_sub) return fail(ENRGY_ERR_ARG, "step has %d sunlit sub-steps, buffer holds %d", n, max_sub);
  for (int j = 0; j < n; ++j) {
    const SubHost& s = c->pre.subs[first + j];
    double* o = out + (size_t)j * 8;
    o[0] = s.e; o[1] = s.n; o[2] = s.u; o[3] = s.b; o[4] = s.d;
    o[5] = s.shade.dc_fix; o[6] = s.shade.dr_fix; o[7] = (double)s.shade.dz;
  }
  *n_out = n;
  return ENRGY_OK;
}

int enrgy_run_async(enrgy_ctx* c, int t0, int t1, double* d_stats, void* stream) {
  if (int e = use_device(c)) return e;
  if (int e = check_run_ready(c, t0, t1)) return e;
  cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
  return with_precision(c, [&](auto r) { return run_typed<decltype(r)>(c, t0, t1, d_stats, s); });
}

int enrgy_run(enrgy_ctx* c, int t0, int t1, double* stats_out) {
  if (int e = use_device(c)) return e;
  if (int e = check_run_ready(c, t0, t1)) return e;
  const int n = t1 - t0;
  double* d_stats = nullptr;
  if (stats_out && n > 0) {
    CU_TRY(c->d_stats.alloc((size_t)n * ENRGY_S_COUNT));
    d_stats = c->d_stats.p;
  }
  const int rc = with_precision(c, [&](auto r) { return run_typed<decltype(r)>(c, t0, t1, d_stats, c->stream); });
  if (rc != ENRGY_OK) return rc;
  if (d_stats) CU_TRY(cudaMemcpyAsync(stats_out, d_stats, (size_t)n * ENRGY_S_COUNT * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  return ENRGY_OK;
}

int enrgy_run_members(enrgy_ctx* c, int n_members, const double* albedo_offset, const double* zm, const double* z_h_or_e,
                      int t0, int t1, double* stats_out, double* totals_out) {
  if (int e = use_device(c)) return e;
  if (n_members < 1 || !albedo_offset) return fail(ENRGY_ERR_ARG, "run_members: at least one member with an albedo offset");
  if (!c->have_dem || !c->have_forcing) return fail(ENRGY_ERR_ARG, "set_dem and set_forcing must precede run_members");
  if (c->stations_on) return fail(ENRGY_ERR_ARG, "run_members: not with the station blend (enrgy_set_stations)");
  if (c->p.msm_layers > 0)
    return fail(ENRGY_ERR_ARG, "run_members: the sub-surface model keeps 8 temperatures per cell and member -- run such members "
                               "one after the other (enrgy_set_member + enrgy_run)");
  drop_early_prepass(c);
  // the handle's own member settings come back afterwards
  const enrgy_params p_saved = c->p;
  const double off_saved = c->albedo_offset;
  auto clip = [](double a) { return std::min(std::max(a, 0.001), 1.0); };
  std::vector<MemberSpec> mem(n_members);
  std::vector<PrepassOutput> pres(n_members);
  int rc = ENRGY_OK;
  std::string err;
  for (int m = 0; m < n_members && rc == ENRGY_OK; ++m) {
    MemberSpec& ms = mem[m];
    ms.offset = std::isnan(albedo_offset[m]) ? 0.0 : albedo_offset[m];
    ms.zm = (zm && !std::isnan(zm[m])) ? zm[m] : p_saved.zm;
    ms.zhe = (z_h_or_e && !std::isnan(z_h_or_e[m])) ? z_h_or_e[m] : p_saved.z_h_or_e;
    if (!(ms.zm > 0) || !(ms.zhe > 0)) { rc = ENRGY_ERR_ARG; err = "run_members: roughness lengths must be > 0"; break; }
    ms.alb_ice = ms.offset != 0.0 ? clip(c->base_albedo_ice + ms.offset) : c->base_albedo_ice;
    ms.alb_snow = ms.offset != 0.0 ? clip(c->base_albedo_snow + ms.offset) : c->base_albedo_snow;
    c->p = p_saved;
    c->p.zm = ms.zm; c->p.z_h_or_e = ms.zhe;
    if (c->p.albedo_const) { c->p.albedo_ice = ms.alb_ice; c->p.albedo_snow = ms.alb_snow; }
    c->albedo_offset = ms.offset;
    PrepassInput in;
    fill_prepass_input(c, in);
    rc = run_prepass(in, pres[m], err);
  }
  if (rc == ENRGY_OK) {
    // the member-invariant records (forcing, insolation, time blocks) are those of the first member
    c->p = p_saved;
    c->p.zm = mem[0].zm; c->p.z_h_or_e = mem[0].zhe;
    if (c->p.albedo_const) { c->p.albedo_ice = mem[0].alb_ice; c->p.albedo_snow = mem[0].alb_snow; }
    c->albedo_offset = mem[0].offset;
    c->pre = pres[0];
    const int n = t1 - t0;
    double* d_stats = nullptr;
    rc = with_precision(c, [&](auto r) {
      using R = decltype(r);
      if (int e = upload_tables<R>(c)) return e;
      c->prepass_done = true;
      if (int e = check_run_ready(c, t0, t1)) return e;
      if (stats_out && n > 0) {
        cudaError_t ce = c->d_stats.alloc((size_t)n_members * n * ENRGY_S_COUNT);
        if (ce != cudaSuccess) return fail(ENRGY_ERR_CUDA, "cudaMalloc of the member statistics failed: %s", cudaGetErrorString(ce));
        d_stats = c->d_stats.p;
      }
      return run_members_typed<R>(c, mem, pres, t0, t1, d_stats, totals_out, c->stream);
    });
    if (rc == ENRGY_OK && d_stats) {
      cudaError_t ce = cudaMemcpyAsync(stats_out, d_stats, (size_t)n_members * n * ENRGY_S_COUNT * sizeof(double),
                                       cudaMemcpyDeviceToHost, c->stream);
      if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->stream);
      if (ce != cudaSuccess) rc = fail(ENRGY_ERR_CUDA, "download of the member statistics failed: %s", cudaGetErrorString(ce));
    }
  } else if (!err.empty()) {
    rc = fail(rc, "%s", err.c_str());
  }
  // back to the handle's own settings: its tables must be rebuilt by the next enrgy_prepass
  c->p = p_saved;
  c->albedo_offset = off_saved;
  c->prepass_done = false;
  return rc;
}

int enrgy_get_member_state(enrgy_ctx* c, int member, int dtype, void* swe, void* total_snow, void* total_ice) {
  if (int e = use_device(c)) return e;
  if (member < 0 || member >= c->members_last) return fail(ENRGY_ERR_ARG, "member %d outside the last run_members (%d members)", member, c->members_last);
  const size_t be = c->band_elems * rsize(c);
  const unsigned char* src[3];
  for (int q = 0; q < 3; ++q) src[q] = c->d_mstate.p + ((size_t)q * c->member_slots + member) * be;
  void* const dst[3] = {swe, total_snow, total_ice};
  return download_state(c, dtype, src, dst);
}

int enrgy_synchronize(enrgy_ctx* c) {
  if (int e = use_device(c)) return e;
  CU_TRY(cudaDeviceSynchronize());
  return ENRGY_OK;
}

int enrgy_dump_steps(enrgy_ctx* c, int t0, int t1, double* out) {
  if (int e = use_device(c)) return e;
  if (int e = check_run_ready(c, t0, t1)) return e;
  if (!out) return fail(ENRGY_ERR_ARG, "out is null");
  if (t1 == t0) return ENRGY_OK;
  return with_precision(c, [&](auto r) { return dump_typed<decltype(r)>(c, t0, t1, out); });
}

int enrgy_shade_masks(enrgy_ctx* c, int step, int max_sub, uint32_t* out, int* n_sub_out) {
  if (int e = use_device(c)) return e;
  if (int e = check_run_ready(c, step, step + 1)) return e;
  if (!out) return fail(ENRGY_ERR_ARG, "out is null");
  if (fused_variant(c, false).insol != kInsolMasked) return fail(ENRGY_ERR_ARG, "shade masks need insol_mode = COMPUTED with shadow = 1");
  const int s0 = c->pre.sub_first[step], n_sub = c->pre.sub_count[step];
  if (n_sub > max_sub) return fail(ENRGY_ERR_ARG, "step has %d sunlit sub-steps, buffer holds %d", n_sub, max_sub);
  if (n_sub_out) *n_sub_out = n_sub;
  if (n_sub == 0) return ENRGY_OK;
  const unsigned* masks = nullptr;
  if (int e = ensure_masks(c, s0, s0 + n_sub, c->stream, &masks)) return e;
  const size_t per = mask_words_per_sub(c, c->band_rows);
  std::vector<unsigned> h((size_t)n_sub * per);
  CU_TRY(cudaMemcpyAsync(h.data(), masks, h.size() * sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  // device layout [sub][row / 8][word][row % 8] -> [sub][row][word]; off-glacier cells and the bits
  // beyond the last column read "sunlit"
  const int words = (c->cols + 31) / 32, dwords = c->pitch / 32;
  for (int j = 0; j < n_sub; ++j)
    for (int r = 0; r < c->band_rows; ++r) {
      uint32_t* dst = out + ((size_t)j * c->band_rows + r) * words;
      for (int w = 0; w < words; ++w) {
        unsigned v = h[(size_t)j * per + (((size_t)(r >> 3) * dwords + w) * 8) + (r & 7)];
        const float* drow = c->h_dem.data() + (size_t)(r + c->band_row0) * c->cols;
        for (int b = 0; b < 32; ++b) {
          const int x = w * 32 + b;
          if (x >= c->cols || !(drow[x] == drow[x])) v |= 1u << b;
        }
        dst[w] = v;
      }
    }
  return ENRGY_OK;
}

int enrgy_sub_range(enrgy_ctx* c, int t0, int t1, int* sub0, int* sub1) {
  if (!c || !sub0 || !sub1) return fail(ENRGY_ERR_ARG, "null argument");
  if (!c->prepass_done) return fail(ENRGY_ERR_ARG, "prepass has not run");
  if (t0 < 0 || t1 > c->n_steps || t0 > t1) return fail(ENRGY_ERR_ARG, "step range [%d, %d) outside [0, %d)", t0, t1, c->n_steps);
  const int total = (int)c->pre.subs.size();
  *sub0 = t0 < c->n_steps ? c->pre.sub_first[t0] : total;
  *sub1 = t1 > t0 ? c->pre.sub_first[t1 - 1] + c->pre.sub_count[t1 - 1] : *sub0;
  return ENRGY_OK;
}

int64_t enrgy_mask_words(enrgy_ctx* c, int rows) {
  if (!c || rows <= 0) return 0;
  return (int64_t)mask_words_per_sub(c, rows);
}

int enrgy_shade_scan(enrgy_ctx* c, int sub0, int sub1, int n_seg, const int* seg_row0, const int* seg_rows,
                     void* const* seg_ptr, void* stream) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem || !c->prepass_done) return fail(ENRGY_ERR_ARG, "set_dem / set_forcing / prepass must precede shade_scan");
  if (fused_variant(c, false).insol != kInsolMasked) return fail(ENRGY_ERR_ARG, "shade_scan needs insol_mode = COMPUTED with shadow = 1");
  if (sub0 < 0 || sub1 > (int)c->pre.subs.size() || sub0 > sub1) return fail(ENRGY_ERR_ARG, "sub-step range outside the run");
  if (n_seg < 1 || n_seg > kMaxSweepSegs || !seg_row0 || !seg_rows || !seg_ptr) return fail(ENRGY_ERR_ARG, "1..%d row segments", kMaxSweepSegs);
  SweepSeg segs[kMaxSweepSegs];
  for (int q = 0; q < n_seg; ++q) {
    if (seg_row0[q] < 0 || seg_rows[q] <= 0 || seg_row0[q] + seg_rows[q] > c->rows || (seg_row0[q] & 7) || !seg_ptr[q])
      return fail(ENRGY_ERR_ARG, "segment %d: rows [%d, %d) must lie inside the raster and start on a multiple of 8", q, seg_row0[q], seg_row0[q] + seg_rows[q]);
    segs[q].row0 = seg_row0[q]; segs[q].rows = seg_rows[q];
    segs[q].rg = round_up(seg_rows[q], 16) / 8; segs[q].words = c->pitch / 32;
    segs[q].ptr = static_cast<unsigned*>(seg_ptr[q]);
  }
  c->ev_sweep.reset();
  return sweep_range(c, sub0, sub1, n_seg, segs, stream ? (cudaStream_t)stream : c->stream);
}

int enrgy_run_masked(enrgy_ctx* c, int t0, int t1, const void* d_masks, double* d_stats, void* stream) {
  if (int e = use_device(c)) return e;
  if (int e = check_run_ready(c, t0, t1)) return e;
  if (fused_variant(c, false).insol != kInsolMasked) return fail(ENRGY_ERR_ARG, "run_masked needs insol_mode = COMPUTED with shadow = 1");
  if (!d_masks && sunlit_subs(c, t0, t1) > 0) return fail(ENRGY_ERR_ARG, "d_masks is null");
  cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
  c->ev_fused.reset();
  const int sub0 = t0 < c->n_steps ? c->pre.sub_first[t0] : 0;
  const int rc = with_precision(c, [&](auto r) {
    return launch_range<decltype(r)>(c, t0, t1, d_stats, s, static_cast<const unsigned*>(d_masks), sub0);
  });
  if (rc == ENRGY_OK) defer_done(c);
  return rc;
}

int enrgy_potential_insolation(enrgy_ctx* c, int step, double* out) {
  if (int e = use_device(c)) return e;
  if (!out) return fail(ENRGY_ERR_ARG, "out is null");
  std::vector<double> tmp((size_t)ENRGY_D_COUNT * c->band_rows * c->cols);
  if (int e = enrgy_dump_steps(c, step, step + 1, tmp.data())) return e;
  std::memcpy(out, tmp.data() + (size_t)ENRGY_D_POT * c->band_rows * c->cols, (size_t)c->band_rows * c->cols * sizeof(double));
  return ENRGY_OK;
}

int enrgy_get_state(enrgy_ctx* c, int dtype, void* swe, void* total_snow, void* total_ice) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "no state before set_dem");
  const unsigned char* const src[3] = {c->d_swe.p, c->d_ts.p, c->d_ti.p};
  void* const dst[3] = {swe, total_snow, total_ice};
  return download_state(c, dtype, src, dst);
}

int enrgy_set_state(enrgy_ctx* c, int dtype, const void* swe, const void* total_snow, const void* total_ice) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "set_dem must precede set_state");
  if (dtype != 32 && dtype != 64) return fail(ENRGY_ERR_ARG, "dtype must be 32 or 64");
  const void* srcs[3] = {swe, total_snow, total_ice};
  unsigned char* dsts[3] = {c->d_swe.p, c->d_ts.p, c->d_ti.p};
  const size_t rs = rsize(c);
  std::vector<unsigned char> host(c->band_elems * rs);
  for (int q = 0; q < 3; ++q) {
    if (!srcs[q]) continue;
    // host-side pad + convert (restart path, not on the hot path)
    for (size_t i = 0; i < c->band_elems; ++i) {
      if (rs == 4) ((float*)host.data())[i] = std::numeric_limits<float>::quiet_NaN();
      else ((double*)host.data())[i] = std::numeric_limits<double>::quiet_NaN();
    }
    for (int r = 0; r < c->band_rows; ++r)
      for (int x = 0; x < c->cols; ++x) {
        const size_t si = (size_t)r * c->cols + x, di = (size_t)r * c->pitch + x;
        const double v = dtype == 32 ? (double)((const float*)srcs[q])[si] : ((const double*)srcs[q])[si];
        if (rs == 4) ((float*)host.data())[di] = (float)v;
        else ((double*)host.data())[di] = v;
      }
    CU_TRY(cudaMemcpyAsync(dsts[q], host.data(), host.size(), cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
  }
  // a restart from a SWE raster of an earlier run: the first-row SWE quirk no longer applies (seeding
  // the totals alone, as Energy.model does for repeated calls, leaves it in force)
  if (swe) c->state_advanced = true;
  return ENRGY_OK;
}

int enrgy_get_layer_temps(enrgy_ctx* c, double* out) {
  if (int e = use_device(c)) return e;
  if (!c->have_msm) return fail(ENRGY_ERR_ARG, "the sub-surface model is not set up");
  if (!out) return fail(ENRGY_ERR_ARG, "out is null");
  const int nb = c->p.msm_layers + 1;
  const size_t rs = rsize(c);
  std::vector<unsigned char> h((size_t)nb * c->band_elems * rs);
  CU_TRY(cudaMemcpyAsync(h.data(), c->d_layer_t.p, h.size(), cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  for (int l = 0; l < nb; ++l)
    for (int r = 0; r < c->band_rows; ++r)
      for (int x = 0; x < c->cols; ++x) {
        const size_t si = (size_t)l * c->band_elems + (size_t)r * c->pitch + x;
        const double v = rs == 4 ? (double)((const float*)h.data())[si] : ((const double*)h.data())[si];
        out[((size_t)l * c->band_rows + r) * c->cols + x] = v;
      }
  return ENRGY_OK;
}

int enrgy_snapshot(enrgy_ctx* c, int save) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "no state before set_dem");
  const size_t bytes = c->band_elems * rsize(c);
  unsigned char* st[3] = {c->d_swe.p, c->d_ts.p, c->d_ti.p};
  const size_t lbytes = c->have_msm ? (size_t)(c->p.msm_layers + 1) * bytes : 0;
  if (save) {
    CU_TRY(c->d_snap.alloc(3 * bytes + lbytes));
    if (lbytes) CU_TRY(cudaMemcpyAsync(c->d_snap.p + 3 * bytes, c->d_layer_t.p, lbytes, cudaMemcpyDeviceToDevice, c->stream));
    for (int q = 0; q < 3; ++q)
      CU_TRY(cudaMemcpyAsync(c->d_snap.p + q * bytes, st[q], bytes, cudaMemcpyDeviceToDevice, c->stream));
    c->snap_valid = true;
    c->snap_advanced = c->state_advanced;
  } else {
    if (!c->snap_valid) return fail(ENRGY_ERR_ARG, "no snapshot to restore");
    if (lbytes) CU_TRY(cudaMemcpyAsync(c->d_layer_t.p, c->d_snap.p + 3 * bytes, lbytes, cudaMemcpyDeviceToDevice, c->stream));
    for (int q = 0; q < 3; ++q)
      CU_TRY(cudaMemcpyAsync(st[q], c->d_snap.p + q * bytes, bytes, cudaMemcpyDeviceToDevice, c->stream));
    c->state_advanced = c->snap_advanced;
  }
  return ENRGY_OK;
}

int enrgy_set_stream(enrgy_ctx* c, void* stream) {
  if (int e = use_device(c)) return e;
  CU_TRY(cudaStreamSynchronize(c->stream));
  c->stream = stream ? (cudaStream_t)stream : c->own_stream;
  return ENRGY_OK;
}

int enrgy_microbench(enrgy_ctx* c, int kind, double* result) {
  if (int e = use_device(c)) return e;
  if (!result || kind < 0 || kind > 3) return fail(ENRGY_ERR_ARG, "bad microbench request");
  CU_TRY(c->d_stage.alloc((size_t)c->sm_count * 8 * 256 * 8));
  const int iters = kind == 1 ? 2000 : 4000;
  double ops = 0.0, best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CU_TRY(cudaEventRecord(c->ev0, c->stream));
    CU_TRY(launch_microbench(kind, c->sm_count, iters, c->d_stage.p, &ops, c->stream));
    CU_TRY(cudaEventRecord(c->ev1, c->stream));
    CU_TRY(cudaEventSynchronize(c->ev1));
    c->launches++;
    float ms = 0.f;
    CU_TRY(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    if (rep > 0 && ms > 0.f) best = std::max(best, ops / (ms * 1e-3));
  }
  *result = (kind <= 1) ? best / 1e12 : best / 1e9;
  return ENRGY_OK;
}

int64_t enrgy_launch_count(enrgy_ctx* c) { return c ? c->launches : 0; }

double enrgy_last_kernel_ms(enrgy_ctx* c) {
  if (!c) return 0.0;
  cudaSetDevice(c->device);
  return c->ev_fused.collect();
}

double enrgy_last_sweep_ms(enrgy_ctx* c) {
  if (!c) return 0.0;
  cudaSetDevice(c->device);
  return c->ev_sweep.collect();
}

int enrgy_defer_snow_total(enrgy_ctx* c, int on) {
  if (int e = use_device(c)) return e;
  if (!c->have_dem) return fail(ENRGY_ERR_ARG, "no state before set_dem");
  if (on) return defer_begin(c, c->d_swe.p, c->band_elems * rsize(c), c->stream);
  defer_last(c);
  return ENRGY_OK;
}

int enrgy_set_mask_budget(enrgy_ctx* c, int64_t bytes) {
  if (!c || bytes <= 0) return fail(ENRGY_ERR_ARG, "bad mask budget");
  c->mask_budget = (size_t)bytes;
  return ENRGY_OK;
}

int enrgy_kernel_info(enrgy_ctx* c, int* regs, int* smem_bytes, int* ctas_per_sm, int* grid) {
  if (!c) return fail(ENRGY_ERR_ARG, "null context");
  if (regs) *regs = c->info.regs;
  if (smem_bytes) *smem_bytes = c->info.smem_bytes;
  if (ctas_per_sm) *ctas_per_sm = c->info.ctas_per_sm;
  if (grid) *grid = c->info.grid;
  return ENRGY_OK;
}

}  // extern "C"
