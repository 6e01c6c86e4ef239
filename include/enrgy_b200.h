/*
 * enrgy_b200 -- C ABI of the B200-native surface-energy-balance engine.
 *
 * Drop-in boundary for ONE hot path of tepextepex/ENRGY: everything `Energy.model` executes per
 * raster cell and per AWS row (reference model.py:183-283).  The reference has no FFI of its own
 * (it is pure Python, SURVEY.md 8b); the entry points below are what a binding for that path has
 * to offer, each citing the reference code it stands in for.  INTEGRATION.md shows the ctypes stub
 * a maintainer of the reference would add to model.py.
 *
 * Conventions: plain C, no exceptions across the boundary; every function returns 0 on success or
 * a negative ENRGY_ERR_* code and leaves a message for enrgy_last_error() (thread-local).  No
 * global state: one handle = one GPU context (row band / ensemble member), several handles may
 * live in one process.  Host rasters are C-contiguous [rows][cols] float32, row 0 = north, NaN =
 * off-glacier (GDAL order as read by reference raster_utils.py:36-53); the caller keeps ownership,
 * the library copies.  There is NO CPU fallback: without a CUDA device enrgy_create fails.
 */
#ifndef ENRGY_B200_H
#define ENRGY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ENRGY_ABI_VERSION 1

/* error codes */
#define ENRGY_OK 0
#define ENRGY_ERR_ARG (-1)       /* bad argument / call order */
#define ENRGY_ERR_CUDA (-2)      /* CUDA runtime error (message holds cudaGetErrorString) */
#define ENRGY_ERR_NODEVICE (-3)  /* no usable CUDA device: the product path has no CPU fallback */
#define ENRGY_ERR_MASK (-4)      /* NaN masks of the input rasters disagree with the DEM's */
#define ENRGY_ERR_RANGE (-5)     /* value outside the reference's accepted range (helpers.py:87) */

/* arithmetic type of the per-cell path */
#define ENRGY_F32 32 /* mirrors the as-shipped float32 rasters/state (model.py:76-80), 1e-4 */
#define ENRGY_F64 64 /* float64 everywhere (float32 wind fill kept, var_classes.py:170), 1e-9 */

/* where the potential insolation raster of a step comes from (reference model.py:464-481) */
#define ENRGY_INSOL_STREAMED 0 /* caller uploads kWh m-2 rasters (the use_precomputed/pickle path) */
#define ENRGY_INSOL_COMPUTED 1 /* computed in the fused kernel (replaces saga_lighting.py:7-53) */

/* columns of the forcing table, one row per AWS CSV row (reference model.py:186-230) */
enum {
  ENRGY_F_TIME = 0,     /* DATE as seconds since 1970-01-01 UTC */
  ENRGY_F_DT,           /* time step [s], helpers.py:63-71 (forward difference, last = previous) */
  ENRGY_F_T_AIR,        /* T_AIR [deg C] */
  ENRGY_F_WIND,         /* WIND_SPEED [m/s], raw: 0 -> 0.1 is applied inside (var_classes.py:81-82) */
  ENRGY_F_PRESSURE,     /* PRESSURE [hPa] */
  ENRGY_F_RH,           /* HUMID as a 0..1 fraction (after helpers.py:74-87) */
  ENRGY_F_CLOUD,        /* CLOUDINESS 0..1 after cloud_corr and clamping (model.py:200-204) */
  ENRGY_F_SWD,          /* SWD [W m-2] measured at the AWS */
  ENRGY_F_LAPSE,        /* air temperature lapse rate of this row [deg C / m] (model.py:213-221) */
  ENRGY_F_ALB_I0,       /* index of the albedo map dated at/before the row (interpolator.py:23-39) */
  ENRGY_F_ALB_I1,       /* index of the albedo map dated at/after the row */
  ENRGY_F_ALB_DAYS,     /* whole days since map I0 (interpolator.py:18) */
  ENRGY_F_ALB_SPAN,     /* whole days between I0 and I1; 0 = use I0 as is (interpolator.py:15-16) */
  ENRGY_F_SNOW_DAYS,    /* whole days since last_snowfall if > 0 else 0 (model.py:314-320) */
  ENRGY_F_COUNT
};

/* columns of the per-step statistics (SUMS over valid cells + counts; means are formed by the
 * caller exactly as var_classes.py:45-56 and model.py:246-252 print them) */
enum {
  ENRGY_S_RS = 0,       /* sum of net shortwave  rs = incoming * (1 - albedo)   model.py:497 */
  ENRGY_S_LWD,          /* sum of downward longwave                             model.py:544 */
  ENRGY_S_LWU,          /* sum of upward longwave                               model.py:543 */
  ENRGY_S_SENS,         /* sum of sensible heat flux                            turbo.py:156 */
  ENRGY_S_LAT,          /* sum of latent heat flux                              turbo.py:182-191 */
  ENRGY_S_ATMO,         /* sum of rs + lwd - lwu + sens + lat                   model.py:411 */
  ENRGY_S_G,            /* sum of the in-glacier flux (0 without the sub-surface model) */
  ENRGY_S_MELT,         /* sum of the flux available for melt                   model.py:434-438 */
  ENRGY_S_SNOW,         /* sum of snow melt [m w.e.]                            msm.py:199 */
  ENRGY_S_ICE,          /* sum of ice melt [m w.e.]                             msm.py:202 */
  ENRGY_S_SWE,          /* sum of SWE BEFORE this step's update                 model.py:248 */
  ENRGY_S_NSNOW,        /* count of cells with SWE > 0 (before the update)      model.py:250 */
  ENRGY_S_NSWE,         /* count of cells with non-NaN SWE (before the update)  model.py:251 */
  ENRGY_S_NVALID,       /* count of cells every flux mean runs over */
  ENRGY_S_COUNT
};

/* columns of the per-step scalars the pre-pass derives at the AWS cell (for solar_output.csv,
 * the POINT_T_SURF column and debugging) */
enum {
  ENRGY_P_L = 0,        /* Monin-Obukhov length [m]           turbo.py:88-137 */
  ENRGY_P_CH,           /* CH = CE of the distributed pass    turbo.py:264-290 */
  ENRGY_P_POT_AWS,      /* potential insolation at the AWS cell [W m-2]  model.py:512-514 */
  ENRGY_P_SW_FACTOR,    /* observed / potential scaling factor            model.py:523-526 */
  ENRGY_P_TSURF_AWS,    /* surface temperature at the AWS cell [deg C]    model.py:347 */
  ENRGY_P_QH_AWS,       /* point sensible flux of the last iteration */
  ENRGY_P_NSUB,         /* number of sunlit sub-steps of the row */
  ENRGY_P_SENS_AWS,     /* distributed sensible flux at the AWS cell [W m-2]  model.py:443 */
  ENRGY_P_LAT_AWS,      /* distributed latent flux at the AWS cell [W m-2]    model.py:444 */
  ENRGY_P_COUNT
};

/* fields of a per-step raster dump (debug views, same arithmetic as the production kernel) */
enum {
  ENRGY_D_RS = 0, ENRGY_D_LWD, ENRGY_D_LWU, ENRGY_D_SENS, ENRGY_D_LAT, ENRGY_D_ATMO, ENRGY_D_MELT,
  ENRGY_D_SNOW, ENRGY_D_ICE, ENRGY_D_ALBEDO, ENRGY_D_POT, ENRGY_D_G,
  ENRGY_D_COUNT
};

#define ENRGY_MAX_LAYERS 8

typedef struct enrgy_params {
  /* --- geometry / AWS (model.py:155, raster_utils.py:85-89) --- */
  double cell_size;      /* [m] */
  double elev_aws;       /* [m] */
  int32_t aws_row;       /* raster line of the AWS cell  (-int((uly - N) / dy)) */
  int32_t aws_col;       /* raster pixel of the AWS cell (int((E - ulx) / dx)) */
  double sensor_z;       /* measurement height z [m] */
  /* --- turbulent fluxes (turbo.py:264-290; config_template.json "turbo") --- */
  double zm;             /* roughness length for momentum; NaN = reference default 0.001 */
  double z_h_or_e;       /* scalar roughness length; NaN = zm / 10 */
  int32_t andreas;       /* 1 = Andreas (1987) scalar roughness, turbo.py:228-261 */
  int32_t _pad0;
  double sensible_corr;  /* model.py:386 */
  double latent_corr;    /* model.py:387 */
  /* --- longwave (model.py:533-545) --- */
  double emissivity;     /* NaN = 0.98 */
  /* --- albedo (model.py:298-337) --- */
  int32_t albedo_const;  /* 1 = constant (ice, snow) pair, 0 = interpolated maps */
  int32_t _pad1;
  double albedo_ice;
  double albedo_snow;
  double max_ice_albedo; /* NaN = 0.45 */
  /* --- melt (var_classes.py:7-15) --- */
  double snow_density;   /* NaN = 387 */
  double ice_density;    /* NaN = 900 */
  /* --- insolation (saga_lighting.py:42-44 options) --- */
  int32_t insol_mode;    /* ENRGY_INSOL_* */
  int32_t shadow;        /* != 0: topographic shading (SAGA -SHADOW), a line sweep over the terrain per sub-step */
  double lat_deg;        /* grid reference latitude / longitude for the sun position */
  double lon_deg;
  double solar_const;    /* NaN = 1367 */
  double transmittance;  /* NaN = 0.70 */
  double hour_step;      /* NaN = 0.25 h.  Computed insolation: a step may hold at most 255 SUNLIT
                            sub-steps of this length, so dt <= 63.75 h always passes at the default;
                            enrgy_prepass refuses a step with more with ENRGY_ERR_RANGE */
  /* --- sub-surface model (model.py:126-149, msm.py:31-107) --- */
  int32_t msm_layers;    /* 0 = off; else number of layer THICKNESSES (boundaries = layers + 1) */
  int32_t _pad2;
  double msm_depths[ENRGY_MAX_LAYERS];
  /* --- row band of a larger raster (multi-GPU, SURVEY 8e) --- */
  int32_t band_row0;     /* first row of this handle's band inside the full DEM; a multiple of 8
                            when shadow != 0 (enrgy_set_params returns ENRGY_ERR_ARG otherwise) */
  int32_t band_rows;     /* rows of the band; 0 = whole raster */
} enrgy_params;

typedef struct enrgy_ctx enrgy_ctx;

/* ABI version / build info ------------------------------------------------------------------ */
int enrgy_abi_version(void);
const char* enrgy_last_error(void);
/* number of CUDA devices visible (0 = none; never falls back to the CPU) */
int enrgy_device_count(void);

/* life cycle: replaces Energy.__init__ state allocation (model.py:74-80) ---------------------- */
/* rows and cols must lie in 1 .. 1048576 (2^20), else ENRGY_ERR_ARG.  The bound keeps every int cell
 * coordinate and the Q16 shear of the shading sweep far from overflow, keeps the float32 cell
 * coordinates of the station blend exact (< 2^24) and u * dz of the sweep exact in float64.  Device
 * memory binds long before it: a raster that does not fit fails with ENRGY_ERR_CUDA when its buffers
 * are allocated (enrgy_set_dem and the calls after it). */
int enrgy_create(int device, int rows, int cols, int precision, enrgy_ctx** out);
int enrgy_destroy(enrgy_ctx* ctx);

/* parameters of model() / config_template.json (model.py:155-158) */
int enrgy_set_params(enrgy_ctx* ctx, const enrgy_params* p);

/* rasters: base DEM (model.py:74), albedo maps (model.py:160-165, already clipped to [0.001, 1]),
 * initial SWE (model.py:122-124; NULL = zeros, model.py:79).  The DEM passed here is the FULL
 * raster even for a row band (it is replicated for the shading rays, SURVEY 8e; without shading only
 * the band and one row on either side are copied to the device). */
int enrgy_set_dem(enrgy_ctx* ctx, const float* dem);
/* optional: the UNCROPPED terrain on the model grid, [rows][cols], NaN = no terrain.  The reference
 * hands SAGA the uncropped DEM file (model.py:469 -> saga_lighting.py:42) and only crops the result,
 * so relief outside the glacier outline shades the glacier and shapes the slopes at its margin.
 * Without this call the (cropped) DEM is its own terrain: off-glacier cells then never cast a shadow.
 * Call after enrgy_set_dem; glacier cells must have terrain under them (ENRGY_ERR_MASK). */
int enrgy_set_terrain(enrgy_ctx* ctx, const float* terrain);
int enrgy_set_albedo_maps(enrgy_ctx* ctx, int n_maps, const float* const* maps);
int enrgy_set_swe(enrgy_ctx* ctx, const float* swe);
/* initial sub-surface boundary temperatures at the AWS reference elevation (model.py:126-143):
 * temps[msm_layers + 1], distributed with -0.006 K/m from elev and capped at 0 inside. */
int enrgy_set_msm(enrgy_ctx* ctx, const double* temps, double elev);

/* ensemble member on an already loaded handle (BASELINE config C5; the reference has no ensemble
 * code -- a member is "the reference run on perturbed inputs"): albedo_offset is added to every
 * albedo map / constant albedo and the result clipped to [0.001, 1] exactly as the loader clips a
 * raster (raster_utils.py:48-50); zm / z_h_or_e replace the roughness lengths (NaN = keep).  The
 * DEM, terrain, albedo maps and forcing stay resident; call enrgy_set_swe (or enrgy_snapshot
 * restore), enrgy_prepass and enrgy_run afterwards. */
int enrgy_set_member(enrgy_ctx* ctx, double albedo_offset, double zm, double z_h_or_e);

/* n_members ensemble members in FUSED passes of the kernel (4 members per pass, a remainder in pairs):
 * everything a member does not change -- terrain, insolation of every sub-step incl. the sunlit masks,
 * lapse-rate meteorology, flux factors, net longwave -- is computed once per cell-step and shared; each
 * member keeps its own SWE / ice-melt total / (1 - albedo) per cell in registers.  Every member starts
 * from the handle's current state and runs steps [t0, t1); the handle's own state is left alone.
 * albedo_offset[n_members]; zm / z_h_or_e [n_members] or NULL (NaN entries = the handle's value);
 * stats_out [n_members][t1 - t0][ENRGY_S_COUNT] or NULL: without it the passes skip the per-step area
 * statistics altogether (a third of a member's share of a step).  totals_out [n_members][4] or NULL:
 * glacier-wide means of the final swe, total_snow, total_ice rasters and the glacier cell count.
 * The state rasters equal enrgy_set_member + enrgy_prepass + enrgy_run of each member on its own bit for
 * bit; the float32 statistics agree to rounding (the passes sum in another order).  Not with the
 * sub-surface model (ENRGY_ERR_ARG).  The handle needs enrgy_prepass again before a plain enrgy_run. */
int enrgy_run_members(enrgy_ctx* ctx, int n_members, const double* albedo_offset, const double* zm,
                      const double* z_h_or_e, int t0, int t1, double* stats_out, double* totals_out);
/* state rasters of one member of the last enrgy_run_members (layout as enrgy_get_state) */
int enrgy_get_member_state(enrgy_ctx* ctx, int member, int dtype, void* swe, void* total_snow, void* total_ice);

/* Several weather stations and cloud attenuation of the shortwave (BASELINE config C4).  The reference
 * supports one AWS (model.py:155, var_classes.py:94-125) and has no cloud term in the shortwave: this is
 * THIS REPO's specification, stated in oracle/enrgy_oracle.py ("several weather stations") and built so
 * that without extra stations it is the reference's arithmetic.  Extra station k sits at (row[k], col[k])
 * of the FULL raster in cell units (cell centres, fractions allowed) at elev[k] m and reports
 * series[k][step][ENRGY_ST_*] on the forcing table's time base (call after enrgy_set_forcing).  Per cell:
 * inverse-squared-distance weights (softened by half a cell) over the primary AWS and the extra stations;
 * T, p, e reduced to the cell's elevation with the reference's lapse formulas and blended; wind, the
 * Monin-Obukhov solve, exchange coefficients, lapse rate, longwave cloudiness and the observed shortwave
 * factor stay the primary station's.  cloud_k >= 0: incoming shortwave times exp(-cloud_k * (blended
 * cloudiness - the primary station's)); NaN: off.  n_extra = 0 runs the blend with the primary station
 * alone (same rasters as a plain run); n_extra < 0 switches it off.  With the sub-surface model the blended
 * T, p and e (and the cloud factor) drive the surface temperature terms and the conduction step of every
 * cell, and the pre-pass integrates the AWS cell in the blend at that cell (its weights give the extra
 * stations a share there too): enrgy_get_point_layers, ENRGY_P_TSURF_AWS and ENRGY_P_SENS_AWS /
 * ENRGY_P_LAT_AWS then describe the AWS cell of the blended field.  (Without the sub-surface model the two
 * flux columns keep the AWS values reduced to the cell's elevation.)  Not with enrgy_run_members.  At most
 * 3 extra stations. */
enum enrgy_station_col {
  ENRGY_ST_T_AIR = 0,   /* T_AIR [deg C] */
  ENRGY_ST_PRESSURE,    /* PRESSURE [hPa] */
  ENRGY_ST_RH,          /* HUMID as a 0..1 fraction (after helpers.py:74-87) */
  ENRGY_ST_CLOUD,       /* CLOUDINESS 0..1 after cloud_corr and clamping (model.py:200-204) */
  ENRGY_ST_COUNT
};
int enrgy_set_stations(enrgy_ctx* ctx, int n_extra, const double* row, const double* col, const double* elev,
                       const double* series, double cloud_k);

/* forcing table [n_steps][ENRGY_F_COUNT] (model.py:182-230).  With in-kernel insolation and no
 * sub-surface model the host pre-pass needs nothing else besides the DEM, so it is started here on a
 * worker thread: call this right after enrgy_set_dem and the pre-pass runs while the albedo / SWE
 * rasters upload; enrgy_prepass() then only joins it (any other call order works, just without the
 * overlap). */
int enrgy_set_forcing(enrgy_ctx* ctx, int n_steps, const double* forcing);

/* streamed insolation (model.py:471-481): kWh m-2 rasters of steps [t0, t0 + n) */
int enrgy_set_insolation(enrgy_ctx* ctx, int t0, int n, const float* pot);

/* pre-pass: per-step scalars at the AWS cell (model.py:347-358, :500-530, turbo.py:88-137) */
/* streamed insolation on a row band that does not hold the AWS cell: the potential insolation AT the AWS
 * cell for steps [t0, t0 + n) [kWh m-2], which the observed / potential shortwave factor needs
 * (model.py:500-530).  enrgy_set_insolation fills it by itself when the cell lies inside the band;
 * enrgy_prepass fails if a resident step has none. */
int enrgy_set_insolation_aws(enrgy_ctx* ctx, int t0, int n, const double* pot_aws);
int enrgy_prepass(enrgy_ctx* ctx);
int enrgy_get_point_scalars(enrgy_ctx* ctx, double* out /* [n_steps][ENRGY_P_COUNT] */);
/* sub-surface model: boundary temperatures of the AWS cell BEFORE each row's update (the columns
 * debug_point_output prints when msm_xy is the AWS cell, model.py:421-426); out [n_steps][msm_layers + 1].
 * With the station blend: the cell integrated in the blended meteorology (enrgy_set_stations). */
int enrgy_get_point_layers(enrgy_ctx* ctx, double* out);
/* the AWS cell's own values for a handle whose row band does not hold it (the sub-surface pre-pass
 * integrates that cell on every rank): its albedo-map values and initial SWE.  Call after
 * enrgy_set_albedo_maps / enrgy_set_swe. */
int enrgy_set_aws_cell(enrgy_ctx* ctx, int n_maps, const double* albedo_at_aws, double swe_at_aws);
/* the same pre-pass WITHOUT a device or a handle (host arithmetic only): the per-row scalars of
 * model.py:347-358 / :500-530 for a full host DEM [rows][cols] -- Monin-Obukhov length, CH, potential
 * insolation and shortwave factor at the AWS cell, sunlit sub-step count.  pot_aws: potential
 * insolation at the AWS cell per row [kWh m-2] in streamed mode, else NULL.  Not available with the
 * sub-surface model (its pre-pass integrates the AWS cell from the loaded state). */
int enrgy_host_prepass(const enrgy_params* params, int precision, int rows, int cols, const float* dem,
                       int n_steps, const double* forcing, const double* pot_aws,
                       double* point_out /* [n_steps][ENRGY_P_COUNT] */);

/* the hot path: steps [t0, t1) of the time loop (model.py:183-261) as fused kernels.
 * stats_out: host [t1 - t0][ENRGY_S_COUNT] float64 or NULL. */
int enrgy_run(enrgy_ctx* ctx, int t0, int t1, double* stats_out);
/* same, asynchronous on a caller stream, statistics left in DEVICE memory d_stats (may be NULL).
 * `stream` is a cudaStream_t passed as void*. */
int enrgy_run_async(enrgy_ctx* ctx, int t0, int t1, double* d_stats, void* stream);
int enrgy_synchronize(enrgy_ctx* ctx);

/* debug views: per-step rasters of steps [t0, t1) WITHOUT advancing the state
 * (what OutputRow / calc_melt see, model.py:451-452, :245).  out: host
 * [t1 - t0][ENRGY_D_COUNT][rows][cols] float64. */
int enrgy_dump_steps(enrgy_ctx* ctx, int t0, int t1, double* out);
/* sunlit sub-steps of one step as the pre-pass derived them: out[n][8] =
 * {east, north, up, B, D, dc_fix, dr_fix, dz}; n_out receives the count (<= max_sub). */
int enrgy_get_substeps(enrgy_ctx* ctx, int step, int max_sub, double* out, int* n_out);
/* bit-packed sunlit masks of one step's sub-steps (bit = 1: lit), [n_sub][rows][ceil(cols/32)];
 * n_sub_out receives the number of sunlit sub-steps (<= max_sub). */
int enrgy_shade_masks(enrgy_ctx* ctx, int step, int max_sub, uint32_t* out, int* n_sub_out);
/* potential insolation raster of one step [kWh m-2], host [rows][cols] float64
 * (the file saga_lighting.py:7-53 would have produced; insolation_pickler.py:12-25 layout) */
int enrgy_potential_insolation(enrgy_ctx* ctx, int step, double* out);

/* ---- shading as separate steps (multi-GPU: the sweep shards by sub-step, the fused kernel by row
 * band, with an exchange of mask rows in between -- enrgy_b200/parallel.py) -------------------------
 * The sunlit sub-steps of the whole run are numbered 0 .. n-1 in row order (enrgy_get_substeps lists
 * those of one row); enrgy_sub_range gives the numbers [sub0, sub1) belonging to the rows [t0, t1).
 * A mask array of a band of `rows` rows holds enrgy_mask_words(ctx, rows) uint32 per sub-step, laid out
 * [round_up(rows, 16) / 8][pitch / 32][8]: bit (col % 32) of word [row / 8][col / 32][row % 8] = lit. */
int enrgy_sub_range(enrgy_ctx* ctx, int t0, int t1, int* sub0, int* sub1);
int64_t enrgy_mask_words(enrgy_ctx* ctx, int rows);
/* sweeps the sub-steps [sub0, sub1) over the FULL raster and writes, for every segment q, the rows
 * [seg_row0[q], seg_row0[q] + seg_rows[q]) into the DEVICE array seg_ptr[q] (which may live on a peer
 * GPU) as [sub1 - sub0] band-local masks; seg_row0 must be multiples of 8; at most 8 segments. */
int enrgy_shade_scan(enrgy_ctx* ctx, int sub0, int sub1, int n_seg, const int* seg_row0, const int* seg_rows,
                     void* const* seg_ptr, void* stream);
/* the fused kernels over the rows [t0, t1) with the caller's masks of this handle's band for exactly
 * the sub-steps of enrgy_sub_range(t0, t1); otherwise like enrgy_run_async.  d_masks may be NULL when
 * those rows have no sunlit sub-step (polar night): no mask is read then. */
int enrgy_run_masked(enrgy_ctx* ctx, int t0, int t1, const void* d_masks, double* d_stats, void* stream);
/* A run the CALLER cuts into several enrgy_run_masked / enrgy_run_async calls (chunks of rows): call with
 * on = 1 before the first and with on = 0 before the last.  The snow-melt total is then formed once, as
 * SWE(start of the run) - SWE(end), exactly as a single call over the whole range forms it, so the
 * rasters do not depend on where the run was cut (enrgy_run does the same for its own chunks). */
int enrgy_defer_snow_total(enrgy_ctx* ctx, int on);
/* device memory enrgy_run may spend on the masks of one chunk of rows (default 16 GiB; a season that
 * does not fit is processed in chunks: sweep, fused kernels, sweep, ...) */
int enrgy_set_mask_budget(enrgy_ctx* ctx, int64_t bytes);

/* state rasters (model.py:76-80, :258-261): dtype 32 -> float*, 64 -> double*; any may be NULL */
int enrgy_get_state(enrgy_ctx* ctx, int dtype, void* swe, void* total_snow, void* total_ice);
int enrgy_set_state(enrgy_ctx* ctx, int dtype, const void* swe, const void* total_snow,
                    const void* total_ice);
/* sub-surface boundary temperatures, host [msm_layers + 1][rows][cols] float64 */
int enrgy_get_layer_temps(enrgy_ctx* ctx, double* out);

/* run every subsequent operation of this handle on the caller's stream (cudaStream_t as void*;
 * NULL = back to the handle's own stream).  Lets a host framework (torch) order its collectives
 * and events with the kernels. */
int enrgy_set_stream(enrgy_ctx* ctx, void* stream);

/* device-side snapshot of the state rasters: save != 0 stores a copy, save == 0 restores it
 * (bench.py rewinds the season between timed passes without touching the host) */
int enrgy_snapshot(enrgy_ctx* ctx, int save);

/* micro-benchmarks for the roofline denominators MEASURED_PEAKS.json lacks (SURVEY 7):
 * kind 0 = FP32 FMA [TFLOP/s], 1 = FP64 FMA [TFLOP/s], 2 = MUFU.RCP [Gop/s], 3 = shared-memory
 * 4-byte loads [Gop/s]; runs ~ms on the context's device, CUDA-event timed. */
int enrgy_microbench(enrgy_ctx* ctx, int kind, double* result);

/* introspection for bench.py / tests: kernels launched so far, device time of the last run [ms] */
int64_t enrgy_launch_count(enrgy_ctx* ctx);
double enrgy_last_kernel_ms(enrgy_ctx* ctx);   /* fused kernels of the last run */
double enrgy_last_sweep_ms(enrgy_ctx* ctx);    /* shading sweeps of the last run / enrgy_shade_scan */
int enrgy_kernel_info(enrgy_ctx* ctx, int* regs, int* smem_bytes, int* ctas_per_sm, int* grid);

#ifdef __cplusplus
}
#endif
#endif /* ENRGY_B200_H */
