// Device-side interface of the fused energy-balance kernels (kernels.cu), used by api.cu.
#pragma once
#include <cuda_runtime.h>

#include "common.cuh"

namespace enrgy {

// insolation source of the fused kernel (template parameter)
constexpr int kInsolStreamed = 0;  // per-step kWh m-2 raster streamed from HBM
constexpr int kInsolComputed = 1;  // terrain normal . sun vector per sub-step, no shadows
constexpr int kInsolMasked = 2;    // ... times the sunlit mask of the sub-step (line sweep, shade.cu)

template <typename R>
struct KernelArgs {
  // geometry (padded device rasters; pitch is a multiple of kTileW, padding cells hold NaN)
  int rows_full, cols, pitch;     // full DEM
  int band_row0, band_rows;       // this handle's row band (rasters below are band-local)
  int rows_pad_full;              // padded row count of the full DEM buffer
  const float* dem;               // full DEM (replicated for shading), pointing at cell (0, 0) of a
                                  // buffer with a NaN apron of kDemApron cells on every side
  int dem_pitch;                  // row stride of the DEM buffer
  // sunlit masks (kInsolMasked): bit-packed, [sub-step][band_rows_pad / 8][mask_words][8] uint32 -- the 8
  // rows of a row group are adjacent, so a warp patch (32 columns x K <= 8 rows) reads one 32-byte sector
  const unsigned* masks;
  int mask_sub0;                  // global index (over all sunlit sub-steps of the run) of the first mask
  int mask_sub_last;              // ... and of the last one (prefetches are clamped to it)
  int mask_words;                 // column words per row = pitch / 32
  size_t mask_sub_stride;         // words between consecutive sub-steps
  const R* nx;                    // [band_rows_pad][pitch] terrain normal (computed insolation)
  const R* ny;
  const R* nz;
  const float* albedo;            // [n_maps][band_rows_pad][pitch]
  size_t map_stride;              // elements between consecutive albedo maps
  int albedo_const;
  R albedo_ice, albedo_snow, max_ice_albedo;
  R albedo_offset;                // ensemble member: added to the map values, clipped to [0.001, 1]
  R elev_aws;
  // state, band-local [band_rows_pad][pitch]
  R* swe;
  R* total_snow;
  R* total_ice;
  const R* swe_ref;               // SWE at the start of a run cut into several launches (null: a.swe itself)
  int update_total_snow;          // 0: an earlier launch of such a run (total_snow is added by the last one)
  // sub-surface model: boundary temperatures [layers + 1][band_rows_pad][pitch] (deg C)
  R* layer_t;
  size_t layer_stride;
  MsmParams<R> msm;
  // streamed insolation [n_steps_resident][band_rows_pad][pitch], step index relative to pot_t0
  const float* pot;
  size_t pot_stride;
  int pot_t0;
  // tables
  const StepRec<R>* steps;        // [n_steps]
  const SubRec<R>* subs;          // [n_subs]
  const TimeBlock* blocks;        // [n_blocks] covering at least [t0, t1)
  int cap_steps, cap_subs;        // capacities the time blocks were cut for (smem staging buffers)
  int block_begin, block_end;     // blocks to process
  int t0, t1;                     // steps to process (clip of the first/last block)
  // work list
  const int2* tiles;              // active tiles (tile row, tile col) of the band
  int n_tiles;
  // fused ensemble members (kernel template NM > 1; BASELINE config C5): the state rasters of member m
  // start member_stride elements after those of member m - 1, its two per-step scalars sit in
  // member_recs[t * NM + m], its albedo offset / constants below
  size_t member_stride;
  const MemberRec<R>* member_recs;
  R member_offset[kMaxFusedMembers];
  R member_albedo_ice[kMaxFusedMembers], member_albedo_snow[kMaxFusedMembers];
  // station blend (kernel template NS > 1; BASELINE config C4): station k sits at (st_row, st_col) in cell
  // units at elevation st_elev (k = 0: the primary AWS); its per-step values in station_recs[t * NS + k]
  int n_stations;
  R st_row[kMaxStations], st_col[kMaxStations], st_elev[kMaxStations];
  const StationRec<R>* station_recs;
  int cloud_on;                   // Beer-Lambert cloud attenuation of the shortwave on
  R cloud_neg_k;                  // -cloud_k
  // statistics: per-CTA partial sums [gridDim.x][t1 - t0][kStatsP] float64
  R* partials;                    // [gridDim.x][t1 - t0][kStatsK (+ kStatsM with the sub-surface model)] in R
  // dump mode: [t1 - t0][ENRGY_D_COUNT][band_rows_pad][pitch] R (may be null)
  R* dump;
  size_t dump_field_stride;
};

struct FinalizeArgs {
  const void* partials;     // [n_ctas][n_steps][row], row = kStatsK (+ kStatsM with msm); float if f32_mode else double
  int msm;                  // sub-surface model on: lwu and g are summed per cell
  int n_ctas, n_steps, t0;
  int lwd_summed;           // station blend: column K_LWD holds sum Tz^4 (else it follows from the DEM moments)
  int nm, member;           // fused members: members per row group and the member to finalize (nm <= 1: plain rows)
  double n_valid;           // valid cells of the band
  double mom[5];            // sum over the band's glacier cells of (dem - elev_aws)^k, k = 0..4
  int f32_mode;             // round the per-step constants the way the float32 kernel saw them
  const StepRec<double>* steps64;  // master copy of the per-step records (float64)
  double* stats;            // [n_steps][ENRGY_S_COUNT]
  // first-row quirk of the reference (model.py:248-252): SWE statistics of step 0 run over every
  // non-NaN cell of the INITIAL raster, including off-glacier cells
  int override_first;
  double swe0_sum, swe0_nsnow, swe0_nvalid;
};

// launch helpers (defined in kernels.cu); all asynchronous on `stream`
template <typename R>
cudaError_t launch_terrain(const float* dem, const float* terrain, int dem_pitch, int rows_full, int cols, int pitch,
                           int band_row0, int band_rows_pad, double cell, R* nx, R* ny, R* nz,
                           cudaStream_t stream);
cudaError_t launch_tile_scan(const float* dem, int pitch, int band_row0, int band_rows, int cols,
                             int tile_h, int tile_w, int tiles_r, int tiles_c, int* counts,
                             cudaStream_t stream);
cudaError_t launch_mask_check(const float* dem, int dem_pitch, const float* other, int pitch,
                              int band_row0, int band_rows, int cols,
                              unsigned long long* counters /*[2]*/, cudaStream_t stream);
template <typename R>
cudaError_t launch_moments(const float* dem, int dem_pitch, int band_row0, int band_rows, int cols, double elev,
                           double* block_out /*[blocks][5]*/, int blocks, cudaStream_t stream);
cudaError_t launch_swe0_stats(const float* swe, int pitch, int band_rows, int cols,
                              double* block_out /*[blocks][3]*/, int blocks, cudaStream_t stream);
template <typename R>
cudaError_t launch_pad_convert(const float* src_pitched, R* dst, size_t n, cudaStream_t stream);
template <typename R>
cudaError_t launch_unpad_state(const R* src, int pitch, int rows, int cols, int dtype, void* dst,
                               cudaStream_t stream);

template <typename R>
cudaError_t launch_nan_offglacier(const float* dem, int dem_pitch, int pitch, int band_row0,
                                  int band_rows, int cols, R* swe, R* tsn, R* tic, cudaStream_t stream);

struct LaunchInfo {
  int regs, smem_bytes, ctas_per_sm, grid, cells_per_thread;
};
// one instance of the fused kernel: insolation source, sub-surface model, dump mode, fused ensemble members
// (nm = 2 or 4, no sub-surface model; stats = false: no per-step statistics, a.partials unused) and blended
// weather stations (ns = kMaxStations, no fused members); 36 combinations per precision exist
struct FusedVariant {
  int insol = kInsolStreamed;
  bool msm = false, dump = false;
  int nm = 1;
  bool stats = true;
  int ns = 1;
};
// the variant's kernel attributes and its full grid (cudaErrorInvalidValue: no such instance)
template <typename R>
cudaError_t configure_energy_balance(const FusedVariant& v, int sm_count, int cap_steps, int cap_subs, LaunchInfo* info);
// grid > 0: that many CTAs, else the full grid; info (may be null) receives the launch's attributes
template <typename R>
cudaError_t launch_energy_balance(const KernelArgs<R>& a, const FusedVariant& v, int sm_count, int grid, LaunchInfo* info,
                                  cudaStream_t stream);
template <typename R>
cudaError_t launch_member_totals(const float* dem, int dem_pitch, int pitch, int band_row0, int band_rows, int cols,
                                 const R* swe, const R* tsn, const R* tic, size_t member_stride, int n_members,
                                 double* block_out /*[n_members][blocks][4]*/, int blocks, cudaStream_t stream);
template <typename R>
void energy_balance_tile(bool msm, int* tile_h, int* tile_w);
// initial boundary temperatures: min(0, t_point[l] + (dem - elev) * -0.006), model.py:133-143
template <typename R>
cudaError_t launch_msm_init(const float* dem, int dem_pitch, int pitch, int band_row0, int band_rows_pad,
                            int n_bounds, const double* t_point /*host*/, double elev, R* layer_t,
                            size_t layer_stride, cudaStream_t stream);

cudaError_t launch_finalize(const FinalizeArgs& f, cudaStream_t stream);

// ---- shading line sweep (shade.cu) ---------------------------------------------------------------
// Scan copy of the terrain: float [na + 2 * kScanRowApron][pitch_s] with -inf for NaN cells and in the
// aprons (kScanRowApron rows above and below, kScanColApron columns left and right), so the sweep
// needs no bounds checks.  The transposed copy serves the column-type sub-steps.
constexpr int kScanRowApron = 8;
constexpr int kScanColApron = 288;
inline int scan_pitch(int nb) { return (nb + 31) / 32 * 32 + 2 * kScanColApron; }
inline size_t scan_elems(int na, int nb) { return (size_t)(na + 2 * kScanRowApron) * scan_pitch(nb); }
// src: [rows][cols] device raster with row stride src_pitch (NaN = no terrain)
cudaError_t launch_scan_prepare(const float* src, int src_pitch, int rows, int cols, float* scan, float* scan_t,
                                cudaStream_t stream);

struct SweepSub {            // one sunlit sub-step to sweep
  int32_t dfix;              // Q16 step of the minor coordinate per step along the sweep axis
  int32_t sigma;             // u = sigma * (index along the sweep axis) grows toward the sun
  double dz;                 // rise of the rays per step [m] (the float32 of the ShadeRec, exactly)
  int32_t out;               // row type: index of the sub-step in the output chunk; column type: index in tmp
  int32_t out2;              // column type: index of the sub-step in the output chunk (transpose target)
};
constexpr int kMaxSweepSegs = 8;
struct SweepSeg {            // rows [row0, row0 + rows) of the raster go to a band-local mask array at ptr
  int32_t row0, rows;        // (row0 and rows multiples of 8, except the last segment's end)
  int32_t rg;                // row groups of the destination = rows_pad / 8
  int32_t words;             // column words per row of the destination
  unsigned* ptr;             // [n_sub][rg][words][8]
};
struct SweepArgs {
  const float* scan;         // cell (0, 0) of the scan copy swept along its rows (row type) ...
  const float* scan_t;       // ... and of the transposed copy (column type)
  int rows, cols;            // raster
  const SweepSub* row_subs; int n_row_subs;
  const SweepSub* col_subs; int n_col_subs;
  int n_seg;
  SweepSeg seg[kMaxSweepSegs];
  unsigned* tmp;             // column type: [n_col_subs][cols][tmp_words] (bit = row % 32 of word row / 32)
  int tmp_words;             // round_up(ceil(rows / 32), 8)
};
inline int sweep_tmp_words(int rows) { return ((rows + 31) / 32 + 7) / 8 * 8; }
// sub-steps one launch_sweep takes: the transpose runs one grid.z slice per column-type sub-step and the
// sweep one grid.y row per 4 row-type sub-steps, and CUDA caps both grid dimensions at 65535
constexpr int kSweepMaxColSubs = 65535;
constexpr int kSweepMaxRowSubs = 4 * 65535;
cudaError_t launch_sweep(const SweepArgs& a, int sm_count, cudaStream_t stream, int* n_launches);
cudaError_t launch_microbench(int kind, int sm_count, int iters, void* scratch, double* ops_per_launch,
                              cudaStream_t stream);

}  // namespace enrgy
