// Shared between the host pre-pass (prepass.cu) and the device kernels (kernels.cu):
// record layouts of the per-step / per-sub-step scalar tables and the physical constants.
//
// Reference (tepextepex/ENRGY) citations are file:line into the upstream checkout.
#pragma once
#include <cstdint>
#include <cmath>

#if defined(__CUDACC__)
#define ENRGY_HD __host__ __device__ __forceinline__
#else
#define ENRGY_HD inline
#endif

namespace enrgy {

// ---- constants (turbo.py:30-40, var_classes.py:7-15, model.py:540) ----------------------------
constexpr double kRair = 287.058;
constexpr double kKarman = 0.4;
constexpr double kGrav = 9.81;
constexpr double kCpAir = 1010.0;
constexpr double kLv = 2.514 * 1e6;
constexpr double kSigma = 5.70 * 1e-8;        // sic: the reference uses 5.70e-8 (SURVEY F11)
constexpr double kLf = 3.34 * 1e5;
constexpr double kCice = 2097.0;
constexpr double kKappaIce = 1.16 * 1e-6;
constexpr double kKappaSnow = 0.40 * 1e-6;
constexpr double kPressureLapse = -0.1145;    // hPa per m, var_classes.py:152
constexpr double kVapourScale = 6300.0;       // e = e0 * 10**(-dz/6300), var_classes.py:162
constexpr double kMsmInitLapse = -0.006;      // model.py:137

// ---- tiling -----------------------------------------------------------------------------------
constexpr int kThreads = 256;                 // block size of the set-up reductions (moments, SWE statistics)
constexpr int kWarps = kThreads / 32;
constexpr int kTileW = 128;                   // raster pitch granularity = widest tile of the fused kernel (4 warp patches of 32 columns)
constexpr int kStatsK = 8;                    // statistics reduced in the kernel (see StatK)
constexpr int kStatsM = 2;                    // + upward longwave and in-glacier flux with the sub-surface model
constexpr int kStatsP = kStatsK + kStatsM;    // columns of a per-CTA partial row
// time block = steps whose records (and sunlit sub-step records) are staged in smem together.  The
// capacities are run-time values (KernelArgs::cap_steps / cap_subs); a block always holds at least
// one whole step, so cap_subs grows to the largest sub-step count of any step (<= 255).
#ifndef ENRGY_STEPS_PER_BLOCK
#define ENRGY_STEPS_PER_BLOCK 64
#endif
constexpr int kStepsPerBlock = ENRGY_STEPS_PER_BLOCK;               // energy balance alone
constexpr int kSubsPerBlock = 256;

// Statistics the kernel reduces per step (the rest of ENRGY_S_* is derived from these by
// linearity in finalize_stats_kernel; DESIGN.md "Statistics").
enum StatK { K_RS = 0, K_LWD, K_SENS, K_LAT, K_MELT, K_SNOW, K_SWE, K_NSNOW };
// extra statistics when the sub-surface model is on (columns kStatsK + ... of a partial row)
enum StatM { M_LWU = 0, M_G };

// sub-surface model constants (msm.py:42-46, var_classes.py:7-15), per run
constexpr int kMaxLayers = 7;                 // layer thicknesses; boundaries = layers + 1
template <typename R>
struct MsmParams {
  int layers;                                 // 0 = sub-surface model off
  R d[kMaxLayers], inv_d[kMaxLayers];         // layer thicknesses [m] and their reciprocals
  R c_ice, k_ice, k_snow, rho_ice, rho_snow;  // heat capacity, diffusivities, densities
  R inv_snow_density;                         // snow depth = swe / snow_density (model.py:428, sic)
  // surface layer of a snow-free cell (snow share 0: conductivity and density are those of ice exactly)
  R g0_ice;                                   // k_ice * c_ice * rho_ice: in-glacier flux per unit temperature gradient
  R crd_ice;                                  // c_ice * rho_ice * d[0] (heat capacity of the layer per m2)
};

// ---- per-step record (24 values, staged per time block by a TMA bulk copy) ---------------------
template <typename R>
struct alignas(16) StepRec {
  R t_air;     // T_AIR at the AWS [deg C]
  R lapse;     // air-temperature lapse rate [K/m]
  R p_hpa;     // PRESSURE at the AWS [hPa]
  R e_aws;     // vapour pressure at the AWS [Pa]               var_classes.py:85
  R c_sens;    // CH * Cp * uz * sensible_corr * 100 Pa/hPa      turbo.py:156, model.py:386
  R c_lat;     // CE * uz * 0.622 * Lv * latent_corr             turbo.py:182, model.py:387
  R c_lwd;     // (0.765 + 0.22 cld^3) * sigma                   model.py:544
  R c_lwu;     // no MSM: eps*sigma*273.15^4 (the flux itself); MSM: eps*sigma   model.py:543
  R c_sw;      // 3.6e6 / dt * (SWD / potential at AWS)          model.py:483-489
  R c_melt;    // dt / Lf / 1000                                 msm.py:194-197
  R alb_w;     // whole days since map i0 / whole days between i0 and i1  interpolator.py:18
  R snow_alb;  // aged snow albedo, < 0 = off                    model.py:318-320
  R dsum;      // sum of the diffuse coefficients of the step's sub-steps (computed insolation)
  R dt;        // time step [s]
  R alb_pair;  // i0 * 256 + i1; on the device an int32 bit pattern in the low word (step_code())
  R sub;       // (first sub-step index relative to the time block) * 256 + number of sub-steps; int32 bits on the device
  // sums over the step's sunlit sub-steps of b * (u, e, n): where the sun stands above every slope of a
  // patch for the whole step, max(cos i, 0) = cos i and the direct beam is dir_u + px dir_e + py dir_n
  R dir_u, dir_e, dir_n;
  R tan2_min;  // min over the sub-steps of tan^2(sun elevation); < 0: no sunlit sub-step
  R inv_dt;    // 1 / dt (sub-surface model: the cold content of the surface layer per second)
  R c_lw0;     // float32, no MSM: c_lwd * K0^4 - lwu with K0 = float(273.15) (net longwave of a cell at K0)
  R c_lw1;     //                  c_lwd * K0^4
  R pad_;
};

// ---- per-step scalars of one ensemble member (fused members): what the roughness lengths change ----
constexpr int kMaxFusedMembers = 4;
template <typename R>
struct alignas(8) MemberRec {
  R c_sens, c_lat;
};

// ---- per-step values of one weather station (station blend, BASELINE config C4) ---------------------
constexpr int kMaxStations = 4;               // the primary AWS + 3
template <typename R>
struct alignas(16) StationRec {
  R t;     // T_AIR [deg C]
  R p;     // PRESSURE [hPa]
  R e;     // vapour pressure [Pa] = RH * e_max(T, P)           var_classes.py:85
  R cn;    // cloudiness minus the primary station's (after cloud_corr and clamping)
};

// ---- per-sub-step record (sun above the horizon only) ------------------------------------------
template <typename R>
struct alignas(16) SubRec {
  R e, n, u;   // unit vector toward the sun (east, north, up)
  R b;         // S0 * tau^(1/u) * width_h / 1000   [kWh m-2 per unit cos(incidence)]
};
// shading direction of a sub-step (precision independent: the mask spec is integers + exact float64)
struct alignas(16) ShadeRec {
  int32_t dc_fix;  // Q16 column step per ray step (east = +col)
  int32_t dr_fix;  // Q16 row step per ray step (north = -row)
  float dz;        // rise of the ray per step [m] (float32 of cell * u / max(|e|,|n|))
  int32_t kmax;    // (unused, kept for the record size)
};
// scan-line family of a direction (oracle/insolation_oracle.py:line_geometry): row type sweeps along
// the rows with u = sigma * row and the column sheared by dfix, column type the other way round
ENRGY_HD void line_geometry(int dc_fix, int dr_fix, bool* row_type, int* sigma, int* dfix) {
  const int adr = dr_fix < 0 ? -dr_fix : dr_fix, adc = dc_fix < 0 ? -dc_fix : dc_fix;
  *row_type = adr >= adc;
  if (*row_type) { *sigma = dr_fix > 0 ? 1 : -1; *dfix = dc_fix; }
  else { *sigma = dc_fix > 0 ? 1 : -1; *dfix = dr_fix; }
}
// sh(u) = round(u * dfix / 2^16).  The product is 64-bit: |dfix| <= 65536 and |u| < 2^20 (rasters up
// to 2^20 cells a side) reach 2^36; the result, at most |u|, fits an int.
ENRGY_HD int shear_q16(int u, int dfix) { return (int)(((long long)u * dfix + 32768) >> 16); }

// time block = consecutive steps whose records and sub-steps fit the smem staging buffers
struct TimeBlock {
  int32_t t_begin, t_end;      // steps [t_begin, t_end)
  int32_t sub_begin, sub_end;  // sub-step records [sub_begin, sub_end)
};

}  // namespace enrgy
