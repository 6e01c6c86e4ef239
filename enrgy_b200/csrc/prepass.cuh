// Host pre-pass: everything `Energy.model` derives ONCE PER AWS ROW (not per cell) before the
// rasters are touched -- the per-step scalars the fused kernel consumes.
//
//   reference model.py:186-230   row parsing, AwsVars (var_classes.py:80-85)
//   reference model.py:347-358   point Monin-Obukhov solve at the AWS cell (turbo.py:88-137)
//   reference turbo.py:264-290   CH = CE of the distributed pass (scalar because z, L are scalars)
//   reference model.py:500-530   observed / potential shortwave scaling factor
//   reference saga_lighting.py:24-44  sub-step schedule and sun position of the insolation tool
//
// float64 throughout, libm transcendental functions, no FMA contraction (-ffp-contract=off), the
// reference's expression order: with the same libm this reproduces the reference's scalars to the
// last bit or two, far inside the 1e-9 parity bar.
#pragma once
#include <string>
#include <vector>

#include "../../include/enrgy_b200.h"
#include "common.cuh"

namespace enrgy {

struct SubHost {
  double e, n, u, b, d;
  ShadeRec shade;
};

struct PrepassInput {
  enrgy_params p;          // defaults already resolved (no NaNs left)
  int precision;           // ENRGY_F32 mirrors the as-shipped float32 point operations
  double albedo_offset = 0.0;   // ensemble member (enrgy_set_member); p.albedo_ice/snow are already shifted
  int rows, cols;          // full raster
  const float* dem;        // full host DEM [rows][cols]; only needed (non-null) for the shading ray of the AWS cell
  float nbhd[9];           // DEM at the AWS cell and its 8 neighbours (row-major 3 x 3, NaN outside the grid)
  int cap_steps = kStepsPerBlock;   // time-block capacities (smem staging buffers of the kernel)
  int cap_subs = kSubsPerBlock;     // ... grown to the largest sub-step count of a single step
  int n_steps;
  const double* forcing;   // [n_steps][ENRGY_F_COUNT]
  const double* pot_aws;   // streamed mode: potential insolation at the AWS cell per step [kWh m-2]
  // state of the AWS cell for the serial sub-surface integration (MSM): albedo maps at the cell,
  // SWE and boundary temperatures at step 0 (the pre-pass always integrates from the first row)
  std::vector<double> alb_aws;
  double swe_aws = 0.0;
  std::vector<double> layer_t_aws;
  // station blend (enrgy_set_stations): extra station k = 1 .. n_extra at (st_row, st_col) of the full raster
  // in cell units, elevation st_elev, series [n_extra][n_steps][ENRGY_ST_COUNT]; with the sub-surface model
  // the AWS cell is integrated in the blended meteorology of that cell
  int n_extra = 0;
  double st_row[kMaxStations] = {}, st_col[kMaxStations] = {}, st_elev[kMaxStations] = {};
  const double* st_series = nullptr;
  double cloud_k = NAN;    // NaN: no cloud attenuation
};

struct PrepassOutput {
  std::vector<StepRec<double>> steps;
  std::vector<SubHost> subs;              // sunlit sub-steps of all steps, in order
  std::vector<int> sub_first, sub_count;  // per step: range into subs
  std::vector<TimeBlock> blocks;
  int cap_steps = 0, cap_subs = 0;        // capacities the blocks were cut for
  std::vector<double> point;              // [n_steps][ENRGY_P_COUNT]
  std::vector<double> point_layers;       // MSM: [n_steps][kMaxLayers + 1] boundary temperatures of the AWS cell BEFORE each row's update
};

// Returns 0 or an ENRGY_ERR_* code with a message in err.
int run_prepass(const PrepassInput& in, PrepassOutput& out, std::string& err);

// exposed for the per-cell kernels' host twin and for tests
void sun_vector(double t_unix, double lat_deg, double lon_deg, double* e, double* n, double* u);
double sat_vapour_pressure(double t_kelvin, double p_pa);                    // turbo.py:368-379
double exchange_coefficient(double z, bool have_l, double l, double zm, double zh);
void point_turbulence(double z, double uz, double tz, double p, double ts, bool ts_f32, double zm,
                      double zh, bool andreas, double* qh, double* l_out);

}  // namespace enrgy
