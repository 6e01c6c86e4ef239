// Host pre-pass (see prepass.cuh).  Host-only translation unit; compiled with -ffp-contract=off.
#include "prepass.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <limits>

namespace enrgy {

namespace {

constexpr double kDeg = 0.017453292519943295;
constexpr double kPi = 3.141592653589793;

// Beljaars & Holtslag (1991) stable / Dyer unstable integrated stability functions,
// scalar branch of turbo.py:308-361 (the model path only ever takes the scalar branch because z
// and L are scalars, SURVEY 3.2).
constexpr double kA = 0.7, kB = 0.75, kC = 5.0, kD = 0.35;

double minus_psi_m(double z, double l) {
  const double zeta = z / l;
  if (zeta >= 0) {
    return kA * zeta + kB * (zeta - kC / kD) * std::exp(-kD * zeta) + kB * kC / kD;
  }
  const double x = std::pow(1 - 16 * zeta, 0.25);
  return -(2 * std::log((1 + x) / 2) + std::log((1 + x * x) / 2) - 2 * std::atan(x) + kPi / 2);
}

double minus_psi_h(double z, double l) {
  const double zeta = z / l;
  if (zeta >= 0) {
    return std::pow(1 + 2 * kA * zeta / 3, 1.5) + kB * (zeta - kC / kD) * std::exp(-kD * zeta) +
           kB * kC / kD - 1;
  }
  const double x = std::pow(1 - 16 * zeta, 0.25);
  return -(2 * std::log((1 + x * x) / 2));
}

// turbo.py:293-305.  `k_uz` is the already formed product k*uz (its rounding differs between the
// point call, float64, and the distributed call, float32 array * weak Python float).
double friction_velocity(double k_uz, double z, bool have_l, double l, double zm) {
  double den = std::log(z / zm);
  if (have_l) den = den + minus_psi_m(z, l);
  return k_uz / den;
}

// turbo.py:199-261
double andreas_z0(double k_uz, double z, double zm, bool have_l, double l) {
  const double ustar = friction_velocity(k_uz, z, have_l, l, zm);
  const double re = ustar * zm / 1.5e-5;
  double b0, b1, b2;
  if (re <= 0.135) {
    b0 = 1.25; b1 = 0; b2 = 0;
  } else if (re <= 2.5) {
    b0 = 0.149; b1 = -0.55; b2 = 0;
  } else {
    b0 = 0.317; b1 = -0.565; b2 = -0.183;
  }
  const double ln_re = std::log(re);
  return zm * std::exp(b0 + b1 * ln_re + b2 * (ln_re * ln_re));
}

}  // namespace

double sat_vapour_pressure(double t_kelvin, double p_pa) {
  const double t = t_kelvin - 273.15;
  const double p = p_pa / 100;
  const double ew = 611.2 * std::exp((17.62 * t) / (243.12 + t));
  const double fp = 1.0016 + 3.15 * 1e-6 * p - 0.074 / p;
  return fp * ew;
}

// turbo.py:264-290 with zh already resolved (constant or Andreas).
double exchange_coefficient(double z, bool have_l, double l, double zm, double zh) {
  const double num = kKarman * kKarman;
  double den;
  if (have_l) {
    const double pm = minus_psi_m(z, l);
    const double ph = minus_psi_h(z, l);
    den = (std::log(z / zm) + pm * (z / l)) * (std::log(z / zh) + ph * (z / l));
  } else {
    den = std::log(z / zm) * std::log(z / zh);
  }
  return num / den;
}

// turbo.py:88-137: neutral first guess, then exactly five updates of (u*, Qh, L).
void point_turbulence(double z, double uz, double tz, double p, double ts, bool ts_f32, double zm,
                      double zh_const, bool andreas, double* qh_out, double* l_out) {
  // (Tz - Ts): Python float minus np.float32 scalar is a float32 operation under NEP 50 when the
  // surface temperature was sampled from a float32 raster (as shipped), model.py:347-350.
  double d_t;
  if (ts_f32) {
    d_t = (double)((float)tz - (float)ts);
  } else {
    d_t = tz - ts;
  }
  const double rho = p / (kRair * tz);
  const double k_uz = kKarman * uz;
  bool have_l = false;
  double l = 0.0, qh = 0.0;
  for (int it = 0; it < 6; ++it) {
    const double ustar = friction_velocity(k_uz, z, have_l, l, zm);
    const double zh = andreas ? andreas_z0(k_uz, z, zm, have_l, l) : zh_const;
    const double ch = exchange_coefficient(z, have_l, l, zm, zh);
    qh = ch * kCpAir * rho * uz * d_t;
    const double num = rho * kCpAir * std::pow(ustar, 3.0) * tz;
    const double den = kKarman * kGrav * qh;
    l = num / den;
    have_l = true;
  }
  *qh_out = qh;
  *l_out = l;
}

void sun_vector(double t_unix, double lat_deg, double lon_deg, double* e, double* n, double* u) {
  // low-precision almanac ephemeris; the same expression order as oracle/insolation_oracle.py
  const double d = t_unix / 86400.0 + 2440587.5 - 2451545.0;
  const double mean_lon = std::fmod(280.460 + 0.9856474 * d, 360.0);
  const double g = std::fmod(357.528 + 0.9856003 * d, 360.0) * kDeg;
  const double lam = (mean_lon + 1.915 * std::sin(g) + 0.020 * std::sin(2.0 * g)) * kDeg;
  const double eps = (23.439 - 0.0000004 * d) * kDeg;
  const double ra = std::atan2(std::cos(eps) * std::sin(lam), std::cos(lam));
  const double dec = std::asin(std::sin(eps) * std::sin(lam));
  const double gmst = std::fmod(280.46061837 + 360.98564736629 * d, 360.0);
  const double ha = (gmst + lon_deg) * kDeg - ra;
  const double phi = lat_deg * kDeg;
  const double sd = std::sin(dec), cd = std::cos(dec);
  const double sp = std::sin(phi), cp = std::cos(phi);
  const double sh = std::sin(ha), ch = std::cos(ha);
  *u = sp * sd + cp * cd * ch;
  *e = -cd * sh;
  *n = sd * cp - cd * sp * ch;
}

namespace {

inline bool valid(float z) { return z == z; }

// terrain normal of the AWS cell on the host (double), same rule as terrain_kernel; nb = 3 x 3
// neighbourhood of the cell, NaN outside the grid
void host_normal(const float* nb, double cell, double* nx, double* ny, double* nz) {
  const double z = nb[4];
  auto one_sided = [&](float a, float b) -> double {
    if (valid(a)) return (double)a - z;
    if (valid(b)) return z - (double)b;
    return 0.0;
  };
  const float zn = nb[1], zs = nb[7], ze = nb[5], zw = nb[3];
  const double gy = (one_sided(zn, zs) - one_sided(zs, zn)) / (2.0 * cell);
  const double gx = (one_sided(ze, zw) - one_sided(zw, ze)) / (2.0 * cell);
  const double inv = 1.0 / std::sqrt(1.0 + gx * gx + gy * gy);
  *nx = -gx * inv;
  *ny = -gy * inv;
  *nz = inv;
}

// the shading specification for ONE cell on the host: the ray of the cell marched along its scan line
// (oracle/insolation_oracle.py:trace_cells; the device sweeps whole lines, shade.cu)
bool host_lit(const float* dem, int rows, int cols, int r, int c, const ShadeRec& s) {
  if (!std::isfinite(s.dz) || (s.dc_fix == 0 && s.dr_fix == 0)) return true;
  bool row_type; int sigma, dfix;
  line_geometry(s.dc_fix, s.dr_fix, &row_type, &sigma, &dfix);
  const double dz = (double)s.dz;
  const int u0 = sigma * (row_type ? r : c);
  const int line = (row_type ? c : r) - shear_q16(u0, dfix);
  const double g0 = (double)dem[(size_t)r * cols + c] - (double)u0 * dz;
  for (int k = 1;; ++k) {
    const int u = u0 + k;
    const int major = sigma * u, minor = line + shear_q16(u, dfix);
    const int rr = row_type ? major : minor, cc = row_type ? minor : major;
    if (rr < 0 || rr >= rows || cc < 0 || cc >= cols) return true;
    const float smp = dem[(size_t)rr * cols + cc];
    if (smp == smp && (double)smp - (double)u * dz > g0) return false;
  }
}

}  // namespace

int run_prepass(const PrepassInput& in, PrepassOutput& out, std::string& err) {
  const enrgy_params& p = in.p;
  const int T = in.n_steps;
  const bool mirror32 = in.precision == ENRGY_F32;
  const bool computed = p.insol_mode == ENRGY_INSOL_COMPUTED;
  out.steps.assign(T, StepRec<double>{});
  out.subs.clear();
  out.sub_first.assign(T, 0);
  out.sub_count.assign(T, 0);
  out.blocks.clear();
  out.point.assign((size_t)T * ENRGY_P_COUNT, 0.0);
  out.point_layers.assign(p.msm_layers > 0 ? (size_t)T * (kMaxLayers + 1) : 0, 0.0);

  if (p.aws_row < 0 || p.aws_row >= in.rows || p.aws_col < 0 || p.aws_col >= in.cols) {
    err = "AWS cell outside the raster";
    return ENRGY_ERR_ARG;
  }
  double nx = 0, ny = 0, nz = 1;
  if (computed) host_normal(in.nbhd, p.cell_size, &nx, &ny, &nz);
  if (computed && p.shadow && in.dem == nullptr) {
    err = "the host DEM copy is missing for the AWS-cell shading ray";
    return ENRGY_ERR_ARG;
  }

  const double zm = p.zm;
  const double zh_const = p.z_h_or_e;
  // sub-surface model: the AWS cell is integrated serially here because its surface temperature
  // feeds the Monin-Obukhov solve of the NEXT row (model.py:347-358)
  const bool msm = p.msm_layers > 0;
  const int nl = p.msm_layers;
  const float z_aws = in.nbhd[4];
  if (!(z_aws == z_aws)) {
    err = "the AWS cell is off-glacier (NaN in the DEM)";
    return ENRGY_ERR_ARG;
  }
  std::vector<double> tl(in.layer_t_aws);
  if (msm && (int)tl.size() != nl + 1) {
    err = "enrgy_set_msm must precede enrgy_prepass when msm_layers > 0";
    return ENRGY_ERR_ARG;
  }
  double swe_cell = in.swe_aws;
  const double delta_cell = (double)z_aws - p.elev_aws;
  const double pw_cell = std::pow(10.0, -delta_cell / kVapourScale);
  // Station blend with the sub-surface model: the AWS cell's integration must see the blended meteorology
  // of that cell, as every other cell does (oracle/enrgy_oracle.py "several weather stations"; station 0 is
  // the primary AWS at the cell itself).  w: the cell's weights, v: the weights folded with the
  // vapour-pressure reduction, d_blend: sum_k w_k (z - z_k).
  const bool station_blend = msm && in.n_extra > 0;
  const int n_st = 1 + in.n_extra;
  double st_w[kMaxStations] = {}, st_v[kMaxStations] = {}, d_blend = 0.0;
  if (station_blend) {
    double q[kMaxStations], tot = 0.0;
    for (int k = 0; k < n_st; ++k) {
      const double dr = k ? (double)p.aws_row - in.st_row[k] : 0.0, dc = k ? (double)p.aws_col - in.st_col[k] : 0.0;
      q[k] = 1.0 / (dr * dr + dc * dc + 0.25);
      tot = k ? tot + q[k] : q[k];
    }
    for (int k = 0; k < n_st; ++k) {
      const double dz = (double)z_aws - (k ? in.st_elev[k] : p.elev_aws);
      st_w[k] = q[k] / tot;
      d_blend = k ? d_blend + st_w[k] * dz : st_w[k] * dz;
      st_v[k] = st_w[k] * std::pow(10.0, -dz / kVapourScale);
    }
  }

  for (int i = 0; i < T; ++i) {
    const double* f = in.forcing + (size_t)i * ENRGY_F_COUNT;
    StepRec<double>& s = out.steps[i];
    double* pt = &out.point[(size_t)i * ENRGY_P_COUNT];
    const double dt = f[ENRGY_F_DT];
    if (!(dt > 0)) {
      err = "time step <= 0 (a one-row AWS file divides by zero in the reference too, helpers.py:67-70)";
      return ENRGY_ERR_RANGE;
    }
    // AwsVars.__post_init__, var_classes.py:80-85
    double wind = f[ENRGY_F_WIND];
    if (wind == 0) wind = 0.1;
    const double t_air = f[ENRGY_F_T_AIR];
    const double tz = t_air + 273.15;
    const double p_hpa = f[ENRGY_F_PRESSURE];
    const double p_pa = p_hpa * 100;
    const double rh = f[ENRGY_F_RH];
    const double e_aws = rh * sat_vapour_pressure(tz, p_pa);

    // point solve for L, model.py:347-358
    const double ts_aws_c = msm ? tl[0] : 0.0;     // no MSM: layer_temperatures[0] is all zeros (F9)
    double ts_k;
    if (mirror32) {
      ts_k = (double)((float)ts_aws_c + 273.15f);
    } else {
      ts_k = ts_aws_c + 273.15;
    }
    double qh, l;
    point_turbulence(p.sensor_z, wind, tz, p_pa, ts_k, mirror32, zm, zh_const, p.andreas != 0, &qh, &l);

    // distributed exchange coefficient, model.py:372-381 -> turbo.py:154,180.  The wind raster
    // is float32 (var_classes.py:170); with Andreas its product with k is a float32 product.
    const float wind32 = (float)wind;
    double zh = zh_const;
    if (p.andreas) {
      const double k_uz32 = (double)(0.4f * wind32);
      zh = andreas_z0(k_uz32, p.sensor_z, zm, true, l);
    }
    const double ch = exchange_coefficient(p.sensor_z, true, l, zm, zh);
    const double uz = (double)wind32;

    s.t_air = t_air;
    s.lapse = f[ENRGY_F_LAPSE];
    s.p_hpa = p_hpa;
    s.e_aws = e_aws;
    s.c_sens = ch * kCpAir * uz * p.sensible_corr * 100;   // x100: the kernel multiplies by hPa
    s.c_lat = ch * uz * 0.622 * kLv * p.latent_corr;
    const double cld = f[ENRGY_F_CLOUD];
    s.c_lwd = (0.765 + 0.22 * std::pow(cld, 3.0)) * kSigma;
    if (p.msm_layers > 0) {
      s.c_lwu = p.emissivity * kSigma;
    } else {
      s.c_lwu = p.emissivity * kSigma * std::pow(ts_k, 4.0);
    }
    {
      const double k0 = (double)273.15f, k04 = (k0 * k0) * (k0 * k0);
      // (float32 kernel: its c_lwd is the float32 of the value above)
      const double c_lwd_k = mirror32 ? (double)(float)s.c_lwd : s.c_lwd;
      s.c_lw1 = c_lwd_k * k04;
      s.c_lw0 = s.c_lw1 - (mirror32 ? (double)(float)s.c_lwu : s.c_lwu);
    }
    s.c_melt = dt / kLf / 1000;
    s.dt = dt;
    s.inv_dt = 1.0 / dt;

    // albedo schedule, interpolator.py:5-20 and model.py:311-320
    const int i0 = (int)f[ENRGY_F_ALB_I0], i1 = (int)f[ENRGY_F_ALB_I1];
    const double span = f[ENRGY_F_ALB_SPAN];
    s.alb_pair = (double)(i0 * 256 + i1);
    s.alb_w = span > 0 ? f[ENRGY_F_ALB_DAYS] / span : 0.0;
    const double snow_days = f[ENRGY_F_SNOW_DAYS];
    s.snow_alb = snow_days > 0 ? 0.40 + 0.44 * std::exp(-0.12 * snow_days) : -1.0;
    if (p.albedo_const) {             // model.py:329-332: where(swe > 0, snow, ice)
      s.snow_alb = p.albedo_snow;
      s.alb_w = 0.0;
      s.alb_pair = 0.0;
    }

    // insolation sub-steps, saga_lighting.py:24-44
    double pot_aws_kwh = 0.0;
    out.sub_first[i] = (int)out.subs.size();
    if (computed) {
      const double dt_h = dt / 3600.0;
      const double hs = p.hour_step;
      int n_sub = (int)std::ceil(dt_h / hs - 1e-9);
      if (n_sub < 1) n_sub = 1;
      double direct = 0.0, dsum = 0.0;
      double dir_u = 0.0, dir_e = 0.0, dir_n = 0.0, tan2_min = std::numeric_limits<double>::infinity();
      for (int j = 0; j < n_sub; ++j) {
        const double w = std::min(hs, dt_h - j * hs);
        const double t_mid = f[ENRGY_F_TIME] + (j * hs + 0.5 * w) * 3600.0;
        SubHost sb;
        sun_vector(t_mid, p.lat_deg, p.lon_deg, &sb.e, &sb.n, &sb.u);
        if (!(sb.u > 0.0)) continue;
        const double tb = std::pow(p.transmittance, 1.0 / sb.u);
        sb.b = p.solar_const * tb * w / 1000.0;
        sb.d = p.solar_const * (0.271 - 0.294 * tb) * sb.u * w / 1000.0 * 0.5;
        const double m = std::max(std::fabs(sb.e), std::fabs(sb.n));
        if (m > 0.0) {
          sb.shade.dc_fix = (int32_t)std::floor(sb.e / m * 65536.0 + 0.5);
          sb.shade.dr_fix = (int32_t)std::floor(-sb.n / m * 65536.0 + 0.5);
          sb.shade.dz = (float)(p.cell_size * sb.u / m);
        } else {
          sb.shade.dc_fix = 0;
          sb.shade.dr_fix = 0;
          sb.shade.dz = std::numeric_limits<float>::infinity();
        }
        sb.shade.kmax = std::max(in.rows, in.cols);
        out.subs.push_back(sb);
        dir_u += sb.b * sb.u; dir_e += sb.b * sb.e; dir_n += sb.b * sb.n;
        {
          const double h2 = sb.e * sb.e + sb.n * sb.n;
          if (h2 > 0.0) tan2_min = std::min(tan2_min, sb.u * sb.u / h2);
        }
        const double cosi = nx * sb.e + ny * sb.n + nz * sb.u;
        double term = sb.b * std::max(cosi, 0.0);
        if (p.shadow && !host_lit(in.dem, in.rows, in.cols, p.aws_row, p.aws_col, sb.shade)) {
          term = 0.0;
        }
        direct = direct + term;
        dsum = dsum + sb.d;
      }
      s.dsum = dsum;
      s.dir_u = dir_u; s.dir_e = dir_e; s.dir_n = dir_n;
      // no sunlit sub-step: never; all at the zenith: the (huge) finite maximum, not inf
      s.tan2_min = (int)out.subs.size() == out.sub_first[i] ? -1.0 : std::min(tan2_min, 1e30);
      pot_aws_kwh = direct + dsum * (1.0 + nz);
    } else {
      s.dsum = 0.0;
      s.dir_u = s.dir_e = s.dir_n = 0.0; s.tan2_min = -1.0;
      pot_aws_kwh = in.pot_aws ? in.pot_aws[i] : 0.0;
    }
    out.sub_count[i] = (int)out.subs.size() - out.sub_first[i];
    if (out.sub_count[i] > 255) {
      err = "more than 255 insolation sub-steps in one time step";
      return ENRGY_ERR_RANGE;
    }

    // kWh -> W and the observed/potential factor, helpers.py:27-60, model.py:512-526
    double pot_w, factor;
    const double swd = f[ENRGY_F_SWD];
    if (mirror32 && !computed) {
      const float pw32 = (((float)pot_aws_kwh * 3.6f) * 1000000.0f) / (float)dt;
      pot_w = (double)pw32;
      factor = pw32 == 0.0f ? 1.0 : (double)((float)swd / pw32);
    } else {
      pot_w = pot_aws_kwh * 3.6 * 1000000 / dt;
      factor = pot_w == 0 ? 1.0 : swd / pot_w;
    }
    s.c_sw = 3.6 * 1000000 / dt * factor;

    // meteorology of the distributed pass at the AWS cell: the AWS values reduced to the cell's elevation,
    // or their blend with the extra stations (above)
    double t_air_c = t_air + delta_cell * f[ENRGY_F_LAPSE];
    double p_c = p_hpa + delta_cell * kPressureLapse;
    double e_c = e_aws * pw_cell;
    double cloud_fac = 1.0;                        // Beer-Lambert factor of the shortwave
    if (station_blend) {
      const double n0 = f[ENRGY_F_CLOUD];
      double mix_t = st_w[0] * t_air, mix_p = st_w[0] * p_hpa, mix_n = 0.0;
      e_c = e_aws * st_v[0];
      for (int k = 1; k < n_st; ++k) {
        const double* v = in.st_series + ((size_t)(k - 1) * T + i) * ENRGY_ST_COUNT;
        const double tk = v[ENRGY_ST_T_AIR], pk = v[ENRGY_ST_PRESSURE];
        mix_t = mix_t + st_w[k] * tk;
        mix_p = mix_p + st_w[k] * pk;
        e_c = e_c + v[ENRGY_ST_RH] * sat_vapour_pressure(tk + 273.15, pk * 100) * st_v[k];
        mix_n = mix_n + st_w[k] * (v[ENRGY_ST_CLOUD] - n0);
      }
      t_air_c = mix_t + d_blend * f[ENRGY_F_LAPSE];
      p_c = mix_p + d_blend * kPressureLapse;
      if (!std::isnan(in.cloud_k)) cloud_fac = std::exp(-in.cloud_k * mix_n);
    }
    // turbulent fluxes of the distributed pass at the AWS cell itself (debug_point_output, model.py:441-448)
    const double tz_c = t_air_c + 273.15;
    const double tsk = ts_aws_c + 273.15;
    const double r_rt = 1.0 / (kRair * tz_c);
    const double sens = (s.c_sens * p_c) * (r_rt * (tz_c - tsk));
    const double f_p = 1.0016 + 3.15 * 1e-6 * p_c - 0.074 / p_c;
    const double es = 611.2 * std::exp((17.62 * ts_aws_c) / (243.12 + ts_aws_c)) * f_p;
    const double lat = (s.c_lat * r_rt) * (e_c - es);
    pt[ENRGY_P_SENS_AWS] = sens;
    pt[ENRGY_P_LAT_AWS] = lat;
    if (msm) {
      // the AWS cell's own energy balance and conduction step (same arithmetic as the kernel)
      for (int lyr = 0; lyr <= nl; ++lyr) out.point_layers[(size_t)i * (kMaxLayers + 1) + lyr] = tl[lyr];
      const double lwd = s.c_lwd * (tz_c * tz_c) * (tz_c * tz_c);
      const double lwu = s.c_lwu * (tsk * tsk) * (tsk * tsk);
      double alb;
      const bool has_snow = swe_cell > 0;
      if (p.albedo_const) {
        alb = has_snow ? p.albedo_snow : p.albedo_ice;
      } else {
        auto member = [&](double a) { return std::min(std::max((double)(float)(a) + in.albedo_offset, (double)0.001f), 1.0); };
        const double x0 = in.alb_aws.empty() ? 0.5 : member(in.alb_aws[i0]);
        const double x1 = in.alb_aws.empty() ? 0.5 : member(in.alb_aws[i1]);
        const double blend = x0 + s.alb_w * (x1 - x0);
        alb = has_snow ? (s.snow_alb >= 0 ? s.snow_alb : blend) : std::min(blend, p.max_ice_albedo);
      }
      const double rs = pot_aws_kwh * s.c_sw * cloud_fac * (1.0 - alb);
      const double atmo = rs + lwd - lwu + sens + lat;
      double sd = swe_cell / p.snow_density;
      double grad_prev = 0.0, mf = 0.0;
      std::vector<double> tn(tl);
      for (int lyr = 0; lyr < nl; ++lyr) {
        const double d = p.msm_depths[lyr];
        const double grad = (tl[lyr + 1] - tl[lyr]) / d;
        const double ratio = sd > d ? 1.0 : sd / d;
        const double kap = ratio * kKappaSnow + (1 - ratio) * kKappaIce;
        const double rho = ratio * p.snow_density + (1 - ratio) * p.ice_density;
        sd = std::max(sd - d, 0.0);
        double dlt;
        if (lyr == 0) {
          const double gfl = kap * grad * kCice * rho;
          const double full = atmo + gfl;
          const double crd = kCice * rho * d;
          const double q0 = -tl[0] * crd / dt;
          mf = std::max(full - q0, 0.0);
          dlt = (full - mf) / crd;
        } else {
          dlt = kap * (grad - grad_prev) / d;
        }
        grad_prev = grad;
        tn[lyr] = tl[lyr] + dlt * dt;
      }
      tl = tn;
      const double we = mf * s.c_melt;
      swe_cell -= std::min(we, swe_cell);
    }

    pt[ENRGY_P_L] = l;
    pt[ENRGY_P_CH] = ch;
    pt[ENRGY_P_POT_AWS] = pot_w;
    pt[ENRGY_P_SW_FACTOR] = factor;
    pt[ENRGY_P_TSURF_AWS] = mirror32 ? (double)((float)ts_k - 273.15f) : ts_k - 273.15;
    pt[ENRGY_P_QH_AWS] = qh;
    pt[ENRGY_P_NSUB] = out.sub_count[i];
  }

  // time blocks: as many consecutive steps as fit the smem staging buffers
  out.cap_steps = std::max(in.cap_steps, 1);
  out.cap_subs = std::max(in.cap_subs, 1);
  for (int i = 0; i < T; ++i) out.cap_subs = std::max(out.cap_subs, out.sub_count[i]);
  int t = 0;
  while (t < T) {
    TimeBlock b;
    b.t_begin = t;
    b.sub_begin = out.sub_first[t];
    int n_sub = 0;
    int e = t;
    while (e < T && e - t < out.cap_steps && n_sub + out.sub_count[e] <= out.cap_subs) {
      n_sub += out.sub_count[e];
      ++e;
    }
    b.t_end = e;
    b.sub_end = b.sub_begin + n_sub;
    out.blocks.push_back(b);
    t = e;
  }
  // sub-step index of each step relative to its time block
  for (const TimeBlock& b : out.blocks) {
    for (int i = b.t_begin; i < b.t_end; ++i) {
      out.steps[i].sub = (double)((out.sub_first[i] - b.sub_begin) * 256 + out.sub_count[i]);
    }
  }
  return ENRGY_OK;
}

}  // namespace enrgy
