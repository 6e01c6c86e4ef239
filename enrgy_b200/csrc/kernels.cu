// Fused surface-energy-balance kernels for sm_100a (B200).
//
// One persistent CTA per resident slot walks a static list of raster tiles.  For each tile every
// thread owns K cells, as K/2 packed pairs (sm_100 f32x2: FFMA2/FADD2/FMUL2), for the WHOLE time
// range: SWE and the ice-melt total live in registers, the per-step AWS scalars are staged per time
// block in shared memory by TMA bulk copies (cp.async.bulk + mbarrier, double buffered), and the only
// global traffic inside the time loop is the daily refresh of the albedo blend, the optional
// streamed insolation raster (4 B per cell-step) and the sunlit masks of the shading sweep (1 bit).
//
// Reference arithmetic being replaced (tepextepex/ENRGY, file:line) -> where it lives here:
//   var_classes.py:113-125  lapse-rate distribution of T, p, e            -> balance() in the step loop
//   turbo.py:140-196        distributed sensible / latent flux            -> balance()
//   turbo.py:368-379        Magnus saturation vapour pressure             -> balance(): surface vapour term
//   model.py:533-545        longwave                                      -> balance(), finalize_stats_kernel
//   model.py:298-337        albedo                                        -> daily blend + balance()
//   model.py:464-497        shortwave from potential insolation           -> balance()
//   saga_lighting.py:42-44  potential insolation incl. shadows (SAGA)     -> sub_step(); sunlit masks from shade.cu
//   model.py:411, :434-438  flux sum and clamp                            -> balance()
//   msm.py:193-203          melt partition                                -> balance()
//   msm.py:31-107           sub-surface conduction (MSM variants)         -> balance()
//   model.py:258-261        state update                                  -> balance(), epilogue
//   var_classes.py:45-56, model.py:246-252  per-step area statistics      -> batch_put / batch_reduce + slots + finalize
#include "kernels.cuh"

#include <cstdio>
#include <cstring>
#include <type_traits>

#include "../../include/enrgy_b200.h"

namespace enrgy {

// =================================================================================================
// small device helpers
// =================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// TMA 1-D bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, unsigned bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// arithmetic traits ------------------------------------------------------------------------------
template <typename R>
struct Num;
template <>
struct Num<float> {
  static __device__ __forceinline__ float rcp(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
  }
  // T + delta * lapse exactly as NumPy float32 evaluates it (rounded product, rounded sum)
  static __device__ __forceinline__ float lapse(float t, float delta, float g) {
    return __fadd_rn(t, __fmul_rn(delta, g));
  }
  static __device__ __forceinline__ float pow10(float x) { return powf(10.0f, x); }
  static __device__ __forceinline__ float exp_(float x) { return expf(x); }
  static __device__ __forceinline__ float rsqrt_(float x) { return 1.0f / sqrtf(x); }
};
template <>
struct Num<double> {
#ifndef ENRGY_F64_FAST_RCP
#define ENRGY_F64_FAST_RCP 1
#endif
  // 1 / x for a normal, finite x far from the exponent limits (products of pressures and temperatures):
  // MUFU.RCP64H seed (20 bits) and two Newton steps, without the IEEE division's slow-path test and
  // fix-up (~1 ulp instead of correctly rounded; the float64 bar is 1e-9)
  static __device__ __forceinline__ double rcp(double x) {
#if ENRGY_F64_FAST_RCP
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
#else
    return 1.0 / x;
#endif
  }
  static __device__ __forceinline__ double lapse(double t, double delta, double g) {
    return t + delta * g;
  }
  static __device__ __forceinline__ double pow10(double x) { return pow(10.0, x); }
  static __device__ __forceinline__ double exp_(double x) { return exp(x); }
  static __device__ __forceinline__ double rsqrt_(double x) { return 1.0 / sqrt(x); }
};

// integer code carried in the low word of a step-record slot (upload_tables)
__device__ __forceinline__ int step_code(const float& x) { return __float_as_int(x); }
__device__ __forceinline__ int step_code(const double& x) { return __double2loint(x); }

// value barrier: the compiler may neither rematerialise x from its inputs nor see through it
__device__ __forceinline__ void keep_in_register(float& x) { asm volatile("" : "+f"(x)); }
__device__ __forceinline__ void keep_in_register(double& x) { asm volatile("" : "+d"(x)); }
__device__ __forceinline__ void keep_in_register(unsigned& x) { asm volatile("" : "+r"(x)); }
template <typename R>
struct V2;

// ---- packed pairs of cells --------------------------------------------------------------------
// sm_100 executes fma/add/mul.f32x2 (SASS FFMA2 / FADD2 / FMUL2) on an aligned register pair: two
// cells per issue slot.  The FP32 pipe takes two cycles for a packed instruction, so the FLOP peak is
// unchanged, but the freed issue slots carry the min/max/select/MUFU work of the other pipes
// (measured on B200, scratch/ffma2_bench.cu: 16 FMA + 8 FMNMX per round take 24.7 clk scalar, 19 clk
// packed).  V2<double> is the same interface over two plain doubles.
template <typename R>
struct V2;
template <>
struct V2<float> {
  unsigned long long v;
  static __device__ __forceinline__ V2 make(float lo, float hi) {
    V2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
    return r;
  }
  static __device__ __forceinline__ V2 splat(float x) { return make(x, x); }
  __device__ __forceinline__ float lo() const { return __uint_as_float((unsigned)(v & 0xffffffffull)); }
  __device__ __forceinline__ float hi() const { return __uint_as_float((unsigned)(v >> 32)); }
};
template <>
struct V2<double> {
  double a, b;
  static __device__ __forceinline__ V2 make(double lo, double hi) { return V2{lo, hi}; }
  static __device__ __forceinline__ V2 splat(double x) { return V2{x, x}; }
  __device__ __forceinline__ double lo() const { return a; }
  __device__ __forceinline__ double hi() const { return b; }
};
__device__ __forceinline__ V2<float> fma2(V2<float> a, V2<float> b, V2<float> c) {
  V2<float> d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d.v) : "l"(a.v), "l"(b.v), "l"(c.v));
  return d;
}
__device__ __forceinline__ V2<float> add2(V2<float> a, V2<float> b) {
  V2<float> d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d.v) : "l"(a.v), "l"(b.v));
  return d;
}
__device__ __forceinline__ V2<float> sub2(V2<float> a, V2<float> b) {
  V2<float> d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d.v) : "l"(a.v), "l"(b.v));
  return d;
}
__device__ __forceinline__ V2<float> mul2(V2<float> a, V2<float> b) {
  V2<float> d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d.v) : "l"(a.v), "l"(b.v));
  return d;
}
__device__ __forceinline__ V2<double> fma2(V2<double> a, V2<double> b, V2<double> c) {
  return V2<double>{a.a * b.a + c.a, a.b * b.b + c.b};
}
__device__ __forceinline__ V2<double> add2(V2<double> a, V2<double> b) { return V2<double>{a.a + b.a, a.b + b.b}; }
__device__ __forceinline__ V2<double> sub2(V2<double> a, V2<double> b) { return V2<double>{a.a - b.a, a.b - b.b}; }
__device__ __forceinline__ V2<double> mul2(V2<double> a, V2<double> b) { return V2<double>{a.a * b.a, a.b * b.b}; }
// delta * lapse rounded to float32 before it is added (NumPy float32 semantics), never contracted
__device__ __forceinline__ V2<float> lapse_product(V2<float> d, float g) {
  return V2<float>::make(__fmul_rn(d.lo(), g), __fmul_rn(d.hi(), g));
}
__device__ __forceinline__ V2<double> lapse_product(V2<double> d, double g) { return V2<double>{d.a * g, d.b * g}; }
__device__ __forceinline__ void keep_in_register(V2<float>& x) { asm volatile("" : "+l"(x.v)); }
__device__ __forceinline__ void keep_in_register(V2<double>&) {}   // (float64 is short of registers: it may rematerialise)

// single IEEE operations (no contraction): the station weights follow NumPy's array arithmetic
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }
// x^2 + y^2 with fixed roundings (no contraction: the same value wherever it is formed)
__device__ __forceinline__ float sq_sum(float x, float y) { return __fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)); }
__device__ __forceinline__ double sq_sum(double x, double y) { return __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)); }

// single-instruction min / max (FMNMX / DMNMX); glacier cells never carry NaN here
__device__ __forceinline__ float fmax_(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ float fmin_(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ double fmax_(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ double fmin_(double a, double b) { return fmin(a, b); }

// ---- per-step area statistics: warp sums in batches of steps ------------------------------------
// Every step a lane parks its NQ per-step values (one "entry"; with fused members one per (step, member)
// pair) in its warp's batch buffer.  Once E entries are parked, lane r adds the 32 lane values of row
// r = entry * NQ + statistic and writes that row's slot: per step NQ stores instead of a shuffle butterfly
// (its shuffles, selects and chain of five shuffle latencies).  The sum adds lanes l and l ^ 16 first, then
// ^ 8, ^ 4, ^ 2, ^ 1: the tree a butterfly over the lanes forms, so the sums are the same bits whichever
// way they are formed, and deterministic.
// Layout: [chunk][row][16 bytes], a chunk being the values of 16 / sizeof(R) consecutive lanes.  The row
// pitch is odd (in chunks): a warp's stores of one row, and a quarter warp's 16-byte loads of one chunk of
// eight consecutive rows, meet every bank at most once.
__host__ __device__ constexpr int stat_batch_pitch(int rows) { return (rows | 1) * 16; }   // bytes between chunks
__host__ __device__ constexpr int stat_batch_bytes(int r_size, int rows) {                  // per warp
  return 32 / (16 / r_size) * stat_batch_pitch(rows);
}
template <typename R, int NQ, int E>
struct StatBatch {
  static constexpr int kRows = E * NQ;
  static constexpr int kPitch = stat_batch_pitch(kRows);
  static constexpr int kLanesPerChunk = 16 / (int)sizeof(R);
  static constexpr int kBytes = stat_batch_bytes((int)sizeof(R), kRows);
  static_assert(E >= 1 && kRows <= 32, "one row per lane");
};
// Statistic q of a batch entry is slot column stat_column(q): without the station blend the longwave
// column (K_LWD) is not summed in the kernel (finalize_stats_kernel takes it from the DEM moments), so the
// batch leaves it out.  Columns kStatsK + M_* are the sub-surface model's.
template <bool LWD>
__host__ __device__ constexpr int stat_column(int q) { return LWD || q < K_LWD ? q : q + 1; }
// where lane `lane` parks its value of row 0
template <typename R, int NQ, int E>
__device__ __forceinline__ int batch_lane(int lane) {
  using B = StatBatch<R, NQ, E>;
  return lane / B::kLanesPerChunk * B::kPitch + lane % B::kLanesPerChunk * (int)sizeof(R);
}
template <typename R, int NQ>
__device__ __forceinline__ void batch_put(unsigned char* lane_buf, int entry, const R (&v)[NQ]) {
#pragma unroll
  for (int q = 0; q < NQ; ++q) *reinterpret_cast<R*>(lane_buf + (entry * NQ + q) * 16) = v[q];
}
// the 32 lane values of the row whose chunk 0 is at `row`, added in the tree order above (packed adds:
// pair i holds lanes 2i, 2i + 1)
template <int PITCH>
__device__ __forceinline__ float lane_sum(const unsigned char* row, float) {
  V2<float> a[8];                                   // lanes (2i, 2i + 1) + (2i + 16, 2i + 17)
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(row + c * PITCH);
    const ulonglong2 y = *reinterpret_cast<const ulonglong2*>(row + (c + 4) * PITCH);
    a[2 * c] = add2(V2<float>{x.x}, V2<float>{y.x});
    a[2 * c + 1] = add2(V2<float>{x.y}, V2<float>{y.y});
  }
#pragma unroll
  for (int h = 4; h > 0; h >>= 1) {
#pragma unroll
    for (int i = 0; i < h; ++i) a[i] = add2(a[i], a[i + h]);
  }
  return a[0].lo() + a[0].hi();
}
template <int PITCH>
__device__ __forceinline__ double lane_sum(const unsigned char* row, double) {
  double a[16];                                     // lanes i + (i + 16)
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const double2 x = *reinterpret_cast<const double2*>(row + c * PITCH);
    const double2 y = *reinterpret_cast<const double2*>(row + (c + 8) * PITCH);
    a[2 * c] = x.x + y.x;
    a[2 * c + 1] = x.y + y.y;
  }
#pragma unroll
  for (int h = 8; h > 0; h >>= 1) {
#pragma unroll
    for (int i = 0; i < h; ++i) a[i] += a[i + h];
  }
  return a[0];
}
// sums the first n_entries entries of the batch into their slots: statistic q of entry e goes to column
// c = stat_column<LWD>(q), slots[e * kStatsK + c] (c < kStatsK) or slots_m[e * kStatsM + c - kStatsK].  The
// caller orders it after the lanes' batch_put and before the next batch_put with __syncwarp.
template <typename R, int NQ, int E, bool LWD>
__device__ __forceinline__ void batch_reduce(const unsigned char* warp_buf, int n_entries, int lane, R* slots, R* slots_m) {
  if (lane < n_entries * NQ) {
    const int e = lane / NQ, c = stat_column<LWD>(lane - e * NQ);
    const R v = lane_sum<StatBatch<R, NQ, E>::kPitch>(warp_buf + lane * 16, R{});
    if (c < kStatsK) slots[e * kStatsK + c] = v;
    else slots_m[e * kStatsM + (c - kStatsK)] = v;
  }
}

// Sum of 8 per-thread values over the 32 lanes with 15 shuffles instead of 40: each butterfly stage
// halves the number of values a lane still carries.  Returns the total of statistic
// stat_of_lane(lane) = 4*bit4 + 2*bit3 + bit2; the same tree as the batches', hence the same bits.  For the
// kernel instances whose shared memory has no room for a batch buffer (StatBatchFor).
template <typename R>
__device__ __forceinline__ R warp_reduce8(const R* v, int lane) {   // v[0 .. 7]
  const unsigned full = 0xffffffffu;
  R a[4], b[2], c;
  bool hi = (lane & 16) != 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const R send = hi ? v[i] : v[i + 4];
    const R keep = hi ? v[i + 4] : v[i];
    a[i] = keep + __shfl_xor_sync(full, send, 16);
  }
  hi = (lane & 8) != 0;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const R send = hi ? a[i] : a[i + 2];
    const R keep = hi ? a[i + 2] : a[i];
    b[i] = keep + __shfl_xor_sync(full, send, 8);
  }
  hi = (lane & 4) != 0;
  {
    const R send = hi ? b[0] : b[1];
    const R keep = hi ? b[1] : b[0];
    c = keep + __shfl_xor_sync(full, send, 4);
  }
  c += __shfl_xor_sync(full, c, 2);
  c += __shfl_xor_sync(full, c, 1);
  return c;
}
__device__ __forceinline__ int stat_of_lane(int lane) {
  return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
}

// =================================================================================================
// set-up kernels
// =================================================================================================
// terrain normal from the 4-neighbourhood; a missing neighbour is mirrored from the opposite one
// (DESIGN.md "Insolation specification"; oracle/insolation_oracle.py:terrain_normals)
template <typename R>
__global__ void terrain_kernel(const float* __restrict__ dem, const float* __restrict__ terr, int dem_pitch, int rows_full,
                               int cols, int pitch, int band_row0, int band_rows_pad, R inv2cell, R* __restrict__ nx,
                               R* __restrict__ ny, R* __restrict__ nz) {
  // `dem` decides which cells are glacier cells; the elevations of the cell and its neighbours come
  // from `terr` -- the same raster, or the uncropped terrain (enrgy_set_terrain): SAGA is handed the
  // uncropped DEM (reference model.py:469 -> saga_lighting.py:42), so slopes at the glacier margin see
  // their real neighbours
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= pitch) return;
  const float qnan = __int_as_float(0x7fc00000);
  auto at = [&](int rr, int cc) -> float {
    if (rr < 0 || rr >= rows_full || cc < 0 || cc >= cols) return qnan;
    return terr[(size_t)rr * dem_pitch + cc];
  };
  for (int rb = blockIdx.y; rb < band_rows_pad; rb += gridDim.y) {
    const int r = rb + band_row0;
    const size_t o = (size_t)rb * pitch + c;
    const bool glacier = r < rows_full && c < cols && dem[(size_t)r * dem_pitch + c] == dem[(size_t)r * dem_pitch + c];
    const float zf = glacier ? at(r, c) : qnan;
    if (!(zf == zf)) {
      nx[o] = (R)qnan; ny[o] = (R)qnan; nz[o] = (R)qnan;
      continue;
    }
    const R z = (R)zf;
    auto one_sided = [&](float a, float b) -> R {
      if (a == a) return (R)a - z;
      if (b == b) return z - (R)b;
      return (R)0;
    };
    const float zn = at(r - 1, c), zs = at(r + 1, c), ze = at(r, c + 1), zw = at(r, c - 1);
    const R gy = (one_sided(zn, zs) - one_sided(zs, zn)) * inv2cell;
    const R gx = (one_sided(ze, zw) - one_sided(zw, ze)) * inv2cell;
    // stored as (nx/nz, ny/nz, nz) = (-gx, -gy, nz): cos(incidence) = nz * (u + px*e + py*n), which
    // costs the time loop two FMAs per sub-step instead of three
    const R inv = Num<R>::rsqrt_((R)1 + gx * gx + gy * gy);
    nx[o] = -gx;
    ny[o] = -gy;
    nz[o] = inv;
  }
}

template <typename R>
cudaError_t launch_terrain(const float* dem, const float* terr, int dem_pitch, int rows_full, int cols, int pitch,
                           int band_row0, int band_rows_pad, double cell, R* nx, R* ny, R* nz,
                           cudaStream_t stream) {
  dim3 grid((pitch + 255) / 256, grid_rows(band_rows_pad));
  terrain_kernel<R><<<grid, 256, 0, stream>>>(dem, terr, dem_pitch, rows_full, cols, pitch, band_row0, band_rows_pad,
                                              (R)(1.0 / (2.0 * cell)), nx, ny, nz);
  return cudaGetLastError();
}
template cudaError_t launch_terrain<float>(const float*, const float*, int, int, int, int, int, int, double, float*, float*, float*, cudaStream_t);
template cudaError_t launch_terrain<double>(const float*, const float*, int, int, int, int, int, int, double, double*, double*, double*, cudaStream_t);

// valid (non-NaN DEM) cells per tile
__global__ void tile_scan_kernel(const float* __restrict__ dem, int pitch, int band_row0,
                                 int band_rows, int cols, int tile_h, int tile_w, int tiles_c,
                                 int* __restrict__ counts) {
  const int tc = blockIdx.x;
  const int tiles_r = (band_rows + tile_h - 1) / tile_h;
  __shared__ int s[32];
  for (int tr = blockIdx.y; tr < tiles_r; tr += gridDim.y) {
    int n = 0;
    for (int i = threadIdx.x; i < tile_h * tile_w; i += blockDim.x) {
      const int rb = tr * tile_h + i / tile_w;
      const int c = tc * tile_w + i % tile_w;
      if (rb < band_rows && c < cols) {
        const float z = dem[(size_t)(rb + band_row0) * pitch + c];
        n += (z == z) ? 1 : 0;
      }
    }
    n = __reduce_add_sync(0xffffffffu, n);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s[w];
      counts[(size_t)tr * tiles_c + tc] = tot;
    }
    __syncthreads();                    // s is refilled by the next row of tiles
  }
}
cudaError_t launch_tile_scan(const float* dem, int pitch, int band_row0, int band_rows, int cols,
                             int tile_h, int tile_w, int tiles_r, int tiles_c, int* counts,
                             cudaStream_t stream) {
  tile_scan_kernel<<<dim3(tiles_c, grid_rows(tiles_r)), 256, 0, stream>>>(dem, pitch, band_row0, band_rows, cols,
                                                                           tile_h, tile_w, tiles_c, counts);
  return cudaGetLastError();
}

// counters[0] += cells valid in the DEM but NaN in `other`; counters[1] += the opposite
__global__ void mask_check_kernel(const float* __restrict__ dem, int dem_pitch,
                                  const float* __restrict__ other, int pitch, int band_row0,
                                  int band_rows, int cols, unsigned long long* counters) {
  unsigned a = 0, b = 0;
  const size_t n = (size_t)band_rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int rb = (int)(i / cols), c = (int)(i % cols);
    const float z = dem[(size_t)(rb + band_row0) * dem_pitch + c];
    const float o = other[(size_t)rb * pitch + c];
    const bool vz = z == z, vo = o == o;
    a += (vz && !vo) ? 1u : 0u;
    b += (!vz && vo) ? 1u : 0u;
  }
  a = __reduce_add_sync(0xffffffffu, a);
  b = __reduce_add_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0) {
    if (a) atomicAdd(&counters[0], (unsigned long long)a);
    if (b) atomicAdd(&counters[1], (unsigned long long)b);
  }
}
cudaError_t launch_mask_check(const float* dem, int dem_pitch, const float* other, int pitch,
                              int band_row0, int band_rows, int cols, unsigned long long* counters,
                              cudaStream_t stream) {
  mask_check_kernel<<<592, 256, 0, stream>>>(dem, dem_pitch, other, pitch, band_row0, band_rows, cols,
                                             counters);
  return cudaGetLastError();
}

// SWE statistics of the initial raster over ALL its non-NaN cells (first CSV row quirk).
// block_out[b] = {sum, count(swe > 0), count(non-NaN)}; summed on the host in block order.
__global__ void swe0_stats_kernel(const float* __restrict__ swe, int pitch, int band_rows, int cols,
                                  double* __restrict__ block_out) {
  double s = 0.0, ns = 0.0, nv = 0.0;
  const size_t n = (size_t)band_rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int rb = (int)(i / cols), c = (int)(i % cols);
    const float v = swe[(size_t)rb * pitch + c];
    if (v == v) {
      s += (double)v;
      nv += 1.0;
      if (v > 0.f) ns += 1.0;
    }
  }
  __shared__ double sh[3][kThreads];
  sh[0][threadIdx.x] = s; sh[1][threadIdx.x] = ns; sh[2][threadIdx.x] = nv;
  __syncthreads();
  for (int off = kThreads / 2; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) {
      for (int q = 0; q < 3; ++q) sh[q][threadIdx.x] += sh[q][threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    for (int q = 0; q < 3; ++q) block_out[blockIdx.x * 3 + q] = sh[q][0];
  }
}
cudaError_t launch_swe0_stats(const float* swe, int pitch, int band_rows, int cols, double* block_out,
                              int blocks, cudaStream_t stream) {
  swe0_stats_kernel<<<blocks, kThreads, 0, stream>>>(swe, pitch, band_rows, cols, block_out);
  return cudaGetLastError();
}

template <typename R>
__global__ void pad_convert_kernel(const float* __restrict__ src, R* __restrict__ dst, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    dst[i] = (R)src[i];
  }
}
template <typename R>
cudaError_t launch_pad_convert(const float* src, R* dst, size_t n, cudaStream_t stream) {
  pad_convert_kernel<R><<<1184, 256, 0, stream>>>(src, dst, n);
  return cudaGetLastError();
}
template cudaError_t launch_pad_convert<float>(const float*, float*, size_t, cudaStream_t);
template cudaError_t launch_pad_convert<double>(const float*, double*, size_t, cudaStream_t);

template <typename R, typename O>
__global__ void unpad_kernel(const R* __restrict__ src, int pitch, int rows, int cols, O* __restrict__ dst) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    dst[i] = (O)src[(size_t)r * pitch + c];
  }
}
template <typename R>
cudaError_t launch_unpad_state(const R* src, int pitch, int rows, int cols, int dtype, void* dst,
                               cudaStream_t stream) {
  if (dtype == 32) {
    unpad_kernel<R, float><<<1184, 256, 0, stream>>>(src, pitch, rows, cols, (float*)dst);
  } else {
    unpad_kernel<R, double><<<1184, 256, 0, stream>>>(src, pitch, rows, cols, (double*)dst);
  }
  return cudaGetLastError();
}
template cudaError_t launch_unpad_state<float>(const float*, int, int, int, int, void*, cudaStream_t);
template cudaError_t launch_unpad_state<double>(const double*, int, int, int, int, void*, cudaStream_t);

// sum over the glacier cells of (dem - elev_aws)^k, k = 0..4, per block (summed on the host in block
// order): the area sum of the downward longwave flux is a quartic in the lapse-rate temperature
template <typename R>
__global__ void moments_kernel(const float* __restrict__ dem, int dem_pitch, int band_row0, int band_rows,
                               int cols, R elev, double* __restrict__ block_out) {
  double m[5] = {0, 0, 0, 0, 0};
  const size_t n = (size_t)band_rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int rb = (int)(i / cols), c = (int)(i % cols);
    const float z = dem[(size_t)(rb + band_row0) * dem_pitch + c];
    if (z == z) {
      const double d = (double)((R)z - elev);       // the kernel's own delta (float32 in F32 mode)
      const double d2 = d * d;
      m[0] += 1.0; m[1] += d; m[2] += d2; m[3] += d2 * d; m[4] += d2 * d2;
    }
  }
  __shared__ double sh[5][kThreads];
  for (int q = 0; q < 5; ++q) sh[q][threadIdx.x] = m[q];
  __syncthreads();
  for (int off = kThreads / 2; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) {
      for (int q = 0; q < 5; ++q) sh[q][threadIdx.x] += sh[q][threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    for (int q = 0; q < 5; ++q) block_out[blockIdx.x * 5 + q] = sh[q][0];
  }
}
template <typename R>
cudaError_t launch_moments(const float* dem, int dem_pitch, int band_row0, int band_rows, int cols, double elev,
                           double* block_out, int blocks, cudaStream_t stream) {
  moments_kernel<R><<<blocks, kThreads, 0, stream>>>(dem, dem_pitch, band_row0, band_rows, cols, (R)elev, block_out);
  return cudaGetLastError();
}
template cudaError_t launch_moments<float>(const float*, int, int, int, int, double, double*, int, cudaStream_t);
template cudaError_t launch_moments<double>(const float*, int, int, int, int, double, double*, int, cudaStream_t);

// off-glacier cells of the state rasters become NaN with the first step (model.py:258: swe -= NaN);
// the fused kernel only visits tiles that hold glacier cells, this covers the rest.
template <typename R>
__global__ void nan_offglacier_kernel(const float* __restrict__ dem, int dem_pitch, int pitch,
                                      int band_row0, int band_rows, int cols, R* __restrict__ swe,
                                      R* __restrict__ tsn, R* __restrict__ tic) {
  const size_t n = (size_t)band_rows * cols;
  const R qnan = (R)__int_as_float(0x7fc00000);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int rb = (int)(i / cols), c = (int)(i % cols);
    const float z = dem[(size_t)(rb + band_row0) * dem_pitch + c];
    if (!(z == z)) {
      const size_t o = (size_t)rb * pitch + c;
      swe[o] = qnan; tsn[o] = qnan; tic[o] = qnan;
    }
  }
}
template <typename R>
cudaError_t launch_nan_offglacier(const float* dem, int dem_pitch, int pitch, int band_row0,
                                  int band_rows, int cols, R* swe, R* tsn, R* tic, cudaStream_t stream) {
  nan_offglacier_kernel<R><<<1184, 256, 0, stream>>>(dem, dem_pitch, pitch, band_row0, band_rows, cols, swe,
                                                     tsn, tic);
  return cudaGetLastError();
}
template cudaError_t launch_nan_offglacier<float>(const float*, int, int, int, int, int, float*, float*, float*, cudaStream_t);
template cudaError_t launch_nan_offglacier<double>(const float*, int, int, int, int, int, double*, double*, double*, cudaStream_t);

// =================================================================================================
// the fused energy-balance kernel
// =================================================================================================
// Warps per CTA: the warps of a CTA share one staged copy of the AWS records.
#ifndef ENRGY_WARPS32
#define ENRGY_WARPS32 4      // float32: 4 CTAs x 4 warps at 128 registers (profiles/r01_summary.md)
#endif
#ifndef ENRGY_WARPS64
#define ENRGY_WARPS64 4      // float64: 3 CTAs x 4 warps at 156 registers, no spills (profiles/r01_summary.md)
#endif
template <typename R, int INSOL>
constexpr int kWarpsFor = sizeof(R) == 4 ? ENRGY_WARPS32 : ENRGY_WARPS64;
__host__ __device__ constexpr int warps_x(int w) { return w >= 4 ? 4 : w; }          // patches side by side in a tile

// Option, OFF: sunlit masks through a per-warp ring in shared memory (float32 plain runs with masks, K = 8):
// the 32-byte sector of sub-step j + kRingAhead is fetched by an asynchronous copy (two lanes, 16 bytes
// each) while sub-step j is computed, and read back with two broadcast LDS.128.  Tried because ncu of the
// LDG version shows 2.2 warps per issued instruction on the long scoreboard and an L1 hit rate of 50 % (the
// CCTL.PF1 prefetch does not land, whatever its distance) -- but measured SLOWER: 16.14 against 15.75 ms
// on 4096^2 x 384 steps; the commit / wait / syncwarp per sub-step cost more than the latency they hide,
// which the other 15 warps of the SM already cover.
#ifndef ENRGY_MASK_RING
#define ENRGY_MASK_RING 0
#endif
constexpr int kRingSlots = 16, kRingAhead = 8;
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Shared-memory carve-up of a CTA.  The capacities of a time block (steps, sunlit sub-steps) are
// run-time values chosen by the host (64 / 256, grown to the largest sub-step count of one step).
template <typename R>
struct SmemPlan {
  int steps, subs, members, stations, slots, slots_m, batch, ring, full, total;   // byte offsets and the total size
};
// nm: ensemble members fused into one pass (1 = a plain run: no member records); ns: weather stations
// blended (1 = the reference's single AWS: no station records)
// One barrier per time block instead of two: the warps' statistic slots are double-buffered, so the flush of
// block b may still be running while block b + 1 fills the other set (ncu: 0.33 warps per issued
// instruction waited at the two barriers).  float32 runs with sunlit masks only, where the warps of a CTA
// drift apart on their mask loads (+5.8 %); without masks the extra 8 KB of shared memory per CTA cost 1 %.
#ifndef ENRGY_ONE_BARRIER
#define ENRGY_ONE_BARRIER 1
#endif
template <typename R, bool MSM, int NM, int INSOL>
constexpr bool kOneBarrier = ENRGY_ONE_BARRIER && sizeof(R) == 4 && !MSM && NM == 1 && INSOL == kInsolMasked;

// batch_bytes: the warps' statistics batch buffers (StatBatchFor)
template <typename R>
__host__ __device__ constexpr SmemPlan<R> smem_plan(int warps, int cap_steps, int cap_subs, bool with_subs, bool msm,
                                                    int nm, int ns, bool with_masks, int batch_bytes) {
  SmemPlan<R> p{};
  int o = 0;
  p.steps = o;   o += 2 * cap_steps * (int)sizeof(StepRec<R>);
  p.subs = o;    o += with_subs ? 2 * cap_subs * (int)sizeof(SubRec<R>) : 0;
  p.members = o; o += nm > 1 ? 2 * cap_steps * nm * (int)sizeof(MemberRec<R>) : 0;
  p.stations = o; o += ns > 1 ? 2 * cap_steps * ns * (int)sizeof(StationRec<R>) : 0;
  const bool two_sets = ENRGY_ONE_BARRIER && sizeof(R) == 4 && !msm && nm == 1 && with_masks;
  p.slots = o;   o += (two_sets ? 2 : 1) * warps * cap_steps * nm * kStatsK * (int)sizeof(R);
  p.slots_m = o; o += msm ? warps * cap_steps * kStatsM * (int)sizeof(R) : 0;
  o = (o + 15) / 16 * 16;
  p.batch = o;   o += batch_bytes;
  p.ring = o;    o += (ENRGY_MASK_RING && with_masks) ? warps * kRingSlots * 32 : 0;
  p.full = o;    o += 16;
  p.total = (o + 127) / 128 * 128;
  return p;
}

// tuning knobs (cells per thread, minimum resident CTAs per SM), overridable at build time
#ifndef ENRGY_K32
#define ENRGY_K32 8
#endif
#ifndef ENRGY_K64
#define ENRGY_K64 4
#endif
#ifndef ENRGY_MINB32
#define ENRGY_MINB32 4
#endif
#ifndef ENRGY_MINB64
#define ENRGY_MINB64 3
#endif

#ifndef ENRGY_SUB_UNROLL
#define ENRGY_SUB_UNROLL 4
#endif
constexpr int kSubUnroll = ENRGY_SUB_UNROLL;   // unroll factor of the insolation sub-step loop
#ifndef ENRGY_MASK_AHEAD
#define ENRGY_MASK_AHEAD 4
#endif
constexpr int kMaskAhead = ENRGY_MASK_AHEAD;   // sunlit masks are prefetched this many sub-steps ahead
// NM > 1: NM ensemble members (BASELINE config C5) in one pass.  Members differ in an albedo offset and
// in the roughness lengths, i.e. in (1 - albedo) and in the two exchange-coefficient scalars of a step;
// the terrain, the insolation of every sub-step (sunlit masks included), the lapse-rate meteorology, the
// reciprocals, the flux factors and the net longwave term of a cell-step are member-invariant and are
// computed ONCE, then each member adds its shortwave term, clamps, melts and updates ITS state
// (swe, total_ice and 1 - albedo per member and cell in registers).  KT = rows of a warp patch in the
// handle's tile list; a pass with fewer cells per thread (K < KT) walks the patch in KT / K parts.
#ifndef ENRGY_MINB_MEMBERS
#define ENRGY_MINB_MEMBERS 3
#endif
// Statistics batch of a kernel instance: entries per batch (0: no buffer, the warp reduces every step with
// warp_reduce8) and the values of an entry.  The batch is as large as one row per lane allows (float64:
// half the lanes), but never so large that the buffer costs the instance a CTA per SM at the default
// time-block capacities: CTAs per SM by shared memory (228 KB per SM, 1 KB of it reserved per CTA) stay at
// least what they were without the buffer, up to the launch bounds' minimum.  Where even one entry costs a
// CTA (float64 with four fused members or with the station blend and its sub-step records), the instance
// keeps the butterfly.
template <typename R, int INSOL, bool MSM, bool DUMP, int NM, bool STATS, int NS>
struct StatBatchFor {
  static constexpr bool kLwd = NS > 1;                                   // K_LWD summed in the kernel
  static constexpr int NQ = kStatsK - (kLwd ? 0 : 1) + (MSM ? kStatsM : 0);
  static constexpr int W = kWarpsFor<R, INSOL>;
  static constexpr int kMinCtas = NM > 2 ? ENRGY_MINB_MEMBERS : sizeof(R) == 4 ? ENRGY_MINB32 : ENRGY_MINB64;
  static constexpr int bytes(int e) { return e > 0 ? W * stat_batch_bytes((int)sizeof(R), e * NQ) : 0; }
  static constexpr int ctas(int e) {
    return 233472 / (smem_plan<R>(W, kStepsPerBlock, kSubsPerBlock, INSOL != kInsolStreamed, MSM, NM, NS,
                                  INSOL == kInsolMasked, bytes(e)).total + 1024);
  }
  static constexpr int pick() {
    // (the sub-surface model: its batches added spills to three of its instances in ptxas)
    if (!STATS || DUMP || MSM) return 0;
    const int target = ctas(0) < kMinCtas ? ctas(0) : kMinCtas;
    // (with sunlit masks at most 2 entries, summed at the end of the step: every arrangement with more spills
    // in ptxas -- the mask loads keep more registers live through the step)
    const int most = INSOL == kInsolMasked ? 2 : (sizeof(R) == 4 ? 32 : 16) / NQ;
    for (int e = most; e > 0; --e)
      if (ctas(e) >= target) return e;
    return 0;
  }
  static constexpr int kEntries = pick();
  static constexpr int kBytes = bytes(kEntries);                         // per CTA
};
// STATS = false (fused members only): no per-step area statistics -- their adds and the warp butterfly
// are a third of a member's share of a step; the season totals come from the final rasters instead.
// NS > 1: up to NS weather stations blended per cell (BASELINE config C4; specification in
// oracle/enrgy_oracle.py "several weather stations"): inverse-squared-distance weights and the weights
// folded with the vapour-pressure reduction live in registers per cell, the stations' per-step values are
// staged like the AWS records; unused stations carry weight zero.  The shortwave is attenuated by the
// cloud field relative to the primary station (Beer-Lambert, one exp per cell-step).  With the sub-surface
// model the blended T, p and e drive the surface terms and the conduction step like the AWS values do.
template <typename R, int K, int INSOL, bool MSM, bool DUMP, int NM = 1, int KT = K, bool STATS = true, int NS = 1>
__global__ void __launch_bounds__(32 * kWarpsFor<R, INSOL>, NM > 2 ? ENRGY_MINB_MEMBERS : sizeof(R) == 4 ? ENRGY_MINB32 : ENRGY_MINB64)
energy_balance_kernel(const KernelArgs<R> a) {
  static_assert(NM == 1 || (!MSM && !DUMP), "fused members: no sub-surface model, no dump");
  static_assert(KT % K == 0, "a patch is walked in whole parts");
  static_assert(STATS || NM > 1, "only fused members run without statistics");
  static_assert(NS == 1 || NM == 1, "station blend: no fused members");
  constexpr int W = kWarpsFor<R, INSOL>;           // warps per CTA
  constexpr int WX = warps_x(W), WY = W / WX;      // patches of a tile: WX across, WY down
  constexpr int NT = 32 * W;                       // threads per CTA
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int cap_steps = a.cap_steps, cap_subs = a.cap_subs;
  using SB = StatBatchFor<R, INSOL, MSM, DUMP, NM, STATS, NS>;
  const SmemPlan<R> plan = smem_plan<R>(W, cap_steps, cap_subs, INSOL != kInsolStreamed, MSM, NM, NS, INSOL == kInsolMasked,
                                         SB::kBytes);
  StationRec<R>* const sm_stations = reinterpret_cast<StationRec<R>*>(smem_raw + plan.stations);  // [2][cap_steps][NS]
  StepRec<R>* const sm_steps = reinterpret_cast<StepRec<R>*>(smem_raw + plan.steps);     // [2][cap_steps]
  SubRec<R>* const sm_subs = reinterpret_cast<SubRec<R>*>(smem_raw + plan.subs);         // [2][cap_subs]
  MemberRec<R>* const sm_members = reinterpret_cast<MemberRec<R>*>(smem_raw + plan.members);  // [2][cap_steps][NM]
  R* const sm_slots0 = reinterpret_cast<R*>(smem_raw + plan.slots);                      // [sets][W][cap_steps][NM][kStatsK]
  constexpr bool ONE_BAR = kOneBarrier<R, MSM, NM, INSOL>;
  unsigned slot_set = 0;                                                                 // flips per time block (ONE_BAR)
  R* const sm_slots_m = reinterpret_cast<R*>(smem_raw + plan.slots_m);                   // [W][cap_steps][kStatsM]
  uint64_t* const sm_full = reinterpret_cast<uint64_t*>(smem_raw + plan.full);           // [2]

  constexpr int TILE_H = WY * KT, TILE_W = 32 * WX;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // this warp's statistics batch: NQ values per entry, E entries (E = 0: no batch, warp_reduce8 per step)
  constexpr int NQ = SB::NQ, E = SB::kEntries;
  const int batch_off = plan.batch + warp * (SB::kBytes / W);               // byte offsets in smem_raw
  int batch_mine = batch_off;                                                 // ... of this lane's value of row 0
  if constexpr (E > 0) batch_mine += batch_lane<R, NQ, E>(lane);
  const R qnan = (R)__int_as_float(0x7fc00000);

  if (tid == 0) {
    mbar_init(&sm_full[0], 1);
    mbar_init(&sm_full[1], 1);
    fence_mbar_init();
  }
  __syncthreads();
  unsigned phase[2] = {0u, 0u};

  auto issue_block = [&](int b, int buf) {
    // one elected thread: stage the per-step records (and sub-step records) of time block b
    const TimeBlock tb = a.blocks[b];
    const unsigned n_steps = (unsigned)(tb.t_end - tb.t_begin);
    const unsigned n_subs = (unsigned)(tb.sub_end - tb.sub_begin);
    unsigned bytes = n_steps * (unsigned)sizeof(StepRec<R>);
    if (INSOL != kInsolStreamed) bytes += n_subs * (unsigned)sizeof(SubRec<R>);
    if (NM > 1) bytes += n_steps * NM * (unsigned)sizeof(MemberRec<R>);
    if (NS > 1) bytes += n_steps * NS * (unsigned)sizeof(StationRec<R>);
    fence_proxy_async();
    mbar_expect_tx(&sm_full[buf], bytes);
    tma_bulk_g2s(sm_steps + buf * cap_steps, a.steps + tb.t_begin, n_steps * (unsigned)sizeof(StepRec<R>),
                 &sm_full[buf]);
    if (INSOL != kInsolStreamed && n_subs) {
      tma_bulk_g2s(sm_subs + buf * cap_subs, a.subs + tb.sub_begin, n_subs * (unsigned)sizeof(SubRec<R>),
                   &sm_full[buf]);
    }
    if (NM > 1) {
      tma_bulk_g2s(sm_members + buf * cap_steps * NM, a.member_recs + (size_t)tb.t_begin * NM,
                   n_steps * NM * (unsigned)sizeof(MemberRec<R>), &sm_full[buf]);
    }
    if (NS > 1) {
      tma_bulk_g2s(sm_stations + buf * cap_steps * NS, a.station_recs + (size_t)tb.t_begin * NS,
                   n_steps * NS * (unsigned)sizeof(StationRec<R>), &sm_full[buf]);
    }
  };

  const int n_steps_run = a.t1 - a.t0;
  // this CTA's rows of per-step sums (in R: in float32 mode the 40 MB of rows stay L2-resident)
  constexpr int kRow = MSM ? kStatsP : kStatsK;
  R* my_partials = a.partials ? a.partials + (size_t)blockIdx.x * n_steps_run * NM * kRow : nullptr;
  constexpr int NB = MSM ? kMaxLayers + 1 : 1;       // boundary temperatures kept per cell

  // per-member constants (NM == 1: the handle's own)
  auto m_offset = [&](int m) -> R { return NM > 1 ? a.member_offset[m] : a.albedo_offset; };
  auto m_alb_ice = [&](int m) -> R { return NM > 1 ? a.member_albedo_ice[m] : a.albedo_ice; };
  const size_t m_stride = NM > 1 ? a.member_stride : 0;     // elements between the state rasters of members

  for (int ti = blockIdx.x; ti < a.n_tiles; ti += gridDim.x)
  for (int part = 0; part < KT / K; ++part) {
    const int2 tile = a.tiles[ti];
    // ---- prologue: per-cell invariants and state into registers --------------------------------
    // A warp owns a compact 32-column x K-row patch (lane = column): every raster access is one
    // coalesced 128 B line per row, and the K = 8 rows are one row group of the sunlit masks.  The K cells
    // of a thread are kept as K/2 PAIRS (rows 2q, 2q+1): all multiply/add arithmetic of the time
    // loop runs on both cells of a pair with one packed instruction (V2, FFMA2/FADD2/FMUL2).
    constexpr int KP = K / 2;
    static_assert(K % 2 == 0, "cells per thread come in pairs");
    using V = V2<R>;
    const int row0 = tile.x * TILE_H + (warp / WX) * KT + part * K;   // band-local row of cell 0
    const int colx = tile.y * TILE_W + (warp % WX) * 32 + lane;   // this lane's column
    V delta2[KP], pw2[NS][KP], nx2[KP], ny2[KP], nz2[KP];   // pw2[k]: (weight of station k) x 10^(-(z - z_k) / 6300)
    V wst2[NS > 1 ? NS : 1][KP];                           // weights of the stations (NS > 1)
    V om2[NM][KP], swe2[NM][KP], tic2[NM][KP];         // per member: 1 - albedo (ice surface), SWE, ice-melt total
    R tl[K][NB];                   // sub-surface boundary temperatures [deg C] (MSM)
    // The reference's top boundary turns float64 after its first tick (NEP 50: float32 array +
    // float64 increment), so its round-off does not random-walk at float32 spacing; the float32
    // kernel keeps that one temperature per cell as a float64 accumulator of float32 increments.
    double t0_acc[MSM ? K : 1];
    unsigned valid_bits = 0;
    int cur_pair = -1;
    R cur_w = (R)-1;
#pragma unroll
    for (int q = 0; q < KP; ++q) {
      R d_[2], p_[NS][2], w_[NS][2], x_[2], y_[2], n_[2], s_[NM][2], t_[NM][2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int i = 2 * q + h;
        const int rowb = row0 + i;
        const size_t o = (size_t)rowb * a.pitch + colx;
        const bool inside = rowb < a.band_rows && colx < a.cols;
        float z = inside ? __ldg(a.dem + (size_t)(rowb + a.band_row0) * a.dem_pitch + colx) : __int_as_float(0x7fc00000);
        const bool v = z == z;
        valid_bits |= v ? (1u << i) : 0u;
        if (!v) z = (float)a.elev_aws;           // keep the arithmetic of masked cells finite
        d_[h] = (R)z - a.elev_aws;               // var_classes.py:114
        // var_classes.py:162.  float32: the reference's power is NumPy's float32 power of a float32
        // exponent (libm, correctly rounded in practice); powf here may be a few ulp off, which the
        // vapour-pressure difference e - es amplifies into the largest float32 error of the whole
        // balance (4e-5 W m-2) -- so the power is taken in float64 and rounded once (prologue only)
        p_[0][h] = (R)pow(10.0, (double)(-d_[h] / (R)kVapourScale));
        w_[0][h] = (R)1;
        if (NS > 1) {
          // inverse squared distance in cell units, softened by half a cell; w_k = q_k / sum_j q_j
          R qk[NS];
          const R rr = (R)(rowb + a.band_row0), cc = (R)colx;
#pragma unroll
          for (int k = 0; k < NS; ++k) {
            const R dr = rr - a.st_row[k], dc = cc - a.st_col[k];
            qk[k] = k < a.n_stations ? div_rn((R)1, add_rn(add_rn(mul_rn(dr, dr), mul_rn(dc, dc)), (R)0.25)) : (R)0;
          }
          R tot = qk[0];
#pragma unroll
          for (int k = 1; k < NS; ++k) tot = add_rn(tot, qk[k]);
          R dsum = (R)0;
#pragma unroll
          for (int k = 0; k < NS; ++k) {
            const R wk = div_rn(qk[k], tot);
            const R dzk = (R)z - a.st_elev[k];
            const R term = mul_rn(wk, dzk);
            dsum = k == 0 ? term : add_rn(dsum, term);
            w_[k][h] = wk;
            p_[k][h] = mul_rn(wk, (R)pow(10.0, (double)(-dzk / (R)kVapourScale)));
          }
          d_[h] = dsum;                            // sum_k w_k (z - z_k) replaces z - elev_aws
        }
        if (INSOL != kInsolStreamed) {
          x_[h] = v ? a.nx[o] : (R)0;
          y_[h] = v ? a.ny[o] : (R)0;
          n_[h] = v ? a.nz[o] : (R)1;
        } else {
          x_[h] = y_[h] = (R)0; n_[h] = (R)1;
        }
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          s_[m][h] = v ? a.swe[m * m_stride + o] : (R)0;
          t_[m][h] = v ? a.total_ice[m * m_stride + o] : (R)0;
        }
        if (MSM) {
#pragma unroll
          for (int l = 0; l < NB; ++l) {
            tl[i][l] = (v && l <= a.msm.layers) ? a.layer_t[(size_t)l * a.layer_stride + o] : (R)0;
          }
          t0_acc[i] = (double)tl[i][0];
        }
      }
      delta2[q] = V::make(d_[0], d_[1]);
      // keep the elevation difference itself in registers: left alone, the compiler re-derives it (and
      // the validity test) from the raw elevation in every step, three extra instructions per cell-step
      keep_in_register(delta2[q]);
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        pw2[k][q] = V::make(p_[k][0], p_[k][1]);
        if (NS > 1) wst2[k][q] = V::make(w_[k][0], w_[k][1]);
      }
      nx2[q] = V::make(x_[0], x_[1]);
      ny2[q] = V::make(y_[0], y_[1]);
      nz2[q] = V::make(n_[0], n_[1]);
#pragma unroll
      for (int m = 0; m < NM; ++m) {
        swe2[m][q] = V::make(s_[m][0], s_[m][1]);
        tic2[m][q] = V::make(t_[m][0], t_[m][1]);
        // 1 - albedo of the ice surface: the constant, or the blend of the bracketing maps (set below)
        om2[m][q] = V::splat(a.albedo_const ? (R)1 - m_alb_ice(m) : (R)0.5);
      }
    }
    // steepest slope of the patch, tan^2 (nx2, ny2 hold the gradient); with a safety factor it decides
    // per step whether the sun stands above every slope of the patch (analytic direct beam below)
    // (float32 only: float64 is short of registers -- the extra path costs it 7 % in spills)
    constexpr bool kAnalyticBeam = INSOL == kInsolComputed && sizeof(R) == 4;
    R patch_g2 = (R)0;
    if (kAnalyticBeam) {
#pragma unroll
      for (int q = 0; q < KP; ++q) {
        patch_g2 = fmax_(patch_g2, fmax_(sq_sum(nx2[q].lo(), ny2[q].lo()), sq_sum(nx2[q].hi(), ny2[q].hi())));
      }
      if (KT > K) {
        // a pass that walks the patch in parts decides for the WHOLE patch, like a plain run does: the two
        // forms of the direct beam differ in the last bits, and fused members must equal single runs
        const int prow0 = row0 - part * K;
        for (int i = 0; i < KT; ++i) {
          const int rowb = prow0 + i;
          if (rowb < a.band_rows && colx < a.cols && (i < part * K || i >= part * K + K)) {
            const size_t o = (size_t)rowb * a.pitch + colx;
            const R gx = a.nx[o], gy = a.ny[o];
            if (gx == gx) patch_g2 = fmax_(patch_g2, sq_sum(gx, gy));
          }
        }
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) patch_g2 = fmax_(patch_g2, __shfl_xor_sync(0xffffffffu, patch_g2, d));
      patch_g2 *= (R)1.00001;
    }
    keep_in_register(valid_bits);
    const bool patch_full = __all_sync(0xffffffffu, valid_bits == ((1u << K) - 1u));
    // sunlit masks of this patch (INSOL == kInsolMasked): word of its 32 columns, its K rows
    const unsigned lane_bit = 1u << lane;
    constexpr bool RING = ENRGY_MASK_RING && INSOL == kInsolMasked && K == 8;
    uint4* const ring = reinterpret_cast<uint4*>(smem_raw + plan.ring) + warp * kRingSlots * 2;   // [kRingSlots][2]
    int ring_next = -0x40000000;                    // next sub-step to fetch (not primed yet)
    const unsigned* const mask_patch =
        INSOL == kInsolMasked
            ? a.masks + ((size_t)(row0 >> 3) * a.mask_words + (size_t)((colx - lane) >> 5)) * 8 + (row0 & 7) -
                  (size_t)a.mask_sub0 * a.mask_sub_stride
            : nullptr;

    int buf = 0;
    if (tid == 0) issue_block(a.block_begin, 0);

    for (int b = a.block_begin; b < a.block_end; ++b, buf ^= 1) {
      if (tid == 0 && b + 1 < a.block_end) issue_block(b + 1, buf ^ 1);
      R* const sm_slots = sm_slots0 + (ONE_BAR ? (size_t)(slot_set & 1u) * W * cap_steps * NM * kStatsK : 0);
      slot_set ^= 1u;
      mbar_wait(&sm_full[buf], phase[buf]);
      phase[buf] ^= 1u;
      const TimeBlock tb = a.blocks[b];
      const int ts = max(tb.t_begin, a.t0), te = min(tb.t_end, a.t1);

      // streamed insolation: first step's values, then one step ahead
      float pot_next[K];
      if (INSOL == kInsolStreamed) {
#pragma unroll
        for (int i = 0; i < K; ++i) {
          const size_t o = (size_t)(ts - a.pot_t0) * a.pot_stride + (size_t)(row0 + i) * a.pitch + colx;
          pot_next[i] = (valid_bits >> i) & 1u ? __ldg(a.pot + o) : 0.f;
        }
      }

      // The step loop exists twice: for patches without off-glacier cells (no masking of the
      // statistics, so the whole balance of a step is one basic block the scheduler can interleave
      // freely: +3 %) and for patches with some.  (Reducing the statistics one step late, so that the
      // shuffle butterfly of step t - 1 overlapped the balance of step t, measured 1 % slower.)
      // Statistics batch: batch_n entries, the last of them entry `end - 1` of the block's slots, are parked in the warp's batch buffer.
      int batch_n = 0;
      auto flush_batch = [&](int end) {
        const int e0 = end - batch_n;
        __syncwarp();
        if constexpr (E > 0)
        batch_reduce<R, NQ, E, SB::kLwd>(smem_raw + batch_off, batch_n, lane, sm_slots + ((size_t)warp * cap_steps * NM + e0) * kStatsK,
                            sm_slots_m + ((size_t)warp * cap_steps + e0) * kStatsM);
        __syncwarp();                                  // read before the next entries overwrite them
        batch_n = 0;
      };
      auto run_steps = [&](auto full_tag) {
      constexpr bool FULL = decltype(full_tag)::value;
      // the codes that steer a step (sub-step range, albedo bracket and weight) are read one step
      // ahead, so that their shared-memory latency is off the path to the step's first branch
      const StepRec<R>* const steps_b = sm_steps + buf * cap_steps - tb.t_begin;
      int sub_next = step_code(steps_b[ts].sub), pair_next = step_code(steps_b[ts].alb_pair);
      R w_next = steps_b[ts].alb_w;
      for (int t = ts; t < te; ++t) {
        // a full batch is summed before the next step rather than at the end of the last one: there the
        // next step's records and the step's own temporaries are live, and the 32 loaded values spill
        if constexpr (E > 0 && NM <= E && INSOL != kInsolMasked) {
          if (batch_n + NM > E) flush_batch((t - tb.t_begin) * NM);
        }
        const StepRec<R> s = steps_b[t];
        const int sub_code = sub_next, pair = pair_next;
        const R alb_w = w_next;
        if (t + 1 < te) {
          sub_next = step_code(steps_b[t + 1].sub);
          pair_next = step_code(steps_b[t + 1].alb_pair);
          w_next = steps_b[t + 1].alb_w;
        }
        // ---- 1 - albedo of the ice surface from this step's bracket of maps (interpolator.py:12-18):
        // the blend weight counts whole days, so the blend is refreshed once a day from the two
        // maps (L2) instead of carrying both in registers and blending every step
        if (!a.albedo_const) {
          if (pair != cur_pair || alb_w != cur_w) {        // uniform across the CTA
            cur_pair = pair;
            cur_w = alb_w;
            const float* m0 = a.albedo + (size_t)(pair >> 8) * a.map_stride;
            const float* m1 = a.albedo + (size_t)(pair & 255) * a.map_stride;
#pragma unroll
            for (int q = 0; q < KP; ++q) {
              R om[NM][2];
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const int i = 2 * q + h;
                const size_t o = (size_t)(row0 + i) * a.pitch + colx;
                const bool v = (valid_bits >> i) & 1u;
                const R y0 = v ? (R)__ldg(m0 + o) : (R)0.5, y1 = v ? (R)__ldg(m1 + o) : (R)0.5;
#pragma unroll
                for (int m = 0; m < NM; ++m) {
                  // + ensemble offset, clipped like the loader clips a raster (identity for offset 0)
                  const R x0 = v ? fmin_(fmax_(y0 + m_offset(m), (R)0.001f), (R)1) : (R)0.5;
                  const R x1 = v ? fmin_(fmax_(y1 + m_offset(m), (R)0.001f), (R)1) : (R)0.5;
                  om[m][h] = ((R)1 - x0) + alb_w * (x0 - x1);
                }
              }
#pragma unroll
              for (int m = 0; m < NM; ++m) om2[m][q] = V::make(om[m][0], om[m][1]);
            }
          }
        }
        float pot_cur[K];
        if (INSOL == kInsolStreamed) {
#pragma unroll
          for (int i = 0; i < K; ++i) pot_cur[i] = pot_next[i];
          if (t + 1 < te) {
#pragma unroll
            for (int i = 0; i < K; ++i) {
              const size_t o = (size_t)(t + 1 - a.pot_t0) * a.pot_stride + (size_t)(row0 + i) * a.pitch + colx;
              pot_next[i] = (valid_bits >> i) & 1u ? __ldg(a.pot + o) : 0.f;
            }
          }
        }

        V pot2[KP];
        auto balance = [&]() {
        // ---- per-cell energy balance -------------------------------------------------------------
        const V zero2 = V::splat((R)0);
        V acc_sens = zero2, acc_lat = zero2;                 // member-invariant flux factors
        V acc_lwd = zero2;                                   // station blend: Tz^4 (no DEM-moment shortcut)
        V acc_rs[NM], acc_mf[NM], acc_snow[NM], acc_swe[NM], acc_lwu = zero2, acc_g = zero2;
        int n_snow[NM];
#pragma unroll
        for (int m = 0; m < NM; ++m) { acc_rs[m] = acc_mf[m] = acc_snow[m] = acc_swe[m] = zero2; n_snow[m] = 0; }
        // albedo of snow-covered cells: the aged value when ageing is on, else the blended map
        // (uniform per step): (1 - alb_snow) = (1 - alb) * keep_map + snow_const
        const V keep_map = V::splat(s.snow_alb >= (R)0 ? (R)0 : (R)1);
        const R ice_floor = (R)1 - a.max_ice_albedo;      // 1 - cap (-inf with constant albedo)
        const V t_aws = V::splat(s.t_air), lapse2 = V::splat(s.lapse), p_aws = V::splat(s.p_hpa), e_aws = V::splat(s.e_aws);
        const V c_lwd = V::splat(s.c_lwd), c_sw = V::splat(s.c_sw), c_melt = V::splat(s.c_melt);
        // per member: the exchange-coefficient scalars of the step (roughness lengths) and, with constant
        // albedo, the snow albedo
        V c_sens[NM], c_lat[NM], snow_const[NM];
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          if (NM > 1) {
            const MemberRec<R> mr = sm_members[(buf * cap_steps + (t - tb.t_begin)) * NM + m];
            c_sens[m] = V::splat(mr.c_sens);
            c_lat[m] = V::splat(mr.c_lat);
            const R sa = a.albedo_const ? a.member_albedo_snow[m] : s.snow_alb;
            snow_const[m] = V::splat(s.snow_alb >= (R)0 ? (R)1 - sa : (R)0);
          } else {
            c_sens[m] = V::splat(s.c_sens);
            c_lat[m] = V::splat(s.c_lat);
            snow_const[m] = V::splat(s.snow_alb >= (R)0 ? (R)1 - s.snow_alb : (R)0);
          }
        }
        const V k273 = V::splat((R)273.15), k_plapse = V::splat((R)kPressureLapse), k_rair = V::splat((R)kRair),
                k_fp0 = V::splat((R)1.0016), k_fp1 = V::splat((R)(3.15 * 1e-6)), k_fp2 = V::splat((R)-0.074);
#pragma unroll
        for (int q = 0; q < KP; ++q) {
          // lapse-rate distribution, var_classes.py:113-125.  float32 evaluates T + delta * lapse the
          // way NumPy float32 does (rounded product, rounded sum)
          // (the product is formed per cell with __fmul_rn: ptxas contracts a packed mul + add into FFMA2)
          // station blend: T, p at the cell = sum_k w_k (station value) + D * lapse, e = sum_k e_k V_k
          V t_st = t_aws, p_st = p_aws, e_st = zero2, cloud_fac = zero2;
          if (NS > 1) {
            const StationRec<R>* const sr = sm_stations + (buf * cap_steps + (t - tb.t_begin)) * NS;
            V cn = zero2;
#pragma unroll
            for (int k = 0; k < NS; ++k) {
              const StationRec<R> r = sr[k];
              // float32: the temperature blend mirrors NumPy's float32 sequence (rounded products, rounded
              // sums) -- one ulp of a Celsius value flips the rounding of the Kelvin value in 2 % of the
              // cells, and Tz - Ts carries that into the sensible flux.  ptxas contracts a packed mul + add,
              // so the products are formed per cell (lapse_product).
              if (k == 0) {
                t_st = sizeof(R) == 4 ? lapse_product(wst2[0][q], r.t) : mul2(wst2[0][q], V::splat(r.t));
                p_st = mul2(wst2[0][q], V::splat(r.p));
                e_st = mul2(pw2[0][q], V::splat(r.e));
              } else {
                t_st = sizeof(R) == 4 ? add2(t_st, lapse_product(wst2[k][q], r.t)) : fma2(wst2[k][q], V::splat(r.t), t_st);
                p_st = fma2(wst2[k][q], V::splat(r.p), p_st);
                e_st = fma2(pw2[k][q], V::splat(r.e), e_st);
                cn = k == 1 ? mul2(wst2[1][q], V::splat(r.cn)) : fma2(wst2[k][q], V::splat(r.cn), cn);
              }
            }
            // Beer-Lambert attenuation by the cloud field relative to the primary station
            if (a.cloud_on) {
              const V x = mul2(cn, V::splat(a.cloud_neg_k));
              cloud_fac = V::make(Num<R>::exp_(x.lo()), Num<R>::exp_(x.hi()));
            }
          }
          const V t_air = sizeof(R) == 4 ? add2(t_st, lapse_product(delta2[q], s.lapse)) : fma2(delta2[q], lapse2, t_st);
          const V tz = add2(t_air, k273);
          // surface temperature: 0 degC without the sub-surface model (SURVEY F9), else the top
          // boundary of the layer stack (model.py:207-210)
          V d_t = sub2(tz, k273);                            // Tz - Ts
          if (MSM) {
            R d[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int i = 2 * q + h;
              const R tzh = h ? tz.hi() : tz.lo();
              d[h] = tzh - (tl[i][0] + (R)273.15);
              if (sizeof(R) == 4) {
                // float32 + sub-surface model: the reference's surface temperature raster turns
                // float64 after the first tick, so its Tz - Ts is float32(Tz) - (t0 + 273.15) without
                // a Kelvin rounding of Ts.  tz - 273.15f is exact (same binade); the second constant
                // is float(273.15) - 273.15.
                d[h] = ((tzh - (R)273.15) + (R)-6.103515625e-06) - tl[i][0];
              }
            }
            d_t = V::make(d[0], d[1]);
          }
          const V p_hpa = fma2(delta2[q], k_plapse, p_st);
          const V e = NS > 1 ? e_st : mul2(pw2[0][q], e_aws);
          // bulk fluxes, turbo.py:140-196 with rho = P / (R Tz) and rho / P = 1 / (R Tz);
          // c_sens carries CH * Cp * uz * 100 (Pa per hPa), c_lat carries CE * uz * 0.622 * Lv
          V r_rt, r_p;                                      // 1 / (R Tz) and 1 / p_hpa
          {
            const V rt = mul2(tz, k_rair);
            if (sizeof(R) == 8) {
              // float64: one division serves both reciprocals (a DP division is ~20 instructions)
              const V den = mul2(rt, p_hpa);
              const V inv = V::make(Num<R>::rcp(den.lo()), Num<R>::rcp(den.hi()));
              r_rt = mul2(inv, p_hpa);
              r_p = mul2(inv, rt);
            } else {
              r_rt = V::make(Num<R>::rcp(rt.lo()), Num<R>::rcp(rt.hi()));
              r_p = V::make(Num<R>::rcp(p_hpa.lo()), Num<R>::rcp(p_hpa.hi()));
            }
          }
          // every flux is (per-step scalar) x (per-cell factor): the scalar rides the FMA chain of the
          // balance and scales the area sums afterwards (finalize_stats_kernel), the loop keeps the factor
          const V x_sens = mul2(p_hpa, mul2(r_rt, d_t));    // sens = c_sens * x_sens
          // saturation vapour pressure of the melting surface, turbo.py:368-379 with t = 0:
          // exp(0) = 1 exactly, so es = 611.2 * f(p).  ez = e_max * (e / e_max) = e (one rounding).
          const V f_p = fma2(r_p, k_fp2, fma2(p_hpa, k_fp1, k_fp0));
          V es_neg = V::splat((R)-611.2);
          if (MSM) {                                        // Magnus term of the surface, turbo.py:377
            R x[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const R t0 = tl[2 * q + h][0];
              x[h] = (R)-611.2 * Num<R>::exp_(((R)17.62 * t0) * Num<R>::rcp((R)243.12 + t0));
            }
            es_neg = V::make(x[0], x[1]);
          }
          const V x_lat = mul2(r_rt, fma2(es_neg, f_p, e)); // lat = c_lat * x_lat
          // longwave, model.py:533-545
          const V tzsq = mul2(tz, tz);
          const V tz4 = mul2(tzsq, tzsq);
          V lwu = V::splat(s.c_lwu);
          if (MSM) {
            R x[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const R t0 = tl[2 * q + h][0];
              if (sizeof(R) == 4) {
                // (273.15 + t0)^4 = 273.15^4 (1 + x)^4, x = t0 / 273.15: keeps the low bits of t0 that
                // a float32 Kelvin temperature would drop
                const R y = t0 * (R)(1.0 / 273.15);
                const R poly = (R)1 + y * ((R)4 + y * ((R)6 + y * ((R)4 + y)));
                x[h] = (s.c_lwu * (R)(273.15 * 273.15 * 273.15 * 273.15)) * poly;
              } else {
                const R ts_k = t0 + (R)273.15;
                const R ts2 = ts_k * ts_k;
                x[h] = s.c_lwu * (ts2 * ts2);
              }
            }
            lwu = V::make(x[0], x[1]);
          }
          // net longwave lwd - lwu.  The area sum of lwd is not reduced here: Tz is linear in the
          // elevation, so it follows from the first four moments of (dem - elev_aws), see
          // finalize_stats_kernel
          V rl;
          if (sizeof(R) == 4 && !MSM) {
            // float32: both terms are ~300 W m-2 and Tz^4 alone would cost 4e-5 W m-2 of rounding.
            // With the (rounded, as in the reference) Tz = K0 + d_t, K0 = float(273.15) and d_t exact:
            //   c_lwd Tz^4 - lwu = (c_lwd K0^4 - lwu) + c_lwd K0^4 ((1 + y)^4 - 1),  y = d_t / K0
            // -- a per-row scalar from the float64 pre-pass plus a term of at most ~30 W m-2.
            // (Horner / Estrin forms in d_t with four per-row coefficients measured 1-2 % slower: the
            // loop waits on dependent packed instructions, and the wider step record costs shared-memory loads)
            const V y = mul2(d_t, V::splat((R)(1.0 / (double)273.15f)));
            const V poly = mul2(y, fma2(y, fma2(y, add2(y, V::splat((R)4)), V::splat((R)6)), V::splat((R)4)));
            rl = fma2(V::splat(s.c_lw1), poly, V::splat(s.c_lw0));
          } else {
            const V lwu_neg = V::make(-lwu.lo(), -lwu.hi());
            rl = fma2(c_lwd, tz4, lwu_neg);
          }
          const bool v_lo = (valid_bits >> (2 * q)) & 1u, v_hi = (valid_bits >> (2 * q + 1)) & 1u;
          // statistics of the member-invariant factors.  Off-glacier cells of a visited patch carry finite
          // dummy values: they are zeroed before the packed adds, on patches that have any (warp-uniform test)
          if (STATS) {
            V m_sens = x_sens, m_lat = x_lat;
            if (!FULL) {
              m_sens = V::make(v_lo ? x_sens.lo() : (R)0, v_hi ? x_sens.hi() : (R)0);
              m_lat = V::make(v_lo ? x_lat.lo() : (R)0, v_hi ? x_lat.hi() : (R)0);
            }
            // (the first pair starts the sums: q is a compile-time constant of the unrolled loop)
            acc_sens = q == 0 ? m_sens : add2(acc_sens, m_sens);
            acc_lat = q == 0 ? m_lat : add2(acc_lat, m_lat);
            if (NS > 1) {
              const V m_lwd = FULL ? tz4 : V::make(v_lo ? tz4.lo() : (R)0, v_hi ? tz4.hi() : (R)0);
              acc_lwd = q == 0 ? m_lwd : add2(acc_lwd, m_lwd);
            }
          }
#pragma unroll
          for (int m = 0; m < NM; ++m) {
          // albedo, model.py:298-337, as 1 - albedo.  Maps: blend of the bracketing maps; snow cells
          // take the aged snow albedo when ageing is on; ice cells are capped.  Constant albedo rides
          // the same formula: om = 1 - ice, snow_alb = snow (so keep_map = 0), cap = +inf.
          const bool snow_lo = swe2[m][q].lo() > (R)0, snow_hi = swe2[m][q].hi() > (R)0;
          const V om_snow = fma2(om2[m][q], keep_map, snow_const[m]);
          const V oma = V::make(snow_lo ? om_snow.lo() : fmax_(om2[m][q].lo(), ice_floor),
                                snow_hi ? om_snow.hi() : fmax_(om2[m][q].hi(), ice_floor));
          // shortwave, model.py:483-497: rs = potential * c_sw * (1 - albedo)
          const V x_rs = (NS > 1 && a.cloud_on) ? mul2(mul2(pot2[q], cloud_fac), oma) : mul2(pot2[q], oma);
          // balance, clamp, melt partition: model.py:411, :434-438, msm.py:193-203
          // rs + lwd - lwu + sens + lat as one FMA chain
          const V atmo = fma2(c_lat[m], x_lat, fma2(c_sens[m], x_sens, fma2(c_sw, x_rs, rl)));
          V mf, gfl = V::splat((R)0);
          if (MSM) {
            // explicit conduction through the layer stack and the surface-layer melt gate,
            // msm.py:31-107 (snow depth = swe / snow_density, model.py:428)
            const MsmParams<R>& mp = a.msm;
            const R dt = s.dt, inv_dt = s.inv_dt;
            R mfh[2], gh[2], grad0[2], sd1[2];
            // Snow-free cells (the ablation zone for most of the season): the snow share of every layer is 0,
            // conductivity and density are those of ice exactly, and the surface layer of the pair runs
            // packed with per-run constants -- 8 packed operations instead of ~70 scalar ones.  Decided per
            // warp, and which cells share a warp depends on where a row band starts and ends: so this path
            // performs, operation for operation, the general path's arithmetic at a snow share of 0 (its
            // constants are that path's intermediates exactly, the reciprocal the same approximation),
            // and a cell's result does not depend on the decision.
            const bool bare = !__any_sync(0xffffffffu, snow_lo || snow_hi);
            if (bare) {
              const V t0v = V::make(tl[2 * q][0], tl[2 * q + 1][0]), t1v = V::make(tl[2 * q][1], tl[2 * q + 1][1]);
              const V grad = mul2(sub2(t1v, t0v), V::splat(mp.inv_d[0]));            // msm.py:18-28
              const V gv = mul2(grad, V::splat(mp.g0_ice));
              const V full = add2(atmo, gv);
              // melt gate: qm = full - q0, q0 = -t0 c rho d / dt (msm.py:88-93)
              const V gate = fma2(t0v, V::splat(mp.crd_ice * inv_dt), full);
              const V mfv = V::make(fmax_(gate.lo(), (R)0), fmax_(gate.hi(), (R)0));
              const V dlt = mul2(sub2(full, mfv), V::splat(Num<R>::rcp(mp.crd_ice)));
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const int i = 2 * q + h;
                const R d_h = h ? dlt.hi() : dlt.lo();
                grad0[h] = h ? grad.hi() : grad.lo();
                mfh[h] = h ? mfv.hi() : mfv.lo();
                gh[h] = h ? gv.hi() : gv.lo();
                sd1[h] = (R)0;
                if (sizeof(R) == 4) {
                  t0_acc[i] += (double)(d_h * dt);
                  tl[i][0] = (R)t0_acc[i];
                } else {
                  tl[i][0] = tl[i][0] + d_h * dt;
                }
              }
            } else {
              // surface layer, msm.py:80-101: the snow share of each cell sets conductivity and density;
              // the pair runs packed (19 packed + 10 scalar instructions instead of ~70 scalar ones)
              const V one2 = V::splat((R)1), d0_2 = V::splat(mp.d[0]), inv_d0 = V::splat(mp.inv_d[0]);
              const V t0v = V::make(tl[2 * q][0], tl[2 * q + 1][0]), t1v = V::make(tl[2 * q][1], tl[2 * q + 1][1]);
              const V sd = mul2(swe2[m][q], V::splat(mp.inv_snow_density));
              const V share = mul2(sd, inv_d0);
              const V ratio = V::make(sd.lo() > mp.d[0] ? (R)1 : share.lo(), sd.hi() > mp.d[0] ? (R)1 : share.hi());   // msm.py:63
              const V omr = sub2(one2, ratio);
              const V kap = fma2(ratio, V::splat(mp.k_snow), mul2(omr, V::splat(mp.k_ice)));
              const V rho = fma2(ratio, V::splat(mp.rho_snow), mul2(omr, V::splat(mp.rho_ice)));
              const V below = sub2(sd, d0_2);
              const V grad = mul2(sub2(t1v, t0v), inv_d0);                                              // msm.py:18-28
              const V c_ice2 = V::splat(mp.c_ice);
              // (association as in the snow-free path above: kap c rho is g0_ice, c rho d is crd_ice at no snow)
              const V gv = mul2(grad, mul2(mul2(kap, c_ice2), rho));
              const V full = add2(atmo, gv);
              const V crd = mul2(mul2(c_ice2, rho), d0_2);
              const V gate = fma2(t0v, mul2(crd, V::splat(inv_dt)), full);          // full - q0, q0 = -t0 c rho d / dt
              const V mfv = V::make(fmax_(gate.lo(), (R)0), fmax_(gate.hi(), (R)0));
              const V dlt = mul2(sub2(full, mfv), V::make(Num<R>::rcp(crd.lo()), Num<R>::rcp(crd.hi())));
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const int i = 2 * q + h;
                const R d_h = h ? dlt.hi() : dlt.lo();
                grad0[h] = h ? grad.hi() : grad.lo();
                mfh[h] = h ? mfv.hi() : mfv.lo();
                gh[h] = h ? gv.hi() : gv.lo();
                sd1[h] = fmax_(h ? below.hi() : below.lo(), (R)0);
                if (sizeof(R) == 4) {
                  t0_acc[i] += (double)(d_h * dt);
                  tl[i][0] = (R)t0_acc[i];
                } else {
                  tl[i][0] = tl[i][0] + d_h * dt;
                }
              }
            }
            // deeper layers, msm.py:103.  Snow that reaches below the surface layer is rare (it takes
            // swe / snow_density > d[0]): where no cell of the warp has any, conductivity is that of ice
            // in every deeper layer (ratio = 0 gives exactly k_ice) and the pair runs packed; the general
            // per-cell loop is the same arithmetic with the snow share carried along.
            if (bare || !__any_sync(0xffffffffu, sd1[0] > (R)0 || sd1[1] > (R)0)) {
              V gp = V::make(grad0[0], grad0[1]);
              V t_h = V::make(tl[2 * q][1], tl[2 * q + 1][1]);
              const V k_ice2 = V::splat(mp.k_ice), dt2 = V::splat(dt);
#pragma unroll
              for (int l = 1; l < kMaxLayers; ++l) {
                if (l < mp.layers) {
                  const V t_n = V::make(tl[2 * q][l + 1], tl[2 * q + 1][l + 1]);
                  const V inv_d2 = V::splat(mp.inv_d[l]);
                  const V grad = mul2(sub2(t_n, t_h), inv_d2);
                  const V dlt = mul2(mul2(k_ice2, sub2(grad, gp)), inv_d2);
                  const V t_new = fma2(dlt, dt2, t_h);
                  tl[2 * q][l] = t_new.lo();
                  tl[2 * q + 1][l] = t_new.hi();
                  gp = grad;
                  t_h = t_n;
                }
              }
            } else {
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const int i = 2 * q + h;
                R sd = sd1[h], grad_prev = grad0[h], t_next = tl[i][1];
#pragma unroll
                for (int l = 1; l < kMaxLayers; ++l) {
                  if (l < mp.layers) {
                    const R t_here = t_next;
                    t_next = tl[i][l + 1];
                    const R grad = (t_next - t_here) * mp.inv_d[l];
                    const R ratio = sd > mp.d[l] ? (R)1 : sd * mp.inv_d[l];
                    const R kap = ratio * mp.k_snow + ((R)1 - ratio) * mp.k_ice;
                    sd = fmax_(sd - mp.d[l], (R)0);
                    const R dlt = kap * (grad - grad_prev) * mp.inv_d[l];
                    grad_prev = grad;
                    tl[i][l] = fma(dlt, dt, t_here);              // (as the packed loop above)
                  }
                }
              }
            }
            mf = V::make(mfh[0], mfh[1]);
            gfl = V::make(gh[0], gh[1]);
          } else {
            mf = V::make(fmax_(atmo.lo(), (R)0), fmax_(atmo.hi(), (R)0));
          }
          const V we = mul2(mf, c_melt);
          const V snow = V::make(fmin_(we.lo(), swe2[m][q].lo()), fmin_(we.hi(), swe2[m][q].hi()));
          const V ice = sub2(we, snow);
          // statistics (off-glacier cells zeroed as above)
          if (STATS) {
          V m_rs = x_rs, m_mf = mf, m_lwu = lwu, m_g = gfl;
          if (!FULL) {
            m_rs = V::make(v_lo ? x_rs.lo() : (R)0, v_hi ? x_rs.hi() : (R)0);
            m_mf = V::make(v_lo ? mf.lo() : (R)0, v_hi ? mf.hi() : (R)0);
            if (MSM) {
              m_lwu = V::make(v_lo ? lwu.lo() : (R)0, v_hi ? lwu.hi() : (R)0);
              m_g = V::make(v_lo ? gfl.lo() : (R)0, v_hi ? gfl.hi() : (R)0);
            }
          }
          acc_rs[m] = q == 0 ? m_rs : add2(acc_rs[m], m_rs);
          acc_mf[m] = q == 0 ? m_mf : add2(acc_mf[m], m_mf);
          acc_snow[m] = q == 0 ? snow : add2(acc_snow[m], snow);        // masked cells: swe = 0 -> snow = 0
          acc_swe[m] = q == 0 ? swe2[m][q] : add2(acc_swe[m], swe2[m][q]);
          if (MSM) {
            acc_lwu = q == 0 ? m_lwu : add2(acc_lwu, m_lwu);
            acc_g = q == 0 ? m_g : add2(acc_g, m_g);
          }
          n_snow[m] += (snow_lo ? 1 : 0) + (snow_hi ? 1 : 0);
          }
          if (DUMP && a.dump != nullptr) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int i = 2 * q + h;
              if ((valid_bits >> i) & 1u) {
                R* d = a.dump + (size_t)(t - a.t0) * ENRGY_D_COUNT * a.dump_field_stride +
                       (size_t)(row0 + i) * a.pitch + colx;
                auto half = [&](const V& x) { return h ? x.hi() : x.lo(); };
                d[ENRGY_D_RS * a.dump_field_stride] = s.c_sw * half(x_rs);
                d[ENRGY_D_LWD * a.dump_field_stride] = s.c_lwd * half(tz4);
                d[ENRGY_D_LWU * a.dump_field_stride] = half(lwu);
                d[ENRGY_D_SENS * a.dump_field_stride] = s.c_sens * half(x_sens);
                d[ENRGY_D_LAT * a.dump_field_stride] = s.c_lat * half(x_lat);
                d[ENRGY_D_ATMO * a.dump_field_stride] = half(atmo);
                d[ENRGY_D_MELT * a.dump_field_stride] = half(mf);
                d[ENRGY_D_SNOW * a.dump_field_stride] = half(snow);
                d[ENRGY_D_ICE * a.dump_field_stride] = half(ice);
                d[ENRGY_D_ALBEDO * a.dump_field_stride] = (R)1 - half(oma);
                d[ENRGY_D_POT * a.dump_field_stride] = half(pot2[q]);
                d[ENRGY_D_G * a.dump_field_stride] = half(gfl);
              }
            }
          }
          // state update, model.py:258-261.  total_snow is not accumulated here: it equals
          // swe(start) - swe(end) and is added once in the epilogue.
          swe2[m][q] = sub2(swe2[m][q], snow);
          tic2[m][q] = add2(tic2[m][q], ice);
          }  // members
        }
        // ---- per-step statistics: one batch entry per member, summed over the warp per batch ----------
        if (!DUMP && STATS) {
          const R sum_sens = acc_sens.lo() + acc_sens.hi(), sum_lat = acc_lat.lo() + acc_lat.hi();
#pragma unroll
          for (int m = 0; m < NM; ++m) {
            R acc[kStatsP];                            // by slot column
            acc[K_RS] = acc_rs[m].lo() + acc_rs[m].hi();
            acc[K_LWD] = NS > 1 ? acc_lwd.lo() + acc_lwd.hi() : (R)0;
            acc[K_SENS] = sum_sens;
            acc[K_LAT] = sum_lat;
            acc[K_MELT] = acc_mf[m].lo() + acc_mf[m].hi();
            acc[K_SNOW] = acc_snow[m].lo() + acc_snow[m].hi();
            acc[K_SWE] = acc_swe[m].lo() + acc_swe[m].hi();
            acc[K_NSNOW] = (R)n_snow[m];
            if constexpr (MSM) {
              acc[kStatsK + M_LWU] = acc_lwu.lo() + acc_lwu.hi();
              acc[kStatsK + M_G] = acc_g.lo() + acc_g.hi();
            }
            if constexpr (E > 0) {
              R v[NQ];
#pragma unroll
              for (int q = 0; q < NQ; ++q) v[q] = acc[stat_column<SB::kLwd>(q)];
              batch_put<R, NQ>(smem_raw + batch_mine, batch_n, v);
              ++batch_n;
              if constexpr (NM > E || INSOL == kInsolMasked) {
                if (batch_n == E) flush_batch((t - tb.t_begin) * NM + m + 1);
              }
            } else {
              const R tot = warp_reduce8<R>(acc, lane);
              if ((lane & 3) == 0)
                sm_slots[((warp * cap_steps + (t - tb.t_begin)) * NM + m) * kStatsK + stat_of_lane(lane)] = tot;
              if constexpr (MSM) {
#pragma unroll
                for (int q = 0; q < kStatsM; ++q) {
                  R x = acc[kStatsK + q];
#pragma unroll
                  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
                  if (lane == 0) sm_slots_m[(warp * cap_steps + (t - tb.t_begin)) * kStatsM + q] = x;
                }
              }
            }
          }
        }
        };
        // ---- potential insolation of the step [kWh m-2] -----------------------------------------
        if (INSOL == kInsolStreamed) {
#pragma unroll
          for (int q = 0; q < KP; ++q) pot2[q] = V::make((R)pot_cur[2 * q], (R)pot_cur[2 * q + 1]);
          balance();
        } else {
          V direct2[KP];
#pragma unroll
          for (int q = 0; q < KP; ++q) direct2[q] = V::splat((R)0);
          auto finish_step = [&]() {
            // direct * nz + dsum * (1 + nz), two instructions
            const V dsum2 = V::splat(s.dsum);
#pragma unroll
            for (int q = 0; q < KP; ++q) pot2[q] = fma2(nz2[q], add2(direct2[q], dsum2), dsum2);
            balance();
          };
          const int j0 = sub_code >> 8, nj = sub_code & 255;
          auto sub_step = [&](int j) {
            const SubRec<R> sb = sm_subs[buf * cap_subs + j];
            const V e2 = V::splat(sb.e), n2 = V::splat(sb.n), u2 = V::splat(sb.u), b2 = V::splat(sb.b);
            // cos(incidence) / nz; nx2, ny2 hold nx/nz, ny/nz (terrain_kernel)
            V c2[KP];
#pragma unroll
            for (int q = 0; q < KP; ++q) c2[q] = fma2(ny2[q], n2, fma2(nx2[q], e2, u2));
            // sunlit bits of the patch's K rows for this sub-step: K consecutive words of the interleaved
            // mask layout [sub-step][row / 8][column word][row % 8] written by the line sweep (shade.cu);
            // the address is warp-uniform (one 32-byte sector per patch and sub-step), bit = lane
            unsigned mw[K];
            if (INSOL == kInsolMasked) {
              const unsigned* mp = mask_patch + (size_t)(tb.sub_begin + j) * a.mask_sub_stride;
              // the sector of the sub-step one row ahead goes to L1 now (no register, one lane)
              if (!RING && lane == 0) {
                const unsigned* ahead = mask_patch + (size_t)min(tb.sub_begin + j + kMaskAhead, a.mask_sub_last) * a.mask_sub_stride;
                asm volatile("prefetch.global.L1 [%0];" ::"l"(ahead));
              }
              if (RING) {
                const int ms = tb.sub_begin + j;
                auto fetch = [&](int x) {
                  if (lane < 2 && x <= a.mask_sub_last)
                    cp_async16(&ring[(x & (kRingSlots - 1)) * 2 + lane], mask_patch + (size_t)x * a.mask_sub_stride + 4 * lane);
                  cp_async_commit();
                };
                if (ms != ring_next - kRingAhead) {          // first sub-step of the tile (or a jump): prime the ring
                  cp_async_wait<0>();
                  __syncwarp();
#pragma unroll
                  for (int p_ = 0; p_ < kRingAhead; ++p_) fetch(ms + p_);
                  ring_next = ms + kRingAhead;
                }
                fetch(ring_next);
                ++ring_next;
                cp_async_wait<kRingAhead>();                 // the copy of sub-step ms has landed
                __syncwarp();
                const uint4 m0 = ring[(ms & (kRingSlots - 1)) * 2], m1 = ring[(ms & (kRingSlots - 1)) * 2 + 1];
                mw[0] = m0.x; mw[1] = m0.y; mw[2 % K] = m0.z; mw[3 % K] = m0.w;
                mw[4 % K] = m1.x; mw[5 % K] = m1.y; mw[6 % K] = m1.z; mw[7 % K] = m1.w;
              } else if (K == 8) {
                const uint4 m0 = __ldg(reinterpret_cast<const uint4*>(mp)), m1 = __ldg(reinterpret_cast<const uint4*>(mp) + 1);
                mw[0] = m0.x; mw[1] = m0.y; mw[2 % K] = m0.z; mw[3 % K] = m0.w;
                mw[4 % K] = m1.x; mw[5 % K] = m1.y; mw[6 % K] = m1.z; mw[7 % K] = m1.w;
              } else if (K == 4) {
                const uint4 m0 = __ldg(reinterpret_cast<const uint4*>(mp));
                mw[0] = m0.x; mw[1] = m0.y; mw[2 % K] = m0.z; mw[3 % K] = m0.w;
              } else {
                const uint2 m0 = __ldg(reinterpret_cast<const uint2*>(mp));
                mw[0] = m0.x; mw[1] = m0.y;
              }
            }
#pragma unroll
            for (int q = 0; q < KP; ++q) {
              R c_lo = fmax_(c2[q].lo(), (R)0), c_hi = fmax_(c2[q].hi(), (R)0);
              if (INSOL == kInsolMasked) {
                c_lo = (mw[2 * q] & lane_bit) ? c_lo : (R)0;
                c_hi = (mw[2 * q + 1] & lane_bit) ? c_hi : (R)0;
              }
              direct2[q] = fma2(b2, V::make(c_lo, c_hi), direct2[q]);
            }
          };
          // (sub-surface model: ONE copy of the balance per loop -- three of them, each with the layer
          // stack of every pair, made a step loop of 160 KB that no longer fitted the instruction caches:
          // ncu showed 2.5 warps per issue waiting for instructions)
          constexpr bool kOneBalance = MSM;
          // hourly rows carry four sunlit sub-steps by day.  That case is straight-line code followed by
          // its own copy of the balance, so that insolation and balance of a step form one basic block
          // (the records load ahead, the chains of consecutive sub-steps and the first reciprocals of
          // the balance interleave); every other count takes the loop.
          if (kAnalyticBeam && patch_g2 < s.tan2_min) {
            // the sun stands above every slope of the patch in every sub-step of the row:
            // max(cos i, 0) = cos i, and the sum over the sub-steps collapses to the row's three sums
            // (two packed FMAs per pair instead of three per pair and sub-step)
            const V du = V::splat(s.dir_u), de = V::splat(s.dir_e), dn = V::splat(s.dir_n);
#pragma unroll
            for (int q = 0; q < KP; ++q) direct2[q] = fma2(ny2[q], dn, fma2(nx2[q], de, du));
            if (!kOneBalance) finish_step();
          } else if (nj == 4) {
            sub_step(j0); sub_step(j0 + 1); sub_step(j0 + 2); sub_step(j0 + 3);
            if (!kOneBalance) finish_step();
          } else {
#pragma unroll(kSubUnroll)
            for (int j = j0; j < j0 + nj; ++j) sub_step(j);
            if (!kOneBalance) finish_step();
          }
          if (kOneBalance) finish_step();
        }
      }  // steps of the time block
      };
      if (patch_full) run_steps(std::true_type{}); else run_steps(std::false_type{});
      if (!DUMP && STATS && E > 0 && batch_n > 0) flush_batch((te - tb.t_begin) * NM);   // the block's last, partial batch

      // ---- flush the block's statistics into this CTA's partial rows (fixed order) ---------------
      __syncthreads();
      if (!DUMP && STATS && my_partials != nullptr) {
        // (fused members: a "step" of this loop is a (step, member) pair; rows are [step][member][kRow])
        constexpr int NQ = MSM ? kStatsP : kStatsK;
        const int n = (te - ts) * NM * NQ;
        for (int idx = tid; idx < n; idx += NT) {
          const int step = idx / NQ, q = idx - step * NQ;
          const int sl = (ts - tb.t_begin) * NM + step;
          if (NS == 1 && q == K_LWD) continue;         // (no station blend: the column is not summed here)
          double sum = 0.0;
#pragma unroll
          for (int w = 0; w < W; ++w) {
            sum += q < kStatsK ? (double)sm_slots[(w * cap_steps * NM + sl) * kStatsK + q]
                               : (double)sm_slots_m[(w * cap_steps + sl) * kStatsM + (q - kStatsK)];
          }
          my_partials[((size_t)(ts - a.t0) * NM + step) * kRow + q] += (R)sum;
        }
      }
      // (ONE_BAR: the next block fills the other set of slots and the other staging buffer; the barrier
      // at ITS end orders this flush before anything of this block is overwritten)
      if (!ONE_BAR) __syncthreads();
    }  // time blocks

    // ---- epilogue: state back to HBM (off-glacier cells become NaN, model.py:258) ---------------
    if (!DUMP) {
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const int rowb = row0 + i;
        if (rowb < a.band_rows && colx < a.cols) {
          const size_t o = (size_t)rowb * a.pitch + colx;
          const bool v = (valid_bits >> i) & 1u;
#pragma unroll
          for (int m = 0; m < NM; ++m) {
            const size_t om = m * m_stride + o;
            const R swe_i = (i & 1) ? swe2[m][i / 2].hi() : swe2[m][i / 2].lo();
            const R tic_i = (i & 1) ? tic2[m][i / 2].hi() : tic2[m][i / 2].lo();
            // total_snow grows by swe(start) - swe(end); the start value is still in HBM -- or, when a run
            // is cut into several launches (chunks of rows), in the copy taken at its start, and only the
            // last launch adds the difference: the result does not depend on the cuts
            const R swe_start = v ? (a.swe_ref ? a.swe_ref[om] : a.swe[om]) : (R)0;
            a.swe[om] = v ? swe_i : qnan;
            if (a.update_total_snow) a.total_snow[om] = v ? a.total_snow[om] + (swe_start - swe_i) : qnan;
            a.total_ice[om] = v ? tic_i : qnan;
          }
          if (MSM) {
#pragma unroll
            for (int l = 0; l < NB; ++l) {
              if (l <= a.msm.layers && v) a.layer_t[(size_t)l * a.layer_stride + o] = tl[i][l];
            }
          }
        }
      }
    }
  }  // tiles (and parts of their patches)
}

// cells per thread: the sub-surface model carries 8 more registers per cell
template <typename R, bool MSM>
struct CellsPerThread {
  static constexpr int kBase = sizeof(R) == 4 ? ENRGY_K32 : ENRGY_K64;
  static constexpr int value = MSM ? ((kBase / 2 + 1) & ~1) : kBase;   // an even number: cells come in pairs
};

template <typename R>
void energy_balance_tile(bool msm, int* tile_h, int* tile_w) {
  const int k = msm ? CellsPerThread<R, true>::value : CellsPerThread<R, false>::value;
  const int w = kWarpsFor<R, kInsolComputed>;
  *tile_w = 32 * warps_x(w);
  *tile_h = (w / warps_x(w)) * k;
}
template void energy_balance_tile<float>(bool, int*, int*);
template void energy_balance_tile<double>(bool, int*, int*);

// fused members and the station blend: half the cells per thread (their per-member state / station weights
// take the registers), the handle's tile list is walked in two parts -- but never less than one pair (the
// float64 sub-surface model already runs one pair, KT = 2)
template <typename R, bool MSM, int NM, int NS = 1>
struct PassShape {
  static constexpr int KT = CellsPerThread<R, MSM>::value;
  static constexpr int K = (NM > 1 || NS > 1) ? (KT / 2 > 2 ? KT / 2 : 2) : KT;
};

// a FusedVariant as template arguments
template <int INSOL, bool MSM, bool DUMP, int NM, bool STATS, int NS>
struct Instance {};

template <typename R, int INSOL, bool MSM, bool DUMP, int NM, bool STATS, int NS>
static cudaError_t configure(Instance<INSOL, MSM, DUMP, NM, STATS, NS>, int sm_count, int cap_steps, int cap_subs,
                             LaunchInfo* info) {
  constexpr int K = PassShape<R, MSM, NM, NS>::K, KT = PassShape<R, MSM, NM, NS>::KT;
  auto kern = energy_balance_kernel<R, K, INSOL, MSM, DUMP, NM, KT, STATS, NS>;
  const int smem = smem_plan<R>(kWarpsFor<R, INSOL>, cap_steps, cap_subs, INSOL != kInsolStreamed, MSM, NM, NS, INSOL == kInsolMasked,
                                StatBatchFor<R, INSOL, MSM, DUMP, NM, STATS, NS>::kBytes).total;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * kWarpsFor<R, INSOL>, smem);
  if (e != cudaSuccess) return e;
  cudaFuncAttributes fa;
  e = cudaFuncGetAttributes(&fa, kern);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  info->regs = fa.numRegs;
  info->smem_bytes = smem;
  info->ctas_per_sm = per_sm;
  info->grid = per_sm * sm_count;
  info->cells_per_thread = K;
  return cudaSuccess;
}

template <typename R, int INSOL, bool MSM, bool DUMP, int NM, bool STATS, int NS>
static cudaError_t launch_one(Instance<INSOL, MSM, DUMP, NM, STATS, NS> inst, const KernelArgs<R>& a, int sm_count,
                              int forced_grid, LaunchInfo* info, cudaStream_t stream) {
  constexpr int K = PassShape<R, MSM, NM, NS>::K, KT = PassShape<R, MSM, NM, NS>::KT;
  LaunchInfo li;
  cudaError_t e = configure<R>(inst, sm_count, a.cap_steps, a.cap_subs, &li);
  if (e != cudaSuccess) return e;
  int grid = forced_grid > 0 ? forced_grid : li.grid;
  li.grid = grid;
  if (info) *info = li;
  if (a.n_tiles == 0 || a.t1 <= a.t0) return cudaSuccess;
  energy_balance_kernel<R, K, INSOL, MSM, DUMP, NM, KT, STATS, NS><<<grid, 32 * kWarpsFor<R, INSOL>, li.smem_bytes, stream>>>(a);
  return cudaGetLastError();
}

// FusedVariant -> template instance; these are all the instances there are
template <typename F>
static cudaError_t dispatch(const FusedVariant& v, F&& f) {
#define ENRGY_CASE(I, M, D, N, S, NS)                                                       \
  if (v.insol == I && v.msm == M && v.dump == D && v.nm == N && v.stats == S && v.ns == NS) \
    return f(Instance<I, M, D, N, S, NS>{});
#define ENRGY_INSOLS(M, D, N, S, NS) ENRGY_CASE(0, M, D, N, S, NS) ENRGY_CASE(1, M, D, N, S, NS) ENRGY_CASE(2, M, D, N, S, NS)
  // plain: (insol, msm, dump)
  ENRGY_INSOLS(false, false, 1, true, 1) ENRGY_INSOLS(true, false, 1, true, 1)
  ENRGY_INSOLS(false, true, 1, true, 1) ENRGY_INSOLS(true, true, 1, true, 1)
  // station blend: (insol, msm, dump)
  ENRGY_INSOLS(false, false, 1, true, kMaxStations) ENRGY_INSOLS(false, true, 1, true, kMaxStations)
  ENRGY_INSOLS(true, false, 1, true, kMaxStations) ENRGY_INSOLS(true, true, 1, true, kMaxStations)
  // fused ensemble members: (insol, nm, stats)
  ENRGY_INSOLS(false, false, 2, true, 1) ENRGY_INSOLS(false, false, 4, true, 1)
  ENRGY_INSOLS(false, false, 2, false, 1) ENRGY_INSOLS(false, false, 4, false, 1)
#undef ENRGY_INSOLS
#undef ENRGY_CASE
  return cudaErrorInvalidValue;
}

template <typename R>
cudaError_t configure_energy_balance(const FusedVariant& v, int sm_count, int cap_steps, int cap_subs, LaunchInfo* info) {
  return dispatch(v, [&](auto inst) { return configure<R>(inst, sm_count, cap_steps, cap_subs, info); });
}
template cudaError_t configure_energy_balance<float>(const FusedVariant&, int, int, int, LaunchInfo*);
template cudaError_t configure_energy_balance<double>(const FusedVariant&, int, int, int, LaunchInfo*);

template <typename R>
cudaError_t launch_energy_balance(const KernelArgs<R>& a, const FusedVariant& v, int sm_count, int grid, LaunchInfo* info,
                                  cudaStream_t stream) {
  return dispatch(v, [&](auto inst) { return launch_one<R>(inst, a, sm_count, grid, info, stream); });
}
template cudaError_t launch_energy_balance<float>(const KernelArgs<float>&, const FusedVariant&, int, int, LaunchInfo*, cudaStream_t);
template cudaError_t launch_energy_balance<double>(const KernelArgs<double>&, const FusedVariant&, int, int, LaunchInfo*, cudaStream_t);

// glacier-wide means of the state rasters of fused members: block_out[(member * blocks + b) * 4 + {0..3}] =
// {sum swe, sum total_snow, sum total_ice, count} over the band's glacier cells (summed on the host in
// block order)
template <typename R>
__global__ void member_totals_kernel(const float* __restrict__ dem, int dem_pitch, int pitch, int band_row0, int band_rows,
                                     int cols, const R* __restrict__ swe, const R* __restrict__ tsn,
                                     const R* __restrict__ tic, size_t member_stride, double* __restrict__ block_out) {
  const int m = blockIdx.y;
  double acc[4] = {0, 0, 0, 0};
  const size_t n = (size_t)band_rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int rb = (int)(i / cols), c = (int)(i % cols);
    const float z = dem[(size_t)(rb + band_row0) * dem_pitch + c];
    if (z == z) {
      const size_t o = m * member_stride + (size_t)rb * pitch + c;
      acc[0] += (double)swe[o]; acc[1] += (double)tsn[o]; acc[2] += (double)tic[o]; acc[3] += 1.0;
    }
  }
  __shared__ double sh[4][kThreads];
  for (int q = 0; q < 4; ++q) sh[q][threadIdx.x] = acc[q];
  __syncthreads();
  for (int off = kThreads / 2; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) {
      for (int q = 0; q < 4; ++q) sh[q][threadIdx.x] += sh[q][threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    for (int q = 0; q < 4; ++q) block_out[((size_t)m * gridDim.x + blockIdx.x) * 4 + q] = sh[q][0];
  }
}
template <typename R>
cudaError_t launch_member_totals(const float* dem, int dem_pitch, int pitch, int band_row0, int band_rows, int cols,
                                 const R* swe, const R* tsn, const R* tic, size_t member_stride, int n_members,
                                 double* block_out, int blocks, cudaStream_t stream) {
  // grid.y = members (<= kMaxFusedMembers); the cells are a grid-stride loop, so no dimension grows with the raster
  member_totals_kernel<R><<<dim3(blocks, n_members), kThreads, 0, stream>>>(dem, dem_pitch, pitch, band_row0, band_rows, cols,
                                                                           swe, tsn, tic, member_stride, block_out);
  return cudaGetLastError();
}
template cudaError_t launch_member_totals<float>(const float*, int, int, int, int, int, const float*, const float*, const float*, size_t, int, double*, int, cudaStream_t);
template cudaError_t launch_member_totals<double>(const float*, int, int, int, int, int, const double*, const double*, const double*, size_t, int, double*, int, cudaStream_t);

// initial boundary temperatures of the sub-surface model, model.py:133-143
template <typename R>
__global__ void msm_init_kernel(const float* __restrict__ dem, int dem_pitch, int pitch, int band_row0,
                                int band_rows_pad, int n_bounds, const R* __restrict__ t_point, R elev,
                                R* __restrict__ layer_t, size_t layer_stride) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= pitch) return;
  const R qnan = (R)__int_as_float(0x7fc00000);
  for (int rb = blockIdx.y; rb < band_rows_pad; rb += gridDim.y) {
    const float z = dem[(size_t)(rb + band_row0) * dem_pitch + c];
    const size_t o = (size_t)rb * pitch + c;
    for (int l = 0; l < n_bounds; ++l) {
      R t = qnan;
      if (z == z) {
        // value + (dem - elev) * -0.006, rounded product and rounded sum like NumPy
        const R d = (R)z - elev;
        if (sizeof(R) == 4) {
          t = (R)__fadd_rn((float)t_point[l], __fmul_rn((float)d, -0.006f));
        } else {
          t = (R)__dadd_rn((double)t_point[l], __dmul_rn((double)d, -0.006));
        }
        if (t > (R)0) t = (R)0;             // ice temperature is limited by the melting point
      }
      layer_t[(size_t)l * layer_stride + o] = t;
    }
  }
}
template <typename R>
cudaError_t launch_msm_init(const float* dem, int dem_pitch, int pitch, int band_row0, int band_rows_pad,
                            int n_bounds, const double* t_point, double elev, R* layer_t, size_t layer_stride,
                            cudaStream_t stream) {
  R h[kMaxLayers + 1];
  for (int l = 0; l < n_bounds; ++l) h[l] = (R)t_point[l];
  R* d = nullptr;
  cudaError_t e = cudaMalloc((void**)&d, sizeof(h));
  if (e != cudaSuccess) return e;
  e = cudaMemcpyAsync(d, h, sizeof(R) * n_bounds, cudaMemcpyHostToDevice, stream);
  if (e == cudaSuccess) {
    dim3 grid((pitch + 255) / 256, grid_rows(band_rows_pad));
    msm_init_kernel<R><<<grid, 256, 0, stream>>>(dem, dem_pitch, pitch, band_row0, band_rows_pad, n_bounds, d,
                                                 (R)elev, layer_t, layer_stride);
    e = cudaGetLastError();
  }
  cudaStreamSynchronize(stream);
  cudaFree(d);
  return e;
}
template cudaError_t launch_msm_init<float>(const float*, int, int, int, int, int, const double*, double, float*, size_t, cudaStream_t);
template cudaError_t launch_msm_init<double>(const float*, int, int, int, int, int, const double*, double, double*, size_t, cudaStream_t);

// =================================================================================================
// micro-benchmarks: the pipe peaks the roofline is quoted against
// =================================================================================================
template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int iters, T a, T b) {
  T x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = (T)(threadIdx.x + i);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = x[i] * a + b;
    }
  }
  T s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += x[i];
  if (s == (T)-1.2345) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void __launch_bounds__(256) mufu_peak_kernel(float* out, int iters) {
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = 1.0f + threadIdx.x + i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
#pragma unroll
      for (int i = 0; i < 8; ++i) asm volatile("rcp.approx.ftz.f32 %0, %0;" : "+f"(x[i]));
    }
  }
  float s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += x[i];
  if (s == -1.2345f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void __launch_bounds__(256) lds_peak_kernel(float* out, int iters) {
  __shared__ float buf[4096];
  for (int i = threadIdx.x; i < 4096; i += 256) buf[i] = (float)i;
  __syncthreads();
  float s = 0;
  int idx = threadIdx.x;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 64; ++r) {
      s += buf[(idx + r * 32) & 4095];
    }
    idx += 1;
  }
  if (s == -1.2345f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
cudaError_t launch_microbench(int kind, int sm_count, int iters, void* scratch, double* ops_per_launch,
                              cudaStream_t stream) {
  const int grid = sm_count * 8;
  const double threads = (double)grid * 256;
  switch (kind) {
    case 0:
      fma_peak_kernel<float><<<grid, 256, 0, stream>>>((float*)scratch, iters, 1.0000001f, 1e-9f);
      *ops_per_launch = threads * iters * 64.0 * 2.0;
      break;
    case 1:
      fma_peak_kernel<double><<<grid, 256, 0, stream>>>((double*)scratch, iters, 1.0000001, 1e-9);
      *ops_per_launch = threads * iters * 64.0 * 2.0;
      break;
    case 2:
      mufu_peak_kernel<<<grid, 256, 0, stream>>>((float*)scratch, iters);
      *ops_per_launch = threads * iters * 64.0;
      break;
    default:
      lds_peak_kernel<<<grid, 256, 0, stream>>>((float*)scratch, iters);
      *ops_per_launch = threads * iters * 64.0;
      break;
  }
  return cudaGetLastError();
}

// =================================================================================================
// statistics: cross-CTA sum in fixed order + the derived columns
// =================================================================================================
__global__ void finalize_stats_kernel(const FinalizeArgs f) {
  // one warp per step: lane l adds the rows of CTAs l, l + 32, ... in that order, then the lanes are
  // added by a butterfly -- a fixed order, so the sums are reproducible run to run
  const int f32_mode = f.f32_mode;
  const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (t >= f.n_steps) return;
  double k[kStatsP];
  for (int q = 0; q < kStatsP; ++q) k[q] = 0.0;
  const int row = f.msm ? kStatsP : kStatsK;
  const int nm = f.nm > 1 ? f.nm : 1;                 // fused members: rows are [cta][step][member][row]
  for (int c = lane; c < f.n_ctas; c += 32) {
    const size_t o = (((size_t)c * f.n_steps + t) * nm + f.member) * row;
    if (f32_mode) {
      const float* p = static_cast<const float*>(f.partials) + o;
      for (int q = 0; q < row; ++q) k[q] += (double)p[q];
    } else {
      const double* p = static_cast<const double*>(f.partials) + o;
      for (int q = 0; q < row; ++q) k[q] += p[q];
    }
  }
#pragma unroll
  for (int q = 0; q < kStatsP; ++q) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) k[q] += __shfl_xor_sync(0xffffffffu, k[q], d);
  }
  if (lane != 0) return;
  const StepRec<double> s = f.steps64[f.t0 + t];
  const double lwu_cell = f32_mode ? (double)(float)s.c_lwu : s.c_lwu;
  const double c_melt = f32_mode ? (double)(float)s.c_melt : s.c_melt;
  // the kernel sums the per-cell factors of the fluxes; their per-step scalars come in here
  k[K_RS] *= f32_mode ? (double)(float)s.c_sw : s.c_sw;
  k[K_SENS] *= f32_mode ? (double)(float)s.c_sens : s.c_sens;
  k[K_LAT] *= f32_mode ? (double)(float)s.c_lat : s.c_lat;
  double* o = f.stats + (size_t)t * ENRGY_S_COUNT;
  const double lwu = f.msm ? k[kStatsK + M_LWU] : f.n_valid * lwu_cell;
  // sum over glacier cells of c_lwd * Tz^4 with Tz = a + g * delta: quartic in the moments of delta
  double lwd_sum;
  {
    const double a = f32_mode ? (double)(float)s.t_air + (double)273.15f : s.t_air + 273.15;
    const double g = f32_mode ? (double)(float)s.lapse : s.lapse;
    const double c_lwd = f32_mode ? (double)(float)s.c_lwd : s.c_lwd;
    const double a2 = a * a, g2 = g * g;
    lwd_sum = c_lwd * (a2 * a2 * f.mom[0] + 4.0 * a2 * a * g * f.mom[1] + 6.0 * a2 * g2 * f.mom[2] +
                       4.0 * a * g2 * g * f.mom[3] + g2 * g2 * f.mom[4]);
  }
  // (station blend: Tz is no polynomial of one variable any more; the kernel summed Tz^4 itself)
  k[K_LWD] = f.lwd_summed ? k[K_LWD] * (f32_mode ? (double)(float)s.c_lwd : s.c_lwd) : lwd_sum;
  o[ENRGY_S_RS] = k[K_RS];
  o[ENRGY_S_LWD] = k[K_LWD];
  o[ENRGY_S_LWU] = lwu;
  o[ENRGY_S_SENS] = k[K_SENS];
  o[ENRGY_S_LAT] = k[K_LAT];
  // linear in the cell values: sum(atmo) = sum(rs) + sum(lwd) - sum(lwu) + sum(sens) + sum(lat)
  o[ENRGY_S_ATMO] = k[K_RS] + k[K_LWD] - lwu + k[K_SENS] + k[K_LAT];
  o[ENRGY_S_G] = f.msm ? k[kStatsK + M_G] : 0.0;
  o[ENRGY_S_MELT] = k[K_MELT];
  o[ENRGY_S_SNOW] = k[K_SNOW];
  // ice = we - snow with we = mf * c_melt
  o[ENRGY_S_ICE] = k[K_MELT] * c_melt - k[K_SNOW];
  o[ENRGY_S_SWE] = k[K_SWE];
  o[ENRGY_S_NSNOW] = k[K_NSNOW];
  o[ENRGY_S_NSWE] = f.n_valid;
  o[ENRGY_S_NVALID] = f.n_valid;
  if (f.override_first && f.t0 + t == 0) {
    o[ENRGY_S_SWE] = f.swe0_sum;
    o[ENRGY_S_NSNOW] = f.swe0_nsnow;
    o[ENRGY_S_NSWE] = f.swe0_nvalid;
  }
}

cudaError_t launch_finalize(const FinalizeArgs& f, cudaStream_t stream) {
  if (f.n_steps <= 0) return cudaSuccess;
  // four steps (warps) per block; a 1-D grid over the steps, independent of the raster size
  finalize_stats_kernel<<<(f.n_steps + 3) / 4, 128, 0, stream>>>(f);
  return cudaGetLastError();
}

}  // namespace enrgy
