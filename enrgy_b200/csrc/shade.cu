// Topographic shading as a line sweep (sm_100a).
//
// Replaces the shadow part of `saga_cmd ta_lighting 2 ... -SHADOW 1` (reference saga_lighting.py:42-44;
// SAGA itself is an external binary, so the specification is this repo's: oracle/insolation_oracle.py,
// "shadow").  All rays of one sub-step share one direction, so the raster is cut into sheared scan
// lines and "is some cell toward the sun above my ray" becomes, per line, a running maximum of
//     g = dem - u * dz          (u = position along the sweep axis, dz = rise of the rays per step)
// swept from the sunward edge: lit = !(M > g); M = max(M, g).  One pass over the terrain per
// sub-step, O(H*W) whatever the relief -- the per-cell ray march it replaces cost O(ray length) per
// cell (profiles/r01_summary.md: 750 instructions per cell-step on rough relief).
//
// Mapping: a THREAD owns V lines (l = Lw + 32 v + lane), their running maxima live in registers as
// float64 (u * dz is exact in float64 and g one correctly rounded subtraction, as in the oracle, so the
// mask is the same on any hardware: DESIGN.md section 5); a WARP owns the
// 32 V consecutive lines of its window and walks the rows from the sunward edge; the rows of the
// terrain are read with coalesced (unaligned) 128-byte loads from a scan copy of the DEM with -inf
// aprons (no bounds checks); the Q warps of a CTA sweep the same window for Q sub-steps of similar
// direction, so they share the terrain rows through L1.  Every row yields V ballots; funnel shifts
// align them to 32-column words (V - 1 full words per window: windows overlap by one word).
// Row-type sub-steps write the fused kernel's mask layout directly; column-type sub-steps sweep the
// transposed copy into a temporary whose 32 x 32 bit blocks transpose_kernel turns around.
#include "kernels.cuh"

#include <cstdio>

#ifndef ENRGY_SWEEP_PIPE
#define ENRGY_SWEEP_PIPE 1
#endif

namespace enrgy {

namespace {

__device__ __forceinline__ long long floor_div(long long a, long long b) {
  long long q = a / b;
  if ((a % b != 0) && ((a < 0) != (b < 0))) --q;
  return q;
}
__device__ __forceinline__ long long ceil_div(long long a, long long b) { return -floor_div(-a, b); }

// ---- scan copies ---------------------------------------------------------------------------------
// scan[(r + RA) * pitch_s + CA + c] = dem(r, c) or -inf; everything else -inf
__global__ void scan_fill_kernel(const float* __restrict__ src, int src_pitch, int rows, int cols,
                                 float* __restrict__ scan, int pitch_s, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int rr = (int)(i / pitch_s) - kScanRowApron, cc = (int)(i % pitch_s) - kScanColApron;
    float v = -INFINITY;
    if (rr >= 0 && rr < rows && cc >= 0 && cc < cols) {
      const float z = src[(size_t)rr * src_pitch + cc];
      if (z == z) v = z;
    }
    scan[i] = v;
  }
}
// interior of the transposed copy: scan_t[(c + RA) * pitch_t + CA + r] = scan(r, c), through a smem tile
__global__ void scan_transpose_kernel(const float* __restrict__ src, int src_pitch, int rows, int cols,
                                      float* __restrict__ scan_t, int pitch_t) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32;
  for (int r0 = blockIdx.y * 32; r0 < rows; r0 += gridDim.y * 32) {
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int r = r0 + i, c = c0 + threadIdx.x;
      float v = -INFINITY;
      if (r < rows && c < cols) {
        const float z = src[(size_t)r * src_pitch + c];
        if (z == z) v = z;
      }
      tile[i][threadIdx.x] = v;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int c = c0 + i, r = r0 + threadIdx.x;
      if (c < cols && r < rows) scan_t[(size_t)(c + kScanRowApron) * pitch_t + kScanColApron + r] = tile[threadIdx.x][i];
    }
    __syncthreads();                    // the tile is refilled by the next block of rows
  }
}

// ---- the sweep -----------------------------------------------------------------------------------
template <bool ROW, int V, int U, int Q>
__global__ void __launch_bounds__(32 * Q) sweep_kernel(const SweepArgs a) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_subs = ROW ? a.n_row_subs : a.n_col_subs;
  const int si = blockIdx.y * Q + warp;
  if (si >= n_subs) return;
  const SweepSub s = (ROW ? a.row_subs : a.col_subs)[si];
  const int na = ROW ? a.rows : a.cols;            // cells along the sweep axis
  const int nb = ROW ? a.cols : a.rows;            // cells across
  const int pitch = (nb + 31) / 32 * 32 + 2 * kScanColApron;
  const float* __restrict__ H = ROW ? a.scan : a.scan_t;
  // u = sigma * (index along the sweep axis) grows toward the sun; the sweep runs from u_hi down
  const int u_hi = s.sigma > 0 ? na - 1 : 0, u_lo = s.sigma > 0 ? 0 : -(na - 1);
  const int sh_max = max(shear_q16(u_lo, s.dfix), shear_q16(u_hi, s.dfix));
  // this warp's lines [Lw, Lw + 32 V): at u they sit over the cells [Lw + sh(u), Lw + sh(u) + 32 V)
  const int Lw = -sh_max + 32 * (V - 1) * (int)blockIdx.x;
  // u range over which that window touches the grid (sh is monotone in u)
  int ua = u_lo, ub = u_hi;
  {
    const long long x1 = -(long long)Lw - 32 * V + 1, x2 = (long long)nb - 1 - Lw;   // x1 <= sh(u) <= x2
    const long long y1 = x1 * 65536 - 32768, y2 = (x2 + 1) * 65536 - 32768 - 1;      // y1 <= u * dfix <= y2
    if (s.dfix > 0) {
      ua = (int)max((long long)ua, ceil_div(y1, s.dfix));
      ub = (int)min((long long)ub, floor_div(y2, s.dfix));
    } else if (s.dfix < 0) {
      ub = (int)min((long long)ub, floor_div(y1, s.dfix));
      ua = (int)max((long long)ua, ceil_div(y2, s.dfix));
    } else if (!(x1 <= 0 && 0 <= x2)) {
      return;
    }
  }
  if (ROW) {
    // rows behind the last row anybody asked for (seen from the sun) need no sweep
    int er0 = a.seg[0].row0, er1 = a.seg[0].row0 + a.seg[0].rows;
    for (int q = 1; q < a.n_seg; ++q) {
      er0 = min(er0, a.seg[q].row0);
      er1 = max(er1, a.seg[q].row0 + a.seg[q].rows);
    }
    ua = s.sigma > 0 ? max(ua, er0) : max(ua, -(er1 - 1));
  }
  if (ua > ub) return;

  double M[V];
#pragma unroll
  for (int v = 0; v < V; ++v) M[v] = -INFINITY;
  const double dz = s.dz;
  const int words_needed = (nb + 31) >> 5;

  // U rows per iteration; the loads of the NEXT iteration are issued before the current one is worked
  // on (two register buffers, the loop body exists twice), so a warp hides a full iteration of memory
  // latency by itself.  Rows past ua are inside the -inf aprons or harmless (nothing is emitted).
  // The rows are loaded in the order u = ub, ub - 1, ub - 2, ...: their shears shear_q16(u, dfix) come from
  // a running 64-bit accumulator q = u * dfix + 32768 (sh = q >> 16), one 64-bit subtraction per row
  // instead of a 64-bit product (|u * dfix| reaches 2^36 on rasters of 2^20 cells a side).
  long long q = (long long)ub * s.dfix + 32768;
  auto load_rows = [&](int u0, float (&h)[U][V], int (&col0)[U]) {
#pragma unroll
    for (int i = 0; i < U; ++i) {
      const int u = u0 - i;
      col0[i] = Lw + (int)(q >> 16);
      q -= s.dfix;
      const float* rowp = H + (long long)(s.sigma * u) * pitch + (col0[i] + lane);
#pragma unroll
      for (int v = 0; v < V; ++v) h[i][v] = __ldg(rowp + 32 * v);
    }
  };
  // Emission.  The V ballots of a row cover the cells col0 .. col0 + 32 V - 1; the words aligned to 32
  // cells start o = -col0 mod 32 bits in, so word j is a funnel shift of ballots j and j + 1 (V - 1 full
  // words per row).  Emitting row by row kept 25 of the 32 lanes idle through ~35 instructions per row (a
  // third of the kernel's instructions) and stored single 4-byte words 32 bytes apart.  Instead the
  // ballots and shears of the 8 rows of a ROW GROUP are parked in shared memory (every lane writes the
  // same words), and when the sweep leaves the group all 32 lanes emit it at once: lane = (word column c,
  // row pair), two funnel shifts each, one 8-byte store -- the four lanes of a column fill one 32-byte
  // sector of the row-interleaved mask layout, the eight columns of a warp 256 contiguous bytes.
  __shared__ __align__(16) unsigned s_bal[Q][8][V];
  __shared__ int s_col0[Q][8];
  unsigned (*bal)[V] = s_bal[warp];
  int* const colv = s_col0[warp];
  int cur_group = -1;                  // row group (index >> 3 along the sweep axis) being collected
  unsigned present = 0;                // its rows seen so far
  const int cidx = lane & 7, rp = lane >> 3;
  auto flush = [&]() {
    __syncwarp();
    if (present != 0u) {
      // smallest first word column of the group's rows (they differ by at most one: the shear moves the
      // window by less than a cell per row)
      const int c_l = colv[cidx];
      const int base_l = ((present >> cidx) & 1u) ? ((c_l + ((-c_l) & 31)) >> 5) : 0x7fffffff;
      const int cmin = __reduce_min_sync(full, base_l);
      const int c = cmin + cidx;
      unsigned w2[2];
      bool ok[2];
#pragma unroll
      for (int z = 0; z < 2; ++z) {
        const int rr = 2 * rp + z;
        const int c0 = colv[rr];
        const int o = (-c0) & 31;
        const int j = c - ((c0 + o) >> 5);
        ok[z] = ((present >> rr) & 1u) && j >= 0 && j <= V - 2 && (unsigned)c < (unsigned)words_needed;
        const int jj = min(max(j, 0), V - 2);
        w2[z] = __funnelshift_r(bal[rr][jj], bal[rr][jj + 1], o);
      }
      const int first = cur_group << 3;                // first row (row type) / column (column type) of the group
      if (ROW) {
        // destination segment of the group (band starts are multiples of 8 rows)
        unsigned* out = nullptr;
        for (int q = 0; q < a.n_seg; ++q) {
          if (first >= a.seg[q].row0 && first < a.seg[q].row0 + a.seg[q].rows)
            out = a.seg[q].ptr + ((size_t)s.out * a.seg[q].rg + ((first - a.seg[q].row0) >> 3)) * a.seg[q].words * 8;
        }
        if (out != nullptr) {
          unsigned* p = out + ((size_t)c << 3) + 2 * rp;
          if (ok[0] && ok[1]) *reinterpret_cast<uint2*>(p) = make_uint2(w2[0], w2[1]);
          else if (ok[0]) p[0] = w2[0];
          else if (ok[1]) p[1] = w2[1];
        }
      } else {
        unsigned* out = a.tmp + (size_t)s.out * a.cols * a.tmp_words;
#pragma unroll
        for (int z = 0; z < 2; ++z)
          if (ok[z]) out[(size_t)(first + 2 * rp + z) * a.tmp_words + c] = w2[z];
      }
    }
    __syncwarp();
  };
  auto process = [&](int u0, const float (&h)[U][V], const int (&col0)[U]) {
#pragma unroll
    for (int i = 0; i < U; ++i) {
      const int u = u0 - i;
      const double udz = (double)u * dz;
      unsigned B[V];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const double g = (double)h[i][v] - udz;
        const bool shaded = M[v] > g;
        M[v] = shaded ? M[v] : g;
        B[v] = __ballot_sync(full, !shaded);
      }
      if (u >= ua) {                                   // (warp-uniform)
        const int idx = s.sigma * u;                   // row (row type) / column (column type), >= 0
        if ((idx >> 3) != cur_group) {
          flush();
          cur_group = idx >> 3;
          present = 0;
        }
        const int pos = idx & 7;
        if (V % 4 == 0) {
#pragma unroll
          for (int v = 0; v < V; v += 4) *reinterpret_cast<uint4*>(&bal[pos][v]) = make_uint4(B[v], B[v + 1], B[(v + 2) % V], B[(v + 3) % V]);
        } else {
#pragma unroll
          for (int v = 0; v < V; ++v) bal[pos][v] = B[v];
        }
        colv[pos] = col0[i];
        present |= 1u << pos;
      }
    }
  };
#if ENRGY_SWEEP_PIPE
  {
    float ha[U][V], hb[U][V];
    int ca[U], cb[U];
    load_rows(ub, ha, ca);
    for (int u0 = ub; u0 >= ua; u0 -= 2 * U) {
      const bool more = u0 - U >= ua;
      if (more) load_rows(u0 - U, hb, cb);
      process(u0, ha, ca);
      if (!more) break;
      if (u0 - 2 * U >= ua) load_rows(u0 - 2 * U, ha, ca);
      process(u0 - U, hb, cb);
    }
  }
#else
  for (int u0 = ub; u0 >= ua; u0 -= U) {
    float h[U][V];
    int col0[U];
    load_rows(u0, h, col0);
    process(u0, h, col0);
  }
#endif
  flush();                                             // the last row group
}

// ---- 32 x 32 bit blocks of the column-type temporaries turned around --------------------------------
// tmp[sub][c][rw] (bit = row % 32) -> destination layout (bit = column % 32).  A warp takes 32 columns
// (one destination column word) x 256 rows: lane = column, two 16-byte loads, eight butterfly transposes.
__global__ void __launch_bounds__(128) transpose_kernel(const SweepArgs a) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int cw = blockIdx.x;                                   // destination column word
  const int rb = blockIdx.y * 4 + (threadIdx.x >> 5);          // block of 8 row words = 256 rows
  if (rb * 8 >= a.tmp_words) return;
  const SweepSub s = a.col_subs[blockIdx.z];
  const int c = cw * 32 + lane;
  unsigned x[8];
  if (c < a.cols) {
    const uint4* p = reinterpret_cast<const uint4*>(a.tmp + ((size_t)s.out * a.cols + c) * a.tmp_words + rb * 8);
    const uint4 p0 = __ldg(p), p1 = __ldg(p + 1);
    x[0] = p0.x; x[1] = p0.y; x[2] = p0.z; x[3] = p0.w; x[4] = p1.x; x[5] = p1.y; x[6] = p1.z; x[7] = p1.w;
  } else {
#pragma unroll
    for (int q = 0; q < 8; ++q) x[q] = 0xffffffffu;
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    unsigned v = x[q];
    // recursive block swap: after the stage with distance d, 2d x 2d blocks are transposed
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned lowmask = d == 1 ? 0x55555555u : d == 2 ? 0x33333333u : d == 4 ? 0x0f0f0f0fu : d == 8 ? 0x00ff00ffu : 0x0000ffffu;
      const unsigned y = __shfl_xor_sync(full, v, d);
      v = (lane & d) ? ((v & ~lowmask) | ((y & ~lowmask) >> d)) : ((v & lowmask) | ((y & lowmask) << d));
    }
    // lane j now holds the word of row 32 (8 rb + q) + j over the columns 32 cw .. 32 cw + 31
    const int row = (rb * 8 + q) * 32 + lane;
    if (row < a.rows) {
      for (int g = 0; g < a.n_seg; ++g) {
        const SweepSeg sg = a.seg[g];
        if (row >= sg.row0 && row < sg.row0 + sg.rows) {
          const int local = row - sg.row0;
          sg.ptr[(((size_t)s.out2 * sg.rg + (local >> 3)) * sg.words + cw) * 8 + (local & 7)] = v;
        }
      }
    }
  }
}

#ifndef ENRGY_SWEEP_V
#define ENRGY_SWEEP_V 8
#endif
#ifndef ENRGY_SWEEP_U
#define ENRGY_SWEEP_U 2
#endif
#ifndef ENRGY_SWEEP_Q
#define ENRGY_SWEEP_Q 4
#endif

}  // namespace

cudaError_t launch_scan_prepare(const float* src, int src_pitch, int rows, int cols, float* scan, float* scan_t,
                                cudaStream_t stream) {
  const int ps = scan_pitch(cols), pt = scan_pitch(rows);
  const size_t ns = scan_elems(rows, cols), nt = scan_elems(cols, rows);
  scan_fill_kernel<<<1184, 256, 0, stream>>>(src, src_pitch, rows, cols, scan, ps, ns);
  // the transposed copy: aprons by the same fill (no source), interior by the tile transpose
  scan_fill_kernel<<<1184, 256, 0, stream>>>(src, src_pitch, 0, 0, scan_t, pt, nt);
  scan_transpose_kernel<<<dim3((cols + 31) / 32, grid_rows((rows + 31) / 32)), dim3(32, 8), 0, stream>>>(
      src, src_pitch, rows, cols, scan_t, pt);
  return cudaGetLastError();
}

cudaError_t launch_sweep(const SweepArgs& a, int sm_count, cudaStream_t stream, int* n_launches) {
  (void)sm_count;
  constexpr int V = ENRGY_SWEEP_V, U = ENRGY_SWEEP_U, Q = ENRGY_SWEEP_Q;
  static_assert(U <= kScanRowApron && 32 * V + 32 <= kScanColApron, "aprons of the scan copy");
  static_assert((long long)Q * 65535 >= kSweepMaxRowSubs, "grid.y of the sweep");
  int n = 0;
  // line groups: windows of 32 V lines every 32 (V - 1) lines over [-sh_max, nb - sh_min); the shear
  // spans at most the length of the sweep axis (|dfix| <= 65536).  grid.x is under 2^21 / 224 + 4 for
  // rasters of up to 2^20 cells a side (the x limit is 2^31 - 1); grid.y counts sub-steps only
  // (kSweepMaxRowSubs); the transpose's grid.y = tmp_words / 32 <= 2^20 / 1024 and its grid.z counts
  // sub-steps (kSweepMaxColSubs).
  auto groups = [&](int na, int nb) { return (nb + na + 32 * V) / (32 * (V - 1)) + 2; };
  if (a.n_row_subs > 0) {
    dim3 grid(groups(a.rows, a.cols), (a.n_row_subs + Q - 1) / Q);
    sweep_kernel<true, V, U, Q><<<grid, 32 * Q, 0, stream>>>(a);
    ++n;
  }
  if (a.n_col_subs > 0) {
    dim3 grid(groups(a.cols, a.rows), (a.n_col_subs + Q - 1) / Q);
    sweep_kernel<false, V, U, Q><<<grid, 32 * Q, 0, stream>>>(a);
    dim3 tg((a.cols + 31) / 32, (a.tmp_words / 8 + 3) / 4, a.n_col_subs);
    transpose_kernel<<<tg, 128, 0, stream>>>(a);
    n += 2;
  }
  if (n_launches) *n_launches = n;
  return cudaGetLastError();
}

}  // namespace enrgy
