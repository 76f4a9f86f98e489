// Non-local means, exact replay of the reference's accumulation order.
//
// Reference: src/pixel/nlmeans_core.c  nlmeans_denoise :315-532 (scatter :95-104, define_patches :107-145,
// pixel_difference :156-165, diff_of_pixels_diff :168-180, init_column_sums :214-264,
// compute_slice_height/width :267-312), dt_fast_mexp2f math/math.h:290-301; callers
// iop/denoiseprofile.c process_nlmeans_cpu :1599-1648 (nlmeans_norm :1456-1470, nlmeans_scattering
// :1474-1499, nlmeans_precondition :1500-1533, nlmeans_backtransform :1580-1597).
//
// The reference's result is order dependent: per ~60x72 chunk and per patch offset, patch distances are
// float running column sums updated incrementally down the rows, and a float running sum along each row;
// contributions are accumulated into the output in patch order.  Bit parity therefore fixes three
// sequential axes.  Mapping: one CTA per reference chunk, patches in order, and per patch
//   phase E  all threads       : e_c(r,col) = (in[r][col].c - in[r+dy][col+dx].c)^2 for the chunk + halo rows/cols,
//                                three planes in shared memory -- every global load of the patch happens here,
//                                fully parallel, so the two serial phases below never wait on memory
//   phase A  threads = columns : the column-sum recurrence down the rows, from E        -> S[row][col] (shared)
//   phase B1 threads = rows    : the running sum along each row                          -> D[row][col] (in place of S)
//   phase B2 threads = pixels  : weights and accumulation; each thread owns a fixed set of chunk pixels and keeps
//                                their RGBA sums in registers across all patches
// and the phases of successive patches are software-pipelined (see nlm_chunks_kernel).
// pixel_difference() is (d0*d0)*n0 + (d1*d1)*n1 + (d2*d2)*n2 and diff_of_pixels_diff() is
// (a0*a0 - b0*b0)*n0 + ...: both are functions of the per-channel squares, so E holds exactly the reference's
// intermediate values and the sums are formed in its order.
// Not HBM bound by construction (SURVEY.md 8d: ~9 kflop/px at K=7); reported against FP32 issue.
#ifndef B200_KERNELS_ON_CPU // tests/emul compiles the group kernel's phases with g++ to check them against the oracle without a GPU
#include "runtime.h"
#include <atomic>
#include <math_constants.h>
#endif
#include <math.h>
#include <stdlib.h>
#include "packed_f32.cuh"

namespace
{
constexpr int SLICE_WIDTH = 72, SLICE_HEIGHT = 60; // nlmeans_core.c:55-56
constexpr int MAX_RADIUS = 4;                      // patch radius 1..4 (:35)
constexpr int MAX_CH = SLICE_HEIGHT + 9;           // compute_slice_height() returns 51..69
constexpr int MAX_CW = SLICE_WIDTH;
constexpr int SW = MAX_CW + 2 * MAX_RADIUS + 2;    // 82 columns of column sums, +1 -> odd stride below
constexpr int SSTRIDE = SW + 1;                    // 83: odd, so lanes = rows hit distinct banks
#ifndef NLM_NT
#define NLM_NT 512
#endif
#ifndef NLM_MINB
#define NLM_MINB 1
#endif
constexpr int NT = NLM_NT;

struct patch_t
{
  short rows, cols;
};

// C's (int)float on the reference's hardware is cvttss2si: the "integer indefinite" 0x80000000 for a NaN and for anything
// beyond the int range, where the device's conversion saturates (and turns a NaN into 0)
__device__ __forceinline__ int cvtt_x86(float v)
{
#ifdef B200_KERNELS_ON_CPU
  return (int)v;
#else
  return (fabsf(v) < 2147483648.0f) ? __float2int_rz(v) : (int)0x80000000;
#endif
}
__device__ __forceinline__ float fast_mexp2(float x) // math/math.h:290-301
{
  const int i1 = 0x3f800000, i2 = 0x3f000000;
  const int k0 = (int)((unsigned)i1 + (unsigned)cvtt_x86(x * (float)(i2 - i1))); // the sum wraps like the reference's two's-complement add
  return __int_as_float(k0 >= 0x800000 ? k0 : 0);
}
#ifndef B200_KERNELS_ON_CPU
struct nlm_args_t
{
  const float4 *in;
  float4 *out;
  const patch_t *patches;
  int n_patches;
  int width, height, chk_h, chk_w, n_cl;
  int radius;
  float center_weight, sharpness, cp_norm;
  float norm[4];
  float weight[4], invert[4];
  int skip_blend;
  int rows_e, plane_e; // rows of one E plane (chunk rows + 2*radius + 1), floats per plane (rows_e * SW)
  int cols_w, sstride_w; // window variant: columns of a window row, odd pitch of its sum planes
};

__device__ __forceinline__ float pixdiff(const float4 a, const float4 b, const float *n) // :156-165
{
  const float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z;
  return d0 * d0 * n[0] + d1 * d1 * n[1] + d2 * d2 * n[2];
}
__device__ __forceinline__ float diff_of_diffs(const float4 p1, const float4 p2, const float4 p3, const float4 p4, const float *n) // :168-180
{
  const float a0 = p1.x - p2.x, a1 = p1.y - p2.y, a2 = p1.z - p2.z;
  const float b0 = p3.x - p4.x, b1 = p3.y - p4.y, b2 = p3.z - p4.z;
  return (a0 * a0 - b0 * b0) * n[0] + (a1 * a1 - b1 * b1) * n[1] + (a2 * a2 - b2 * b2) * n[2];
}

// patch geometry of nlmeans_denoise() :345-372 for one chunk; uniform across the CTA
struct patch_geo_t
{
  int srow, scol, row_min, row_max, row_top, row_bot, col_min, col_max, pcol_min, pcol_max;
  long long poff;
  bool valid;
};
__device__ __forceinline__ patch_geo_t patch_geo(const nlm_args_t &a, int p, int chunk_top, int chunk_bot, int chunk_left, int chunk_right)
{
  patch_geo_t g;
  g.valid = p >= 0 && p < a.n_patches;
  if(!g.valid) return g;
  const int radius = a.radius, width = a.width, height = a.height;
  g.srow = a.patches[p].rows;
  g.scol = a.patches[p].cols;
  g.row_min = max(chunk_top, max(0, -g.srow));
  g.row_max = min(chunk_bot, height - max(0, g.srow));
  g.valid = g.row_min < g.row_max;
  g.row_top = max(g.row_min, max(radius, radius - g.srow));
  g.row_bot = min(g.row_max, height - 1 - max(radius, radius + g.srow));
  g.col_min = max(chunk_left, -g.scol);
  g.col_max = min(chunk_right, width - g.scol);
  g.pcol_min = chunk_left - min(radius, min(chunk_left, chunk_left + g.scol));
  g.pcol_max = chunk_right + min(radius, min(width - chunk_right, width - (chunk_right + g.scol)));
  g.poff = (long long)g.srow * width + g.scol;
  return g;
}

// Software pipeline over the patches, two __syncthreads per patch.  Warps 0..2 ("serial") own the two recurrences,
// the other warps ("parallel") own every global load and the accumulation:
//     interval 1:  serial A(i)   -- column sums of patch i from E[i&1] into S[i&1]     | parallel B2(i-1) from S[(i-1)&1]
//     interval 2:  serial B1(i)  -- distortions of patch i, in place in S[i&1]          | parallel E(i+1) into E[(i+1)&1]
// so the recurrences (3 busy warps) run under the latency-bound parallel phases instead of between them.
constexpr int SERIAL_T = 96;                       // >= SW columns and >= MAX_CH rows
constexpr int PNT = NT - SERIAL_T;                 // parallel threads
constexpr int OWNP = (MAX_CH * MAX_CW + PNT - 1) / PNT;
static_assert(SERIAL_T >= SW && SERIAL_T >= MAX_CH, "serial warps must cover one row and one column of a chunk");

__global__ void __launch_bounds__(NT, NLM_MINB) nlm_chunks_kernel(const __grid_constant__ nlm_args_t a)
{
  extern __shared__ __align__(16) float smem[];
  float *const Ebuf = smem;                                    // 2 x 3 planes [rows_e][SW]
  float *const Sbuf = smem + 6 * a.plane_e;                    // 2 x [chunk rows][SSTRIDE]
  const int tid = threadIdx.x;
  const bool serial = tid < SERIAL_T;
  const int ptid = tid - SERIAL_T;                             // index among the parallel threads
  const int it = blockIdx.x / a.n_cl, il = blockIdx.x - it * a.n_cl;
  const int chunk_top = it * a.chk_h, chunk_left = il * a.chk_w;
  const int chunk_bot = min(chunk_top + a.chk_h, a.height), chunk_right = min(chunk_left + a.chk_w, a.width);
  const int width = a.width, height = a.height, radius = a.radius;
  const int cbase = chunk_left - radius - 1;              // column of S[.][0] and E[.][0]
  const int ncols = (chunk_right + radius) - cbase;       // <= SW
  const int s_plane = a.chk_h * SSTRIDE;
  const float4 *const in = a.in;
  const float n0 = a.norm[0], n1 = a.norm[1], n2 = a.norm[2];

  // the pixels a parallel thread owns: pixel ptid + k*PNT of the chunk, row-major
  const int cw = chunk_right - chunk_left, ch = chunk_bot - chunk_top;
  float4 acc[OWNP];
  int own[OWNP]; // (image row << 16) | image column, or -1 (frames < 32768 px a side)
#pragma unroll
  for(int k = 0; k < OWNP; k++)
  {
    acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int idx = ptid + k * PNT;
    const int rr = idx / cw;
    own[k] = (!serial && rr < ch) ? (((chunk_top + rr) << 16) | (chunk_left + (idx - rr * cw))) : -1;
  }
  // phase E walks (row, col) entries ptid, ptid+PNT, ... of an ncols-wide grid without dividing in the loop
  const int e_r0 = ptid / ncols, e_c0 = ptid - e_r0 * ncols, e_dr = PNT / ncols, e_dc = PNT - e_dr * ncols;

  // ---- phase E: squared per-channel differences of every pixel pair the patch touches (parallel threads) --------
  auto phase_e = [&](int p) {
    const patch_geo_t g = patch_geo(a, p, chunk_top, chunk_bot, chunk_left, chunk_right);
    if(!g.valid) return;
    float *const E0 = Ebuf + (p & 1) * 3 * a.plane_e, *const E1 = E0 + a.plane_e, *const E2 = E1 + a.plane_e;
    const int erow0 = g.row_min - radius;                         // image row of E[0][.]
    const int n_erows = (g.row_max - g.row_min) + 2 * radius + 1; // rows row_min-radius .. row_max+radius
    int rr = e_r0, cc = e_c0;
    while(rr < n_erows)
    {
      const int r = erow0 + rr, col = cbase + cc;
      if(col >= g.pcol_min && col < g.pcol_max && r >= 0 && r < height && r + g.srow >= 0 && r + g.srow < height)
      {
        const float4 *px = in + (size_t)r * width + col;
        const float4 x = __ldg(px), y = __ldg(px + g.poff);
        const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z;
        const int e = rr * SW + cc;
        E0[e] = d0 * d0;
        E1[e] = d1 * d1;
        E2[e] = d2 * d2;
      }
      rr += e_dr;
      cc += e_dc;
      if(cc >= ncols)
      {
        cc -= ncols;
        rr++;
      }
    }
  };
  // ---- phase A: column sums down the rows, one serial thread per column ----------------------------------------
  auto phase_a = [&](int p) {
    const patch_geo_t g = patch_geo(a, p, chunk_top, chunk_bot, chunk_left, chunk_right);
    if(!g.valid || tid >= ncols) return;
    const float *const E0 = Ebuf + (p & 1) * 3 * a.plane_e, *const E1 = E0 + a.plane_e, *const E2 = E1 + a.plane_e;
    float *const S = Sbuf + (p & 1) * s_plane;
    const int erow0 = g.row_min - radius;
    const int col = cbase + tid;
    const bool live = col >= g.pcol_min && col < g.pcol_max;
    float cs = 0.0f;
    if(live)
    { // init_column_sums(), :214-264, at row = row_min
      const int row = g.row_min;
      const int rmin = row - min(radius, min(row, row + g.srow));
      const int rmax = row + min(radius, min(height - 1 - row, height - 1 - (row + g.srow)));
      float sum = 0.0f;
      for(int r = rmin; r <= rmax; r++)
      {
        const int e = (r - erow0) * SW + tid;
        sum += E0[e] * n0 + E1[e] * n1 + E2[e] * n2; // pixel_difference(), :156-165
      }
      cs = sum;
    }
    // Rows [row_min, lim_a) add the entering row (:424-440), [lim_a, row_bot) add entering minus leaving (:441-466),
    // rows >= max(row_top, row_bot) with a successor subtract the leaving row (:467-483).  All three are the middle
    // formula with the absent row's squares replaced by +0 (x - 0 = x, and -(u+v+w) is formed by the same roundings
    // as (-u)+(-v)+(-w)), so the loop is branch-free.
    const int lim_a = min(g.row_top, g.row_bot);
    int eb = (g.row_min + 1 + radius - erow0) * SW + tid, et = (g.row_min - radius - erow0) * SW + tid;
    float *sp = S + tid;
    for(int row = g.row_min; row < g.row_max; row++, eb += SW, et += SW, sp += SSTRIDE)
    {
      const bool use_b = live && row < g.row_bot;
      const bool use_t = live && row >= lim_a && (row < g.row_bot || (row >= g.row_top && row + 1 < g.row_max));
      const float b0 = use_b ? E0[eb] : 0.0f, b1 = use_b ? E1[eb] : 0.0f, b2 = use_b ? E2[eb] : 0.0f;
      const float t0 = use_t ? E0[et] : 0.0f, t1 = use_t ? E1[et] : 0.0f, t2 = use_t ? E2[et] : 0.0f;
      *sp = cs;
      cs += (b0 - t0) * n0 + (b1 - t1) * n1 + (b2 - t2) * n2;
    }
  };
  // ---- phase B1: running distortion along each row, one serial thread per row (:384-387,409) --------------------
  auto phase_b1 = [&](int p) {
    const patch_geo_t g = patch_geo(a, p, chunk_top, chunk_bot, chunk_left, chunk_right);
    if(!g.valid || tid >= g.row_max - g.row_min || g.col_min >= g.col_max) return;
    float *const Sr = Sbuf + (p & 1) * s_plane + tid * SSTRIDE - cbase; // Sr[col] = column sum of `col` for this row
    float distortion = 0.0f;
    for(int i = g.col_min - radius; i < min(g.col_min + radius, g.col_max); i++) distortion += Sr[i];
    for(int col = g.col_min; col < g.col_max; col++)
    {
      distortion += (Sr[col + radius] - Sr[col - radius - 1]);
      Sr[col - radius - 1] = distortion; // that slot is never read again: keep D[col] there
    }
  };
  // ---- phase B2: weights and accumulation into the owned pixels' registers (parallel threads) -------------------
  auto phase_b2 = [&](int p) {
    const patch_geo_t g = patch_geo(a, p, chunk_top, chunk_bot, chunk_left, chunk_right);
    if(!g.valid || g.col_min >= g.col_max) return;
    const float *const S = Sbuf + (p & 1) * s_plane;
#pragma unroll
    for(int k = 0; k < OWNP; k++)
    {
      const int row = own[k] >> 16, col = own[k] & 0xffff;
      if(own[k] < 0 || row < g.row_min || row >= g.row_max || col < g.col_min || col >= g.col_max) continue;
      const float4 *px = in + (size_t)row * width + col;
      const float4 q = __ldg(px + g.poff);
      const float dist = S[(row - g.row_min) * SSTRIDE + (col - radius - 1 - cbase)];
      float wt;
      if(a.center_weight < 0)
        wt = fast_mexp2(dist * a.sharpness); // :389-402
      else
      { // :404-420
        const float4 c = __ldg(px);
        const float d0 = c.x - q.x, d1 = c.y - q.y, d2 = c.z - q.z;
        const float pd = d0 * d0 * a.cp_norm + d1 * d1 * a.cp_norm + d2 * d2 * a.cp_norm;
        const float dissimilarity = (dist + pd) / (1.0f + a.center_weight);
        wt = fast_mexp2(fmaxf(0.0f, dissimilarity * a.sharpness - 2.0f));
      }
      acc[k].x += q.x * wt;
      acc[k].y += q.y * wt;
      acc[k].z += q.z * wt;
      acc[k].w += 1.0f * wt;
    }
  };

  if(!serial) phase_e(0);
  __syncthreads();
  for(int i = 0; i <= a.n_patches; i++)
  {
    if(serial)
      phase_a(i);
    else
      phase_b2(i - 1);
    __syncthreads();
    if(serial)
      phase_b1(i);
    else
      phase_e(i + 1);
    __syncthreads();
  }

  // ---- normalise (and blend) : :485-519 ---------------------------------------------------------------
#pragma unroll
  for(int k = 0; k < OWNP; k++)
  {
    if(own[k] < 0) continue;
    const float4 v = acc[k];
    const size_t g = (size_t)(own[k] >> 16) * width + (own[k] & 0xffff);
    float4 o;
    if(a.skip_blend)
      o = make_float4(v.x / v.w, v.y / v.w, v.z / v.w, v.w / v.w);
    else
    {
      const float4 i4 = __ldg(in + g);
      o.x = (i4.x * a.invert[0]) + (v.x / v.w * a.weight[0]);
      o.y = (i4.y * a.invert[1]) + (v.y / v.w * a.weight[1]);
      o.z = (i4.z * a.invert[2]) + (v.z / v.w * a.weight[2]);
      o.w = (i4.w * a.invert[3]) + (v.w / v.w * a.weight[3]);
    }
    a.out[g] = o;
  }
}

// ---- window variant: the chunk's own pixels (+halo) and the patch-shifted pixels both live in shared memory ------
// Per chunk the unshifted window P is loaded once; per patch only the shifted window Q is fetched (cp.async, every
// load of the patch in flight at once).  Everything else is shared-memory work:
//   U  (all threads)      U[row][col] = the column-sum update of that row (the branch-free form above)
//   A  (threads = columns) exclusive running sum of U down the rows, in place            -> column sums
//   V  (all threads)      V[row][col] = colsum[col+radius] - colsum[col-radius-1]
//   B1 (threads = rows)   inclusive running sum of V along the row, in place             -> distortions
//   B2 (all threads)      weights from the distortions, shifted pixels from Q, accumulation in registers
// so the two recurrences that fix the reference's float rounding order shrink to one add per element.
// Needs both windows in shared memory (radius <= 2 at the usual chunk sizes); selected with B200_NLM_WINDOW=1.
#ifndef NLM_WNT
#define NLM_WNT 512
#endif
constexpr int WNT = NLM_WNT;
constexpr int WOWN = (MAX_CH * MAX_CW + WNT - 1) / WNT;

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src)
{
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float pair_pd(const float4 x, const float4 y, float n0, float n1, float n2)
{ // pixel_difference(), :156-165
  const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z;
  return d0 * d0 * n0 + d1 * d1 * n1 + d2 * d2 * n2;
}

__global__ void __launch_bounds__(WNT, 1) nlm_chunks_win_kernel(const __grid_constant__ nlm_args_t a)
{
  extern __shared__ __align__(16) float smem[];
  const int colsw = a.cols_w, ss = a.sstride_w;
  float4 *const Pw = reinterpret_cast<float4 *>(smem);          // [rows_e][colsw] unshifted pixels
  float4 *const Qw = Pw + a.rows_e * colsw;                     // [rows_e][colsw] pixels at the patch offset
  float *const S = reinterpret_cast<float *>(Qw + a.rows_e * colsw); // [chunk rows][ss] U, then column sums
  float *const S2 = S + a.chk_h * ss;                           // [chunk rows][ss] V, then distortions
  const int tid = threadIdx.x;
  const int it = blockIdx.x / a.n_cl, il = blockIdx.x - it * a.n_cl;
  const int chunk_top = it * a.chk_h, chunk_left = il * a.chk_w;
  const int chunk_bot = min(chunk_top + a.chk_h, a.height), chunk_right = min(chunk_left + a.chk_w, a.width);
  const int width = a.width, height = a.height, radius = a.radius;
  const int cbase = chunk_left - radius - 1;              // image column of window column 0
  const int ncols = (chunk_right + radius) - cbase;       // <= colsw
  const int wrow0 = chunk_top - radius;                   // image row of window row 0
  const int nwrows = (chunk_bot - chunk_top) + 2 * radius + 1;
  const float4 *const in = a.in;
  const float n0 = a.norm[0], n1 = a.norm[1], n2 = a.norm[2];

  const int cw = chunk_right - chunk_left, ch = chunk_bot - chunk_top;
  float4 acc[WOWN];
  int own[WOWN]; // (chunk-local row << 16) | chunk-local column, or -1
#pragma unroll
  for(int k = 0; k < WOWN; k++)
  {
    acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int idx = tid + k * WNT;
    const int rr = idx / cw;
    own[k] = rr < ch ? ((rr << 16) | (idx - rr * cw)) : -1;
  }
  // entries tid, tid+WNT, ... of an ncols-wide grid, walked without dividing
  const int e_r0 = tid / ncols, e_c0 = tid - e_r0 * ncols, e_dr = WNT / ncols, e_dc = WNT - e_dr * ncols;

  // ---- the unshifted window, once per chunk ----------------------------------------------------------------
  for(int rr = e_r0, cc = e_c0; rr < nwrows;)
  {
    const int r = wrow0 + rr, col = cbase + cc;
    if(r >= 0 && r < height && col >= 0 && col < width) cp_async16(Pw + rr * colsw + cc, in + (size_t)r * width + col);
    rr += e_dr;
    cc += e_dc;
    if(cc >= ncols)
    {
      cc -= ncols;
      rr++;
    }
  }

  for(int p = 0; p < a.n_patches; p++)
  {
    const int srow = a.patches[p].rows, scol = a.patches[p].cols;
    const int row_min = max(chunk_top, max(0, -srow)), row_max = min(chunk_bot, height - max(0, srow));
    if(row_min >= row_max) continue; // uniform
    const int row_top = max(row_min, max(radius, radius - srow));
    const int row_bot = min(row_max, height - 1 - max(radius, radius + srow));
    const int col_min = max(chunk_left, -scol), col_max = min(chunk_right, width - scol);
    const int pcol_min = chunk_left - min(radius, min(chunk_left, chunk_left + scol));
    const int pcol_max = chunk_right + min(radius, min(width - chunk_right, width - (chunk_right + scol)));
    const long long poff = (long long)srow * width + scol;
    const int nrows = row_max - row_min;
    const int lim_a = min(row_top, row_bot);

    // ---- Q: the shifted window (the only global traffic of the patch) ------------------------------------
    for(int rr = e_r0, cc = e_c0; rr < nwrows;)
    {
      const int r = wrow0 + rr, col = cbase + cc;
      if(r >= 0 && r < height && r + srow >= 0 && r + srow < height && col >= 0 && col + scol >= 0 && col < width && col + scol < width)
        cp_async16(Qw + rr * colsw + cc, in + (size_t)r * width + col + poff);
      rr += e_dr;
      cc += e_dc;
      if(cc >= ncols)
      {
        cc -= ncols;
        rr++;
      }
    }
    cp_async_wait_all();
    __syncthreads();

    // ---- U: per-row update of every column sum ---------------------------------------------------------
    for(int rr = e_r0, cc = e_c0; rr < nrows;)
    {
      const int row = row_min + rr, col = cbase + cc;
      const bool live = col >= pcol_min && col < pcol_max;
      const bool use_b = live && row < row_bot;
      const bool use_t = live && row >= lim_a && (row < row_bot || (row >= row_top && row + 1 < row_max));
      float b0 = 0.f, b1 = 0.f, b2 = 0.f, t0 = 0.f, t1 = 0.f, t2 = 0.f;
      if(use_b)
      {
        const int w = (row + 1 + radius - wrow0) * colsw + cc;
        const float4 x = Pw[w], y = Qw[w];
        const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z;
        b0 = d0 * d0;
        b1 = d1 * d1;
        b2 = d2 * d2;
      }
      if(use_t)
      {
        const int w = (row - radius - wrow0) * colsw + cc;
        const float4 x = Pw[w], y = Qw[w];
        const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z;
        t0 = d0 * d0;
        t1 = d1 * d1;
        t2 = d2 * d2;
      }
      S[rr * ss + cc] = (b0 - t0) * n0 + (b1 - t1) * n1 + (b2 - t2) * n2;
      rr += e_dr;
      cc += e_dc;
      if(cc >= ncols)
      {
        cc -= ncols;
        rr++;
      }
    }
    __syncthreads();

    // ---- A: column sums = init_column_sums() at row_min, then the running sum of U down the rows --------
    if(tid < ncols)
    {
      const int col = cbase + tid;
      float cs = 0.0f;
      if(col >= pcol_min && col < pcol_max)
      { // :214-264
        const int row = row_min;
        const int rmin = row - min(radius, min(row, row + srow));
        const int rmax = row + min(radius, min(height - 1 - row, height - 1 - (row + srow)));
        float sum = 0.0f;
        for(int r = rmin; r <= rmax; r++)
        {
          const int w = (r - wrow0) * colsw + tid;
          sum += pair_pd(Pw[w], Qw[w], n0, n1, n2);
        }
        cs = sum;
      }
      float *sp = S + tid;
      constexpr int UW = 8; // updates fetched ahead of the running sum
      for(int rr0 = 0; rr0 < nrows; rr0 += UW, sp += UW * ss)
      {
        float u[UW];
#pragma unroll
        for(int k = 0; k < UW; k++) u[k] = (rr0 + k < nrows) ? sp[k * ss] : 0.0f;
#pragma unroll
        for(int k = 0; k < UW; k++)
          if(rr0 + k < nrows)
          {
            sp[k * ss] = cs;
            cs += u[k];
          }
      }
    }
    __syncthreads();

    // ---- V: what each step of the row recurrence adds (:409) --------------------------------------------
    {
      const int nc = col_max - col_min;
      if(nc > 0)
      {
        const int v_r0 = tid / nc, v_c0 = tid - v_r0 * nc, v_dr = WNT / nc, v_dc = WNT - v_dr * nc;
        for(int rr = v_r0, cc = v_c0; rr < nrows;)
        {
          const int k = col_min + cc - cbase;
          S2[rr * ss + k] = S[rr * ss + k + radius] - S[rr * ss + k - radius - 1];
          rr += v_dr;
          cc += v_dc;
          if(cc >= nc)
          {
            cc -= nc;
            rr++;
          }
        }
      }
    }
    __syncthreads();

    // ---- B1: running distortion along each row, one thread per row (:384-387,409) -----------------------
    if(tid < nrows && col_min < col_max)
    {
      const float *const Sr = S + tid * ss - cbase;
      float *const Vr = S2 + tid * ss - cbase;
      float distortion = 0.0f;
      for(int i = col_min - radius; i < min(col_min + radius, col_max); i++) distortion += Sr[i];
      constexpr int UW = 8;
      for(int col0 = col_min; col0 < col_max; col0 += UW)
      {
        float v[UW];
#pragma unroll
        for(int k = 0; k < UW; k++) v[k] = (col0 + k < col_max) ? Vr[col0 + k] : 0.0f;
#pragma unroll
        for(int k = 0; k < UW; k++)
          if(col0 + k < col_max)
          {
            distortion += v[k];
            Vr[col0 + k] = distortion;
          }
      }
    }
    __syncthreads();

    // ---- B2: weights and accumulation into the owned pixels' registers ------------------------------------
    if(col_min < col_max)
    {
#pragma unroll
      for(int k = 0; k < WOWN; k++)
      {
        const int row = chunk_top + (own[k] >> 16), col = chunk_left + (own[k] & 0xffff);
        if(own[k] < 0 || row < row_min || row >= row_max || col < col_min || col >= col_max) continue;
        const int w = (row - wrow0) * colsw + (col - cbase);
        const float4 q = Qw[w];
        const float dist = S2[(row - row_min) * ss + (col - cbase)];
        float wt;
        if(a.center_weight < 0)
          wt = fast_mexp2(dist * a.sharpness); // :389-402
        else
        { // :404-420
          const float4 c = Pw[w];
          const float d0 = c.x - q.x, d1 = c.y - q.y, d2 = c.z - q.z;
          const float pd = d0 * d0 * a.cp_norm + d1 * d1 * a.cp_norm + d2 * d2 * a.cp_norm;
          const float dissimilarity = (dist + pd) / (1.0f + a.center_weight);
          wt = fast_mexp2(fmaxf(0.0f, dissimilarity * a.sharpness - 2.0f));
        }
        acc[k].x += q.x * wt;
        acc[k].y += q.y * wt;
        acc[k].z += q.z * wt;
        acc[k].w += 1.0f * wt;
      }
    }
    __syncthreads(); // Q and the distortions are overwritten by the next patch
  }
  cp_async_wait_all(); // a chunk none of whose patches ran never waited for P

  // ---- normalise (and blend) : :485-519 ---------------------------------------------------------------
#pragma unroll
  for(int k = 0; k < WOWN; k++)
  {
    if(own[k] < 0) continue;
    const float4 v = acc[k];
    const size_t g = (size_t)(chunk_top + (own[k] >> 16)) * width + chunk_left + (own[k] & 0xffff);
    float4 o;
    if(a.skip_blend)
      o = make_float4(v.x / v.w, v.y / v.w, v.z / v.w, v.w / v.w);
    else
    {
      const float4 i4 = __ldg(in + g);
      o.x = (i4.x * a.invert[0]) + (v.x / v.w * a.weight[0]);
      o.y = (i4.y * a.invert[1]) + (v.y / v.w * a.weight[1]);
      o.z = (i4.z * a.invert[2]) + (v.z / v.w * a.weight[2]);
      o.w = (i4.w * a.invert[3]) + (v.w / v.w * a.weight[3]);
    }
    a.out[g] = o;
  }
}

#endif // B200_KERNELS_ON_CPU

#include "nlm_group.cuh"

// scatter(), :95-104: evaluated in double, truncated to int
int scatter(float scale, float scattering, int i1, int i2)
{
  const int a1 = abs(i1), a2 = abs(i2);
  const int sg = (i1 > 0) - (i1 < 0);
  return (int)(scale * ((a1 * a1 * a1 + 7.0 * a1 * sqrt((double)a2)) * sg * scattering / 6.0 + i1));
}
int slice_height(int height) // :267-296
{
  if(height % SLICE_HEIGHT == 0) return SLICE_HEIGHT;
  int best = height % SLICE_HEIGHT, best_incr = 0;
  for(int incr = 1; incr < 10; incr++)
  {
    const int plus_rem = height % (SLICE_HEIGHT + incr);
    if(plus_rem == 0) return SLICE_HEIGHT + incr;
    if(plus_rem > best)
    {
      best_incr = +incr;
      best = plus_rem;
    }
    const int minus_rem = height % (SLICE_HEIGHT - incr);
    if(minus_rem == 0) return SLICE_HEIGHT - incr;
    if(minus_rem > best)
    {
      best_incr = -incr;
      best = minus_rem;
    }
  }
  return SLICE_HEIGHT + best_incr;
}
int slice_width(int width) // :299-312
{
  int sl = SLICE_WIDTH;
  int rem = width % sl;
  if(rem < SLICE_WIDTH / 2 && (width % (sl - 4)) > rem)
  {
    sl -= 4;
    rem = width % sl;
    if(rem < SLICE_WIDTH / 2 && (width % (sl - 4)) > rem) sl -= 4;
  }
  return sl;
}

// ---- host side of the group kernel: geometry of the window and of the column-sum planes, patches in flight ---------
// false: the chunk window plus two planes do not fit `smem_optin` bytes (or the radius is beyond the kernel's rings)
bool grp_plan(grp_args_t &g, int n_patches, int width, int height, int radius, float center_weight, float sharpness, const float norm[4],
              const float weight[4], const float invert[4], int skip_blend, int shift_max, int smem_optin, int g_cap)
{
  if(radius < 1 || radius > 2) return false; // the rings of 7 and 9 rows do not fit the register file next to the pixel sums
  g.n_patches = n_patches;
  g.width = width;
  g.height = height;
  g.chk_h = slice_height(height);
  g.chk_w = slice_width(width);
  g.n_cl = (width + g.chk_w - 1) / g.chk_w;
  g.radius = radius;
  g.center_weight = center_weight;
  g.sharpness = sharpness;
  const int pw = 2 * radius + 1;
  g.cp_norm = center_weight * pw * pw; // compute_center_pixel_norm(), :147-153
  g.div_d = 1.0f + center_weight;      // :416
  g.div_rcp = 1.0f / g.div_d;
  for(int c = 0; c < 4; c++)
  {
    g.norm[c] = norm[c];
    g.weight[c] = weight[c];
    g.invert[c] = invert[c];
  }
  g.skip_blend = skip_blend;
  g.hs = shift_max;
  g.wrows = g.chk_h + 2 * radius + 1 + 2 * shift_max;
  g.wcols = g.chk_w + 2 * radius + 2 * shift_max;
  g.splane = (g.chk_h + 1) * GRP_SP;
  if(g.chk_h > MAX_CH || g.chk_w > MAX_CW || g.wcols > GRP_WP_WIDE || g.chk_w + 2 * radius + 1 > GRP_SP) return false;
  g.wp = g.wcols <= GRP_WP_NARROW ? GRP_WP_NARROW : GRP_WP_WIDE;
  const long long wbytes = (long long)g.wrows * 3 * g.wp * 4, sbytes = (long long)g.splane * 4;
  if(wbytes + 2 * sbytes + GRP_MAXG * 4 > smem_optin) return false;
  int G = (int)((smem_optin - wbytes - GRP_MAXG * 4) / sbytes);
  G = (G < g_cap ? G : g_cap);
  G = (G < GRP_MAXG ? G : GRP_MAXG) & ~1;
  if(G < 2) return false;
  g.G = G;
  return true;
}
int grp_pairs_per_thread(const grp_args_t &g) { return (((g.chk_h + 1) / 2) * g.chk_w + GRP_NT - 1) / GRP_NT; }
size_t grp_pipe_smem_bytes(const grp_args_t &g, int wp) { return ((size_t)g.wrows * 3 * wp + (size_t)2 * PIPE_SLOTS * g.splane + (size_t)g.n_patches) * sizeof(float); }
size_t grp_smem_bytes(const grp_args_t &g) { return ((size_t)g.wrows * 3 * g.wp + (size_t)g.G * g.splane + GRP_MAXG) * sizeof(float); }
// Markstein's division is the reference's division as long as nothing underflows on the way; where it could (x below
// 2^-44 with these bounds) the weight is 1 whatever the last bit of the quotient, because x / d * sharpness < 2^-24
// vanishes against the 2 it is subtracted from.  An infinite x enters the sequence as FLT_MAX: FLT_MAX / d * sharpness
// is beyond 128 with these bounds, so its weight is the 0 the reference gets from the infinity.
bool grp_division_by_constant(const grp_args_t &g)
{
  return !(g.center_weight < 0) && g.div_d >= 1.0f && g.div_d <= 1048576.0f && g.sharpness >= 1e-30f && g.sharpness <= 1048576.0f;
}
// define_patches(), :107-145; returns the largest |shift|
int grp_define_patches(patch_t *patches, int search_radius, float scale, float scattering, int decimate)
{
  int k = 0, dec = decimate, shift_max = 0;
  for(int ri = -search_radius; ri <= search_radius; ri++)
    for(int ci = -search_radius; ci <= search_radius; ci++)
    {
      if(dec && (++dec & 1)) continue;
      patches[k].rows = (short)scatter(scale, scattering, ri, ci);
      patches[k].cols = (short)scatter(scale, scattering, ci, ri);
      const int ar = abs((int)patches[k].rows), ac = abs((int)patches[k].cols);
      if(ar > shift_max) shift_max = ar;
      if(ac > shift_max) shift_max = ac;
      k++;
    }
  return shift_max;
}

// the pipelined kernel (nlm_pipe_kernel): chunks of up to 64 rows, the narrow window, a ring of PIPE_SLOTS pair slots
bool grp_pipe_fits(const grp_args_t &g, int smem_optin, int wp)
{
  return g.wcols <= PIPE_WCOLS_MAX && g.chk_h <= PIPE_MAX_ROWS && (long long)grp_pipe_smem_bytes(g, wp) <= smem_optin;
}

#ifndef B200_KERNELS_ON_CPU
template <int R, int CFG> cudaError_t launch_pipe_r(const grp_args_t &g, bool norm1, bool profiled, bool divc, unsigned grid, size_t smem, cudaStream_t stream)
{
#define PIPE_LAUNCH(N1, PR, DC)                                                                                        \
  do                                                                                                                   \
  {                                                                                                                    \
    cudaError_t e = cudaFuncSetAttribute(nlm_pipe_kernel<R, N1, PR, DC, CFG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if(e != cudaSuccess) return e;                                                                                     \
    {                                                                                                                  \
      ::b200::timed_launch timed(::b200::TIMED_NLM, stream);                                                           \
      nlm_pipe_kernel<R, N1, PR, DC, CFG><<<grid, pipe_cfg<CFG>::NT, smem, stream>>>(g);                              \
    }                                                                                                                  \
    return cudaGetLastError();                                                                                         \
  } while(0)
  if(!profiled)
  {
    if(norm1) PIPE_LAUNCH(true, false, false);
    PIPE_LAUNCH(false, false, false);
  }
  if(divc)
  {
    if(norm1) PIPE_LAUNCH(true, true, true);
    PIPE_LAUNCH(false, true, true);
  }
  if(norm1) PIPE_LAUNCH(true, true, false);
  PIPE_LAUNCH(false, true, false);
#undef PIPE_LAUNCH
}

template <int R, int WP, int KP> cudaError_t launch_group_r(const grp_args_t &g, bool norm1, bool profiled, bool divc, unsigned grid, size_t smem, cudaStream_t stream)
{
#define GRP_LAUNCH(N1, PR, DC)                                                                                         \
  do                                                                                                                   \
  {                                                                                                                    \
    cudaError_t e = cudaFuncSetAttribute(nlm_group_kernel<R, WP, N1, PR, DC, KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if(e != cudaSuccess) return e;                                                                                     \
    {                                                                                                                  \
      ::b200::timed_launch timed(::b200::TIMED_NLM, stream);                                                           \
      nlm_group_kernel<R, WP, N1, PR, DC, KP><<<grid, GRP_NT, smem, stream>>>(g);                                      \
    }                                                                                                                  \
    return cudaGetLastError();                                                                                         \
  } while(0)
  if(!profiled)
  {
    if(norm1) GRP_LAUNCH(true, false, false);
    GRP_LAUNCH(false, false, false);
  }
  if(divc)
  {
    if(norm1) GRP_LAUNCH(true, true, true);
    GRP_LAUNCH(false, true, true);
  }
  if(norm1) GRP_LAUNCH(true, true, false);
  GRP_LAUNCH(false, true, false);
#undef GRP_LAUNCH
}

// the group kernel, if the chunk window and two or more planes of column sums fit; *launched tells
int launch_group(const nlm_args_t &a, int shift_max, int smem_optin, int n_chunks, cudaStream_t stream, int *launched)
{
  *launched = 0;
  grp_args_t g;
  g.in = a.in;
  g.out = a.out;
  g.patches = a.patches;
  int g_cap = GRP_MAXG;
  if(const char *e = getenv("B200_NLM_G")) g_cap = atoi(e);
  if(!grp_plan(g, a.n_patches, a.width, a.height, a.radius, a.center_weight, a.sharpness, a.norm, a.weight, a.invert, a.skip_blend,
               shift_max, smem_optin, g_cap))
    return B200_OK;
  const bool profiled = !(a.center_weight < 0);
  const bool norm1 = a.norm[0] == 1.0f && a.norm[1] == 1.0f && a.norm[2] == 1.0f;
  const bool divc = grp_division_by_constant(g) && !getenv("B200_NLM_IEEE_DIV");
  cudaError_t e;
  const unsigned grid = (unsigned)n_chunks;
  const int pipe_wp = pipe_cfg<0>::WP;
  if(grp_pipe_fits(g, smem_optin, pipe_wp) && !getenv("B200_NLM_NO_PIPE"))
  {
    const size_t psmem = grp_pipe_smem_bytes(g, pipe_wp);
    const bool halves = !getenv("B200_NLM_WHOLE_SLOTS"); // development switch: the whole-pair slots everywhere
    if(halves)
      e = a.radius == 1 ? launch_pipe_r<1, 0>(g, norm1, profiled, divc, grid, psmem, stream) : launch_pipe_r<2, 0>(g, norm1, profiled, divc, grid, psmem, stream);
    else
      e = a.radius == 1 ? launch_pipe_r<1, 1>(g, norm1, profiled, divc, grid, psmem, stream) : launch_pipe_r<2, 1>(g, norm1, profiled, divc, grid, psmem, stream);
    if(e != cudaSuccess) return ::b200::fail(B200_ERR_CUDA, "nlmeans: pipelined kernel launch: %s", cudaGetErrorString(e));
    *launched = 1;
    return B200_OK;
  }
  const size_t smem = grp_smem_bytes(g);
  const int variant = (a.radius == 2 ? 4 : 0) + (g.wp == GRP_WP_WIDE ? 2 : 0) + (grp_pairs_per_thread(g) > GRP_KP_MIN ? 1 : 0);
  switch(variant)
  {
    case 0: e = launch_group_r<1, GRP_WP_NARROW, GRP_KP_MIN>(g, norm1, profiled, divc, grid, smem, stream); break;
    case 1: e = launch_group_r<1, GRP_WP_NARROW, GRP_KP_MAX>(g, norm1, profiled, divc, grid, smem, stream); break;
    case 2: e = launch_group_r<1, GRP_WP_WIDE, GRP_KP_MIN>(g, norm1, profiled, divc, grid, smem, stream); break;
    case 3: e = launch_group_r<1, GRP_WP_WIDE, GRP_KP_MAX>(g, norm1, profiled, divc, grid, smem, stream); break;
    case 4: e = launch_group_r<2, GRP_WP_NARROW, GRP_KP_MIN>(g, norm1, profiled, divc, grid, smem, stream); break;
    case 5: e = launch_group_r<2, GRP_WP_NARROW, GRP_KP_MAX>(g, norm1, profiled, divc, grid, smem, stream); break;
    case 6: e = launch_group_r<2, GRP_WP_WIDE, GRP_KP_MIN>(g, norm1, profiled, divc, grid, smem, stream); break;
    default: e = launch_group_r<2, GRP_WP_WIDE, GRP_KP_MAX>(g, norm1, profiled, divc, grid, smem, stream); break;
  }
  if(e != cudaSuccess) return ::b200::fail(B200_ERR_CUDA, "nlmeans: group kernel launch: %s", cudaGetErrorString(e));
  *launched = 1;
  return B200_OK;
}
#endif // B200_KERNELS_ON_CPU
} // namespace

#ifndef B200_KERNELS_ON_CPU
namespace b200
{
// nlmeans_denoise(), :315-532, on device RGBA buffers.  in != out.
int nlmeans_denoise_dev(const float *d_in, float *d_out, int width, int height, float scattering, float scale, float luma,
                        float chroma, float center_weight, float sharpness, int radius, int search_radius, int decimate,
                        const float norm[4], cudaStream_t stream)
{
  if(radius < 0 || radius > MAX_RADIUS) return fail(B200_ERR_UNSUPPORTED, "nlmeans: patch radius %d outside 0..%d", radius, MAX_RADIUS);
  if(search_radius < 0 || search_radius > 64) return fail(B200_ERR_ARG, "nlmeans: search radius %d", search_radius);
  int n_patches = (2 * search_radius + 1) * (2 * search_radius + 1);
  if(decimate) n_patches = (n_patches + 1) / 2;
  patch_t *h_patches = (patch_t *)malloc(sizeof(patch_t) * (size_t)n_patches);
  if(!h_patches) return fail(B200_ERR_NOMEM, "nlmeans: host allocation");
  const int h_shift_max = grp_define_patches(h_patches, search_radius, scale, scattering, decimate);
  void *d_patches = nullptr;
  int rc = scratch(SLOT_SMALL + 1, sizeof(patch_t) * (size_t)n_patches, &d_patches);
  if(rc)
  {
    free(h_patches);
    return rc;
  }
  cudaError_t e = cudaMemcpyAsync(d_patches, h_patches, sizeof(patch_t) * (size_t)n_patches, cudaMemcpyHostToDevice, stream);
  if(e == cudaSuccess) e = cudaStreamSynchronize(stream); // h_patches is freed below
  free(h_patches);
  if(e != cudaSuccess) return fail(B200_ERR_CUDA, "nlmeans: patch upload: %s", cudaGetErrorString(e));

  nlm_args_t a;
  a.in = (const float4 *)d_in;
  a.out = (float4 *)d_out;
  a.patches = (const patch_t *)d_patches;
  a.n_patches = n_patches;
  a.width = width;
  a.height = height;
  a.chk_h = slice_height(height);
  a.chk_w = slice_width(width);
  a.n_cl = (width + a.chk_w - 1) / a.chk_w;
  const int n_ct = (height + a.chk_h - 1) / a.chk_h;
  a.radius = radius;
  a.center_weight = center_weight;
  a.sharpness = sharpness;
  const int pw = 2 * radius + 1;
  a.cp_norm = center_weight * pw * pw; // compute_center_pixel_norm(), :147-153
  for(int c = 0; c < 4; c++) a.norm[c] = norm[c];
  a.weight[0] = luma;
  a.weight[1] = a.weight[2] = chroma;
  a.weight[3] = 1.0f;
  a.invert[0] = 1.0f - luma;
  a.invert[1] = a.invert[2] = 1.0f - chroma;
  a.invert[3] = 0.0f;
  a.skip_blend = (luma == 1.0 && chroma == 1.0) ? 1 : 0;
  if(width >= 32768 || height >= 32768) return fail(B200_ERR_UNSUPPORTED, "nlmeans: frames beyond 32767 px a side are not supported");
  if(a.chk_h > MAX_CH || a.chk_w > MAX_CW) return fail(B200_ERR_ARG, "nlmeans: chunk %dx%d exceeds the kernel's tile", a.chk_w, a.chk_h);

  a.rows_e = a.chk_h + 2 * radius + 1;
  a.plane_e = a.rows_e * SW;
  a.cols_w = a.chk_w + 2 * radius + 2;
  a.sstride_w = a.cols_w | 1;
  // per device, 0 until the kernels' shared-memory attributes are set: one atomic, so no thread sees "set" without the
  // limit.  Two threads may both set them, to the same values.
  static std::atomic<int> smem_optin[16] = {};
  int dev = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  int optin = smem_optin[dev & 15].load(std::memory_order_acquire);
  if(!optin)
  {
    const int smem_max = 2 * (3 * (MAX_CH + 2 * MAX_RADIUS + 1) * SW + MAX_CH * SSTRIDE) * (int)sizeof(float);
    B200_CUDA_TRY(cudaFuncSetAttribute(nlm_chunks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    B200_CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    B200_CUDA_TRY(cudaFuncSetAttribute(nlm_chunks_win_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
    smem_optin[dev & 15].store(optin, std::memory_order_release);
  }
  // The group kernel (nlm_group.cuh) wherever the pixels a chunk reads for every patch, plus at least two planes of
  // column sums, fit the shared memory of an SM: every module default does (K = 7 with P <= 4 and no scattering).
  if(!getenv("B200_NLM_CHUNKS") && !getenv("B200_NLM_WINDOW"))
  {
    int launched = 0;
    if((rc = launch_group(a, h_shift_max, optin, n_ct * a.n_cl, stream, &launched))) return rc;
    if(launched) return B200_OK;
  }
  const long long win_bytes = 2LL * a.rows_e * a.cols_w * 16 + 2LL * a.chk_h * a.sstride_w * 4;
  // Measured at 45 MP, K=7, P=1: E-plane kernel 126 ms, window kernel 137 ms (both bit-exact; the window kernel
  // moves all global traffic into one cp.async fill per patch but spends twice the instructions on index
  // arithmetic in its parallel phases).  The window kernel stays selectable for that follow-up work.
  const bool use_window = getenv("B200_NLM_WINDOW") != nullptr;
  if(use_window && win_bytes <= optin)
    nlm_chunks_win_kernel<<<(unsigned)(n_ct * a.n_cl), WNT, (size_t)win_bytes, stream>>>(a);
  else
  {
    const int smem_bytes = 2 * (3 * a.plane_e + a.chk_h * SSTRIDE) * (int)sizeof(float); // E and S double-buffered
    nlm_chunks_kernel<<<(unsigned)(n_ct * a.n_cl), NT, smem_bytes, stream>>>(a);
  }
  B200_CUDA_TRY(cudaGetLastError());
  return B200_OK;
}

int denoise_vst_forward(const b200_piece_t *piece, const b200_denoiseprofile_data_t *d, const float *d_in, float *d_out,
                        size_t npx, bool nlm, cudaStream_t s);
int denoise_vst_backward(const b200_piece_t *piece, const b200_denoiseprofile_data_t *d, float *d_buf, size_t npx, bool nlm,
                         cudaStream_t s);
int denoise_alpha_copy(const float *d_in, float *d_out, size_t npx, cudaStream_t s);

// process_nlmeans_cpu(), denoiseprofile.c:1599-1648
int denoiseprofile_nlmeans_dev(const b200_piece_t *piece, const b200_denoiseprofile_data_t *d, const float *d_in, float *d_out,
                               cudaStream_t s)
{
  const int width = piece->roi_in.width, height = piece->roi_in.height;
  const size_t npx = (size_t)width * height;
  const float scale = fminf(fminf((float)piece->roi_in.scale, 2.0f), 1.0f);
  const int P = (int)ceilf(d->radius * scale);
  int K = (int)d->nbhood;
  float scattering = d->scattering;
  { // nlmeans_scattering(), :1474-1499.  dt_dev_pixelpipe_has_preview_output() is read as "preview pipe".
    const bool has_preview = piece->pipe_type == B200_PIPE_PREVIEW;
    if(has_preview || piece->pipe_type == B200_PIPE_THUMBNAIL)
    {
      const int maxk = (int)((K * K * K + 7.0 * K * sqrt((double)K)) * scattering / 6.0 + K);
      K = K < 3 ? K : 3;
      scattering = (float)((maxk - K) * 6.0 / (K * K * K + 7.0 * K * sqrt((double)K)));
    }
    if(!has_preview)
    {
      const int maxk = (int)((K * K * K + 7.0 * K * sqrt((double)K)) * scattering / 6.0 + K);
      const int k4 = K < 4 ? K : 4;
      const float ks = K * scale;
      K = (int)((float)k4 > ks ? (float)k4 : ks);
      scattering = (float)((maxk - K) * 6.0 / (K * K * K + 7.0 * K * sqrt((double)K)));
    }
  }
  float norm = .045f / ((2 * P + 1) * (2 * P + 1)); // nlmeans_norm(), :1456-1470
  if(!d->fix_anscombe_and_nlmeans_norm) norm = .015f / (2 * P + 1);
  const float central_pixel_weight = d->central_pixel_weight * scale;

  void *pre = nullptr;
  int rc = scratch(SLOT_TMP0, npx * 16, &pre);
  if(rc) return rc;
  if((rc = denoise_vst_forward(piece, d, d_in, (float *)pre, npx, true, s))) return rc;
  const float norm2[4] = { 1.0f, 1.0f, 1.0f, 1.0f };
  if((rc = nlmeans_denoise_dev((const float *)pre, d_out, width, height, scattering, scale, 1.0f, 1.0f, central_pixel_weight, norm, P,
                               K, 0, norm2, s)))
    return rc;
  if((rc = denoise_vst_backward(piece, d, d_out, npx, true, s))) return rc;
  if(piece->mask_display & B200_DISPLAY_MASK) return denoise_alpha_copy(d_in, d_out, npx, s); // :1645-1646
  return B200_OK;
}
} // namespace b200
#endif // B200_KERNELS_ON_CPU
