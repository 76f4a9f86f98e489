// AMaZE demosaic (Aliasing Minimization and Zipper Elimination) for B200 / sm_100a.
//
// What the reference computes: src/iop/demosaic/amaze.cc amaze_demosaic_RT :181-1419 (RawTherapee's
// amaze_interpolate_RT as vendored there).  Parity contract: bit-identical to that source under C float semantics
// (oracle/restate/amaze_oracle.c, pinned against amaze.cc compiled in place) with the tile scratch zeroed per tile.
// What shapes the kernel:
//   * the result depends on the reference's 160-px tile grid (128 kept, origin -16): several planes are updated in
//     place in raster order, so one CTA processes exactly one reference tile at a time;
//   * the scratch planes alias by lifetime exactly as in the reference (:298-328): a read that lands on a location its
//     own producer never wrote sees what the aliased plane left there, so the layout is part of the contract.  The
//     reference carries its scratch from tile to tile (thread-count dependent, ~0.007 % of the pixels); here it is
//     zeroed per tile (oracle scratch_mode 1);
//   * three sweeps are sequential by construction and are evaluated in the reference's order:
//       - hcd / vcd variance choice and saturation bounds (:580-686): hcd runs along each row (stride 2), vcd down
//         each column (stride 2 rows) -> one thread per chain;
//       - hvwt (:899) and pmwt (:1117) refinement: row r reads the already refined row r-1 -> rows in order, sites of a
//         row in parallel;
//   * mixed precision of the source is kept (`0.5 - varwt`, `cfa * 2.0 / ...`, `2.0 * (...)` are double).
// 14 float planes of 160x160 per tile (1.45 MB) do not fit in shared memory: each persistent CTA owns a scratch region
// in global memory; the row-sequential refinements stage their half plane in shared memory, the chain sweeps fetch the
// operands of four steps at a time.
#include "runtime.h"
#include <atomic>
#include <math.h>

namespace
{
constexpr int TS = 160, TSH = TS / 2;
#ifndef AMAZE_NT
#define AMAZE_NT 640
#endif
#ifndef AMAZE_MINB
#define AMAZE_MINB 2
#endif
constexpr int NT = AMAZE_NT;       // a multiple of 160: 160 columns x NT/160 row groups, or 80 site columns x NT/80 row groups
static_assert(NT % TS == 0 && NT >= 640, "the chain sweeps need 2 x 304 threads");
constexpr int RG4 = NT / TS, RG8 = NT / TSH;
constexpr size_t FULL = sizeof(float) * TS * TS, HALF = sizeof(float) * TS * TSH, PAD = 2 * 64;
constexpr size_t SCRATCH_BYTES = 14 * FULL + TS * TSH + 18 * PAD; // amaze.cc:283 without the alignment slack
constexpr size_t SCRATCH_STRIDE = (SCRATCH_BYTES + 255) / 256 * 256;

struct amaze_args_t
{
  const float *in;
  float *out;
  char *scratch;
  int width, height;
  uint32_t filters;
  float clip_pt, clip_pt8;
  int ntx, ntiles;
  int ex, ey;
};

struct hv_t
{
  float h, v;
};

__device__ __forceinline__ int fc(int row, int col, uint32_t f)
{
  return (int)((f >> (((((unsigned)row << 1) & 14u) + ((unsigned)col & 1u)) << 1)) & 3u);
}
__device__ __forceinline__ float amz_min(float a, float b) { return (b < a) ? b : a; } // std::min
__device__ __forceinline__ float amz_max(float a, float b) { return (a < b) ? b : a; } // std::max
__device__ __forceinline__ float LIMF(float a, float b, float c) { return amz_max(b, amz_min(a, c)); }
__device__ __forceinline__ float ULIMF(float a, float b, float c) { return (b < c) ? LIMF(a, b, c) : LIMF(a, c, b); }
__device__ __forceinline__ float SQ(float x) { return x * x; }
__device__ __forceinline__ float mixf(float a, float b, float c) { return a * (b - c) + c; }
__device__ __forceinline__ float clampnan(float x, float m, float M)
{ // amaze.cc:60-75
  if(!(fabsf(x) <= 3.402823466e+38f)) // inf or NaN
    return (x < m) ? m : ((x > M) ? M : x);
  return x;
}
__device__ __forceinline__ float exp_add(float d, int n)
{ // xmul2f / xdiv2f / xdivf, :77-122
  unsigned u = __float_as_uint(d);
  if(u & 0x7FFFFFFFu) u += (unsigned)(n << 23);
  return __uint_as_float(u);
}
#define XMUL2(x) exp_add((x), 1)
#define XDIV2(x) exp_add((x), -1)
#define XDIV4(x) exp_add((x), -2)
#define GMIN(a, b) (((a) < (b)) ? (a) : (b))

// one element of the in-place variance choice + saturation bound sweep (:583-684) for hcd (lo/hi = left/right raw
// neighbours) or vcd (lo/hi = up/down); prev is the already updated element two steps back along the chain
__device__ float cd_update(float prev, float cur, float next, float ap, float ac, float an, bool green, float cf, float lo, float hi, float clip_pt)
{
  const float eps = 1e-5f;
  const float var = 3.f * (SQ(prev) + SQ(cur) + SQ(next)) - SQ(prev + cur + next);
  const float altvar = 3.f * (SQ(ap) + SQ(ac) + SQ(an)) - SQ(ap + ac + an);
  float cd = cur;
  if(altvar < var) cd = ac;
  if(green)
  {
    const float G = -cd + cf;
    if(cd > 0)
    {
      if(3.f * cd > (G + cf))
        cd = -ULIMF(G, lo, hi) + cf;
      else
      {
        const float wt = 1.f - 3.f * cd / (eps + G + cf);
        cd = wt * cd + (1.f - wt) * (-ULIMF(G, lo, hi) + cf);
      }
    }
    if(G > clip_pt) cd = -ULIMF(G, lo, hi) + cf;
  }
  else
  {
    const float G = cd + cf;
    if(cd < 0)
    {
      if(3.f * cd < -(G + cf))
        cd = ULIMF(G, lo, hi) - cf;
      else
      {
        const float wt = 1.f + 3.f * cd / (eps + G + cf);
        cd = wt * cd + (1.f - wt) * (ULIMF(G, lo, hi) - cf);
      }
    }
    if(G > clip_pt) cd = ULIMF(G, lo, hi) - cf;
  }
  return cd;
}

// One chain of that sweep: elements i0, i0 + S, ... (n of them), neighbours of a site at +-N (S = 2N).  Everything a
// step reads except `prev` is original data (the chain only ever rewrites elements behind it), so the operands of four
// steps are fetched together before the dependent arithmetic runs: one memory round trip per four steps.
template <int S, int N> __device__ __forceinline__ void cd_chain(float *cd, const float *alt, const float *cfa, int i0, int n, bool green, float clip_pt)
{
  float prev = cd[i0 - S], cur = cd[i0], ap = alt[i0 - S], ac = alt[i0], lo = cfa[i0 - N];
  for(int k = 0; k < n; k += 4)
  {
    const int i = i0 + k * S;
    float nx[4], an[4], cf[4], hi[4];
#pragma unroll
    for(int u = 0; u < 4; u++)
    { // reads past the end of a short chain stay inside the scratch region and are not used
      nx[u] = cd[i + (u + 1) * S];
      an[u] = alt[i + (u + 1) * S];
      cf[u] = cfa[i + u * S];
      hi[u] = cfa[i + u * S + N];
    }
#pragma unroll
    for(int u = 0; u < 4; u++)
      if(k + u < n)
      {
        const float nv = cd_update(prev, cur, nx[u], ap, ac, an[u], green, cf[u], lo, hi[u], clip_pt);
        cd[i + u * S] = nv;
        prev = nv;
        cur = nx[u];
        ap = ac;
        ac = an[u];
        lo = hi[u];
      }
  }
}

// a half plane (160 x 80 floats) to and from shared memory for the row-sequential refinements
constexpr int ROW_T = 96; // the three warps that hold a row's 80 sites
__device__ __forceinline__ void stage_in(float *sm, const float *g, int tid)
{
  for(int k = tid; k < TS * TSH / 4; k += NT) reinterpret_cast<float4 *>(sm)[k] = reinterpret_cast<const float4 *>(g)[k];
}
__device__ __forceinline__ void stage_out(float *g, const float *sm, int tid)
{
  for(int k = tid; k < TS * TSH / 4; k += NT) reinterpret_cast<float4 *>(g)[k] = reinterpret_cast<const float4 *>(sm)[k];
}
__device__ __forceinline__ void row_barrier() { asm volatile("bar.sync 1, 96;" ::: "memory"); }

#define FULL_LOOP(a)                                   \
  for(int rr = (a) + y4; rr < rr1 - (a); rr += RG4)    \
  {                                                    \
    const int cc = x160;                               \
    if(cc >= (a) && cc < cc1 - (a))                    \
    {                                                  \
      const int i = rr * TS + cc;
#define SITE_LOOP(a)                                              \
  for(int rr = (a) + y8; rr < rr1 - (a); rr += RG8)               \
  {                                                               \
    const int cc = (a) + (fc(rr, 2, f) & 1) + 2 * x80;            \
    if(cc < cc1 - (a))                                            \
    {                                                             \
      const int i = rr * TS + cc;
#define NYQ_LOOP                                                                       \
  for(int rr = nystartrow + y8; rr < nyendrow; rr += RG8)                              \
  {                                                                                    \
    const int i = rr * TS + nystartcol + (fc(rr, 2, f) & 1) + 2 * x80;                 \
    if(i < rr * TS + nyendcol)                                                         \
    {
#define END_LOOP \
  }              \
  }

#ifdef B200_AMAZE_PROF
// development aid (tools/prof_amaze.py): cycles of CTA 0 between the section marks, summed over its tiles
__device__ unsigned long long g_amaze_prof[40];
#define AMAZE_PROF_MARK()                                         \
  do                                                              \
  {                                                               \
    if(blockIdx.x == 0 && tid == 0)                               \
    {                                                             \
      const long long now_ = clock64();                           \
      g_amaze_prof[prof_k] += (unsigned long long)(now_ - prof_t); \
      prof_t = now_;                                              \
    }                                                             \
    prof_k++;                                                     \
  } while(0)
#else
#define AMAZE_PROF_MARK() \
  do                      \
  {                       \
  } while(0)
#endif

__global__ void __launch_bounds__(NT, AMAZE_MINB) amaze_tiles_kernel(const amaze_args_t a)
{
  __shared__ int s_ny[4];
  extern __shared__ __align__(16) float s_half[]; // TS * TSH floats
  const int tid = threadIdx.x;
  const int x160 = tid % TS, y4 = tid / TS, x80 = tid % TSH, y8 = tid / TSH;
  const uint32_t f = a.filters;
  const int width = a.width, height = a.height;
  const float clip_pt = a.clip_pt, clip_pt8 = a.clip_pt8;
  const int ts = TS, tsh = TSH;
  const int v1 = ts, v2 = 2 * ts, v3 = 3 * ts, p1 = -ts + 1, p2 = -2 * ts + 2, p3 = -3 * ts + 3, m1 = ts + 1, m2 = 2 * ts + 2, m3 = 3 * ts + 3;
  const float eps = 1e-5f, epssq = 1e-10f, arthresh = 0.75f;
  const float gaussodd[4] = { 0.14659727707323927f, 0.103592713382435f, 0.0732036125103057f, 0.0365543548389495f };
  const float nyqthresh = 0.5f;
  const float gaussgrad[6] = { nyqthresh * 0.07384411893421103f, nyqthresh * 0.06207511968171489f, nyqthresh * 0.0521818194747806f,
                               nyqthresh * 0.03687419286733595f, nyqthresh * 0.03099732204057846f, nyqthresh * 0.018413194161458882f };
  const float gausseven[2] = { 0.13719494435797422f, 0.05640252782101291f };
  const float gquinc[4] = { 0.169917f, 0.108947f, 0.069855f, 0.0287182f };

  // scratch layout, amaze.cc:283-329
  char *const data = a.scratch + (size_t)blockIdx.x * SCRATCH_STRIDE;
  float *const rgbgreen = (float *)data;
  float *const delhvsqsum = (float *)((char *)rgbgreen + FULL + PAD);
  float *const dirwts0 = (float *)((char *)delhvsqsum + FULL + PAD);
  float *const dirwts1 = (float *)((char *)dirwts0 + FULL + PAD);
  float *const vcd = (float *)((char *)dirwts1 + FULL + PAD);
  float *const hcd = (float *)((char *)vcd + FULL + PAD);
  float *const vcdalt = (float *)((char *)hcd + FULL + PAD);
  float *const hcdalt = (float *)((char *)vcdalt + FULL + PAD);
  float *const cddiffsq = (float *)((char *)hcdalt + FULL + PAD);
  float *const hvwt = (float *)((char *)cddiffsq + FULL + 2 * PAD);
  float *const Dgrb0 = vcdalt, *const Dgrb1 = vcdalt + TS * TSH;
  float *const delp = cddiffsq;
  float *const delm = (float *)((char *)delp + HALF + PAD);
  float *const rbint = delm;
  hv_t *const Dgrb2 = (hv_t *)((char *)hvwt + HALF + PAD);
  float *const dgintv = (float *)Dgrb2;
  float *const dginth = (float *)((char *)dgintv + FULL + PAD);
  float *const Dgrbsq1m = (float *)((char *)dginth + FULL + PAD);
  float *const Dgrbsq1p = (float *)((char *)Dgrbsq1m + HALF + PAD);
  float *const cfa = (float *)((char *)Dgrbsq1p + HALF + PAD);
  float *const pmwt = delhvsqsum;
  float *const rbm = vcd;
  float *const rbp = (float *)((char *)rbm + HALF + PAD);
  unsigned char *const nyquist = (unsigned char *)((char *)cfa + FULL + PAD);
  unsigned char *const nyquist2 = (unsigned char *)cddiffsq;
  float *const nyqutest = (float *)((char *)nyquist + TS * TSH + PAD);

  for(int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x)
  {
#ifdef B200_AMAZE_PROF
    int prof_k = 0;
    long long prof_t = clock64();
#endif
    const int ty = tile / a.ntx, tx = tile - ty * a.ntx;
    const int top = -16 + ty * (TS - 32), left = -16 + tx * (TS - 32);
    const int bottom = min(top + TS, height + 16), right = min(left + TS, width + 16);
    const int rr1 = bottom - top, cc1 = right - left;
    const int rrmin = top < 0 ? 16 : 0, ccmin = left < 0 ? 16 : 0;
    const int rrmax = bottom > height ? height - top : rr1;
    const int ccmax = right > width ? width - left : cc1;

    __syncthreads(); // the previous tile's output pass is done with the scratch
    { // scratch zeroed per tile (oracle scratch_mode 1; also covers memset(&nyquist[3*tsh], ...) :338)
      float4 *p = reinterpret_cast<float4 *>(data);
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      for(size_t k = tid; k < SCRATCH_STRIDE / 16; k += NT) p[k] = z;
    }
    if(tid < 4) s_ny[tid] = (tid == 0) ? (1 << 30) : (tid == 2 ? (1 << 30) : -1); // start row (min), end row (max), start col (min), end col (max)
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- tile load with the mirrored 16-px border at the frame edges, :357-455 -----------------------------------
    // The reference fills nine regions one after the other with the linear index rr*ts + cc and no bound on it: when the
    // frame edge sits less than 16 px before the tile edge, the right border runs over into column 0.. of the next row
    // (replacing what the left border put there) and the lower border runs past row 159 into the padding and the
    // Nyquist flags.  Both reach kept pixels, so the regions are written with the same indices in the same order.
#define PUT(idx_, src_)                         \
  do                                            \
  {                                             \
    const float t_ = __ldg(a.in + (src_));      \
    cfa[idx_] = t_;                             \
    rgbgreen[idx_] = t_;                        \
  } while(0)
    {
      const int ncc = ccmax - ccmin;
      // upper border, inner part, lower border (:357-391): pairwise disjoint targets
      if(rrmin > 0)
        for(int k = tid; k < 16 * ncc; k += NT)
        {
          const int rr = k / ncc, cc = ccmin + (k - rr * ncc);
          PUT(rr * TS + cc, (size_t)(32 - rr + top) * width + (cc + left));
        }
      for(int rr = rrmin + y4; rr < rrmax; rr += RG4)
      {
        const int cc = x160;
        if(cc >= ccmin && cc < ccmax) PUT(rr * TS + cc, (size_t)(rr + top) * width + (cc + left));
      }
      if(rrmax < rr1)
        for(int k = tid; k < 16 * ncc; k += NT)
        {
          const int rr = k / ncc, cc = ccmin + (k - rr * ncc);
          PUT((rrmax + rr) * TS + cc, (size_t)(height - rr - 2) * width + (left + cc));
        }
      __syncthreads();
      if(ccmin > 0) // left border, :395-403
        for(int k = tid; k < 16 * (rrmax - rrmin); k += NT)
        {
          const int rr = rrmin + (k >> 4), cc = k & 15;
          PUT(rr * TS + cc, (size_t)(rr + top) * width + (32 - cc + left));
        }
      __syncthreads();
      if(ccmax < cc1) // right border, :406-414
        for(int k = tid; k < 16 * (rrmax - rrmin); k += NT)
        {
          const int rr = rrmin + (k >> 4), cc = k & 15;
          PUT(rr * TS + ccmax + cc, (size_t)(top + rr) * width + (width - cc - 2));
        }
      __syncthreads();
      // the corners mirror about row/column 32, not 16 (:417-455); in the reference's order
      if(rrmin > 0 && ccmin > 0 && tid < 256) PUT((tid >> 4) * TS + (tid & 15), (size_t)(32 - (tid >> 4)) * width + (32 - (tid & 15)));
      __syncthreads();
      if(rrmax < rr1 && ccmax < cc1 && tid < 256)
        PUT((rrmax + (tid >> 4)) * TS + ccmax + (tid & 15), (size_t)(height - (tid >> 4) - 2) * width + (width - (tid & 15) - 2));
      __syncthreads();
      if(rrmin > 0 && ccmax < cc1 && tid < 256) PUT((tid >> 4) * TS + ccmax + (tid & 15), (size_t)(32 - (tid >> 4)) * width + (width - (tid & 15) - 2));
      __syncthreads();
      if(rrmax < rr1 && ccmin > 0 && tid < 256) PUT((rrmax + (tid >> 4)) * TS + (tid & 15), (size_t)(height - (tid >> 4) - 2) * width + (32 - (tid & 15)));
    }
#undef PUT
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- gradients and direction weights, :460-470 ---------------------------------------------------------------
    FULL_LOOP(2)
    const float delh = fabsf(cfa[i + 1] - cfa[i - 1]);
    const float delv = fabsf(cfa[i + v1] - cfa[i - v1]);
    dirwts0[i] = eps + fabsf(cfa[i + v2] - cfa[i]) + fabsf(cfa[i] - cfa[i - v2]) + delv;
    dirwts1[i] = eps + fabsf(cfa[i + 2] - cfa[i]) + fabsf(cfa[i] - cfa[i - 2]) + delh;
    delhvsqsum[i] = SQ(delh) + SQ(delv);
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- vertical / horizontal colour differences, :474-577 ------------------------------------------------------
    FULL_LOOP(4)
    const bool fcswitch = ((fc(rr, 4, f) & 1) ^ ((cc - 4) & 1)) != 0;
    const float c0 = cfa[i];
    const float cru = cfa[i - v1] * (dirwts0[i - v2] + dirwts0[i]) / (dirwts0[i - v2] * (eps + c0) + dirwts0[i] * (eps + cfa[i - v2]));
    const float crd = cfa[i + v1] * (dirwts0[i + v2] + dirwts0[i]) / (dirwts0[i + v2] * (eps + c0) + dirwts0[i] * (eps + cfa[i + v2]));
    const float crl = cfa[i - 1] * (dirwts1[i - 2] + dirwts1[i]) / (dirwts1[i - 2] * (eps + c0) + dirwts1[i] * (eps + cfa[i - 2]));
    const float crr = cfa[i + 1] * (dirwts1[i + 2] + dirwts1[i]) / (dirwts1[i + 2] * (eps + c0) + dirwts1[i] * (eps + cfa[i + 2]));
    const float guha = cfa[i - v1] + XDIV2(c0 - cfa[i - v2]);
    const float gdha = cfa[i + v1] + XDIV2(c0 - cfa[i + v2]);
    const float glha = cfa[i - 1] + XDIV2(c0 - cfa[i - 2]);
    const float grha = cfa[i + 1] + XDIV2(c0 - cfa[i + 2]);
    float guar = (fabsf(1.f - cru) < arthresh) ? c0 * cru : guha;
    float gdar = (fabsf(1.f - crd) < arthresh) ? c0 * crd : gdha;
    float glar = (fabsf(1.f - crl) < arthresh) ? c0 * crl : glha;
    float grar = (fabsf(1.f - crr) < arthresh) ? c0 * crr : grha;
    const float hwt = dirwts1[i - 1] / (dirwts1[i - 1] + dirwts1[i + 1]);
    const float vwt = dirwts0[i - v1] / (dirwts0[i + v1] + dirwts0[i - v1]);
    const float Gintvha = vwt * gdha + (1.f - vwt) * guha;
    const float Ginthha = hwt * grha + (1.f - hwt) * glha;
    float vc, hc, va, ha;
    if(fcswitch)
    {
      vc = c0 - (vwt * gdar + (1.f - vwt) * guar);
      hc = c0 - (hwt * grar + (1.f - hwt) * glar);
      va = c0 - Gintvha;
      ha = c0 - Ginthha;
    }
    else
    {
      vc = (vwt * gdar + (1.f - vwt) * guar) - c0;
      hc = (hwt * grar + (1.f - hwt) * glar) - c0;
      va = Gintvha - c0;
      ha = Ginthha - c0;
    }
    if(c0 > clip_pt8 || Gintvha > clip_pt8 || Ginthha > clip_pt8)
    {
      guar = guha;
      gdar = gdha;
      glar = glha;
      grar = grha;
      vc = va;
      hc = ha;
    }
    vcd[i] = vc;
    hcd[i] = hc;
    vcdalt[i] = va;
    hcdalt[i] = ha;
    dgintv[i] = GMIN(SQ(guha - gdha), SQ(guar - gdar));
    dginth[i] = GMIN(SQ(glha - grha), SQ(glar - grar));
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- smaller-variance choice and saturation bounds, in place in raster order, :580-686 -----------------------
    // hcd: one thread per (row, column parity) walks its row; vcd: one thread per (column, row parity) walks its column
    // The two sweeps touch different planes and run side by side on the two halves of the CTA.
    {
      const int nrows = rr1 - 8, ncols = cc1 - 8; // rows / columns 4 .. rr1-5 / cc1-5
      if(tid < 2 * nrows)
      {
        const int rr = 4 + (tid >> 1), q = tid & 1;
        const bool green = ((fc(rr, 4, f) & 1) != 0) ^ (q != 0);
        cd_chain<2, 1>(hcd, hcdalt, cfa, rr * TS + 4 + q, (cc1 - 8 - q + 1) >> 1, green, clip_pt);
      }
      else if(tid >= NT / 2 && tid - NT / 2 < 2 * ncols)
      {
        const int t = tid - NT / 2;
        const int cc = 4 + (t >> 1), q = t & 1;
        const bool green = ((fc(4 + q, 4, f) & 1) != 0) ^ (((cc - 4) & 1) != 0);
        cd_chain<2 * TS, TS>(vcd, vcdalt, cfa, (4 + q) * TS + cc, (rr1 - 8 - q + 1) >> 1, green, clip_pt);
      }
    }
    AMAZE_PROF_MARK(); // chains done (thread 0 walks an hcd row)
    __syncthreads();
    FULL_LOOP(4)
    const bool green = ((fc(rr, 4, f) & 1) ^ ((cc - 4) & 1)) != 0;
    if(!green) cddiffsq[i] = SQ(vcd[i] - hcd[i]);
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- adaptive H/V weight at R/B sites, :688-746 --------------------------------------------------------------
    SITE_LOOP(6)
    const float uave = vcd[i] + vcd[i - v1] + vcd[i - v2] + vcd[i - v3];
    const float dave = vcd[i] + vcd[i + v1] + vcd[i + v2] + vcd[i + v3];
    const float lave = hcd[i] + hcd[i - 1] + hcd[i - 2] + hcd[i - 3];
    const float rave = hcd[i] + hcd[i + 1] + hcd[i + 2] + hcd[i + 3];
    float Dgrbvvaru = SQ(vcd[i] - uave) + SQ(vcd[i - v1] - uave) + SQ(vcd[i - v2] - uave) + SQ(vcd[i - v3] - uave);
    float Dgrbvvard = SQ(vcd[i] - dave) + SQ(vcd[i + v1] - dave) + SQ(vcd[i + v2] - dave) + SQ(vcd[i + v3] - dave);
    float Dgrbhvarl = SQ(hcd[i] - lave) + SQ(hcd[i - 1] - lave) + SQ(hcd[i - 2] - lave) + SQ(hcd[i - 3] - lave);
    float Dgrbhvarr = SQ(hcd[i] - rave) + SQ(hcd[i + 1] - rave) + SQ(hcd[i + 2] - rave) + SQ(hcd[i + 3] - rave);
    const float hwt = dirwts1[i - 1] / (dirwts1[i - 1] + dirwts1[i + 1]);
    const float vwt = dirwts0[i - v1] / (dirwts0[i + v1] + dirwts0[i - v1]);
    const float vcdvar = epssq + vwt * Dgrbvvard + (1.f - vwt) * Dgrbvvaru;
    const float hcdvar = epssq + hwt * Dgrbhvarr + (1.f - hwt) * Dgrbhvarl;
    Dgrbvvaru = (dgintv[i]) + (dgintv[i - v1]) + (dgintv[i - v2]);
    Dgrbvvard = (dgintv[i]) + (dgintv[i + v1]) + (dgintv[i + v2]);
    Dgrbhvarl = (dginth[i]) + (dginth[i - 1]) + (dginth[i - 2]);
    Dgrbhvarr = (dginth[i]) + (dginth[i + 1]) + (dginth[i + 2]);
    const float vcdvar1 = epssq + vwt * Dgrbvvard + (1.f - vwt) * Dgrbvvaru;
    const float hcdvar1 = epssq + hwt * Dgrbhvarr + (1.f - hwt) * Dgrbhvarl;
    const float varwt = hcdvar / (vcdvar + hcdvar);
    const float diffwt = hcdvar1 / (vcdvar1 + hcdvar1);
    if((0.5 - (double)varwt) * (0.5 - (double)diffwt) > 0 && fabsf(0.5f - diffwt) < fabsf(0.5f - varwt))
      hvwt[i >> 1] = varwt;
    else
      hvwt[i >> 1] = diffwt;
    END_LOOP

    AMAZE_PROF_MARK();
    // ---- Nyquist texture test, :748-815 (cddiffsq and delhvsqsum are complete: barrier above) --------------------
    SITE_LOOP(6)
    const float t
        = (gaussodd[0] * cddiffsq[i] + gaussodd[1] * (cddiffsq[(i - m1)] + cddiffsq[(i + p1)] + cddiffsq[(i - p1)] + cddiffsq[(i + m1)])
           + gaussodd[2] * (cddiffsq[(i - v2)] + cddiffsq[(i - 2)] + cddiffsq[(i + 2)] + cddiffsq[(i + v2)])
           + gaussodd[3] * (cddiffsq[(i - m2)] + cddiffsq[(i + p2)] + cddiffsq[(i - p2)] + cddiffsq[(i + m2)]))
          - (gaussgrad[0] * delhvsqsum[i] + gaussgrad[1] * (delhvsqsum[i - v1] + delhvsqsum[i + 1] + delhvsqsum[i - 1] + delhvsqsum[i + v1])
             + gaussgrad[2] * (delhvsqsum[i - m1] + delhvsqsum[i + p1] + delhvsqsum[i - p1] + delhvsqsum[i + m1])
             + gaussgrad[3] * (delhvsqsum[i - v2] + delhvsqsum[i - 2] + delhvsqsum[i + 2] + delhvsqsum[i + v2])
             + gaussgrad[4]
                   * (delhvsqsum[i - v2 - 1] + delhvsqsum[i - v2 + 1] + delhvsqsum[i - ts - 2] + delhvsqsum[i - ts + 2] + delhvsqsum[i + ts - 2]
                      + delhvsqsum[i + ts + 2] + delhvsqsum[i + v2 - 1] + delhvsqsum[i + v2 + 1])
             + gaussgrad[5] * (delhvsqsum[i - m2] + delhvsqsum[i + p2] + delhvsqsum[i - p2] + delhvsqsum[i + m2]));
    nyqutest[i >> 1] = t;
    if(t > 0.f)
    {
      nyquist[i >> 1] = 1;
      atomicMin(&s_ny[0], rr);
      atomicMax(&s_ny[1], rr);
      atomicMin(&s_ny[2], cc);
      atomicMax(&s_ny[3], cc);
    }
    END_LOOP
    __syncthreads();
    int nystartrow = s_ny[0] == (1 << 30) ? 0 : s_ny[0], nyendrow = s_ny[1] < 0 ? 0 : s_ny[1];
    int nystartcol = s_ny[2] == (1 << 30) ? ts + 1 : s_ny[2], nyendcol = s_ny[3] < 0 ? 0 : s_ny[3];
    const bool doNyquist = nystartrow != nyendrow && nystartcol != nyendcol;
    if(doNyquist)
    { // :819-884
      nyendrow++;
      nyendcol++;
      nystartcol -= (nystartcol & 1);
      nystartrow = max(8, nystartrow);
      nyendrow = min(rr1 - 8, nyendrow);
      nystartcol = max(8, nystartcol);
      nyendcol = min(cc1 - 8, nyendcol);
      // memset(&nyquist2[4 * tsh], 0, (ts - 8) * tsh) -- nyquist2 aliases cddiffsq, whose consumers are done
      for(int k = tid; k < (TS - 8) * TSH / 4; k += NT) reinterpret_cast<unsigned *>(nyquist2 + 4 * TSH)[k] = 0u;
      __syncthreads();
      NYQ_LOOP
      const unsigned t = (nyquist[(i - v2) >> 1] + nyquist[(i - m1) >> 1] + nyquist[(i + p1) >> 1] + nyquist[(i - 2) >> 1] + nyquist[(i + 2) >> 1]
                          + nyquist[(i - p1) >> 1] + nyquist[(i + m1) >> 1] + nyquist[(i + v2) >> 1]);
      nyquist2[i >> 1] = t > 4 ? 1 : (t < 4 ? 0 : nyquist[i >> 1]);
      END_LOOP
      __syncthreads();
      NYQ_LOOP
      if(nyquist2[i >> 1])
      { // area interpolation
        float sumcfa = 0.f, sumh = 0.f, sumv = 0.f, sumsqh = 0.f, sumsqv = 0.f, areawt = 0.f;
        for(int u = -6; u < 7; u += 2)
        {
          int i1 = i + (u * ts) - 6;
          for(int w = -6; w < 7; w += 2, i1 += 2)
            if(nyquist2[i1 >> 1])
            {
              const float ct = cfa[i1];
              sumcfa += ct;
              sumh += (cfa[i1 - 1] + cfa[i1 + 1]);
              sumv += (cfa[i1 - v1] + cfa[i1 + v1]);
              sumsqh += SQ(ct - cfa[i1 - 1]) + SQ(ct - cfa[i1 + 1]);
              sumsqv += SQ(ct - cfa[i1 - v1]) + SQ(ct - cfa[i1 + v1]);
              areawt += 1;
            }
        }
        sumh = sumcfa - XDIV2(sumh);
        sumv = sumcfa - XDIV2(sumv);
        areawt = XDIV2(areawt);
        const float hcdvar = epssq + fabsf(areawt * sumsqh - sumh * sumh);
        const float vcdvar = epssq + fabsf(areawt * sumsqv - sumv * sumv);
        hvwt[i >> 1] = hcdvar / (vcdvar + hcdvar);
      }
      END_LOOP
    }
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- hvwt refined in place, row after row (:893-899); then green at R/B sites (:901-911) ---------------------
    // (the half plane is staged in shared memory: 144 dependent rows at shared-memory latency, three warps and a named barrier)
    stage_in(s_half, hvwt, tid);
    __syncthreads();
    if(tid < ROW_T)
      for(int rr = 8; rr < rr1 - 8; rr++)
      {
        const int i = rr * TS + 8 + (fc(rr, 2, f) & 1) + 2 * tid;
        if(tid < TSH && i < rr * TS + cc1 - 8)
        {
          const float hvwtalt = XDIV4(s_half[(i - m1) >> 1] + s_half[(i + p1) >> 1] + s_half[(i - p1) >> 1] + s_half[(i + m1) >> 1]);
          const float cur = s_half[i >> 1];
          s_half[i >> 1] = fabsf(0.5f - cur) < fabsf(0.5f - hvwtalt) ? hvwtalt : cur;
        }
        row_barrier();
      }
    __syncthreads();
    stage_out(hvwt, s_half, tid);
    __syncthreads();
    AMAZE_PROF_MARK(); // hvwt rows done
    SITE_LOOP(8)
    Dgrb0[i >> 1] = mixf(hvwt[i >> 1], vcd[i], hcd[i]);
    const float g = cfa[i] + Dgrb0[i >> 1];
    rgbgreen[i] = g;
    // rgbgreen at the four neighbours is still the raw value there (green sites are never written)
    Dgrb2[i >> 1].h = nyquist2[i >> 1] ? SQ(g - XDIV2(rgbgreen[i - 1] + rgbgreen[i + 1])) : 0.f;
    Dgrb2[i >> 1].v = nyquist2[i >> 1] ? SQ(g - XDIV2(rgbgreen[i - v1] + rgbgreen[i + v1])) : 0.f;
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- Nyquist refinement with green curvatures, :918-955 ------------------------------------------------------
    if(doNyquist)
    {
      NYQ_LOOP
      if(nyquist2[i >> 1])
      {
        const float gvarh
            = epssq
              + (gquinc[0] * Dgrb2[i >> 1].h + gquinc[1] * (Dgrb2[(i - m1) >> 1].h + Dgrb2[(i + p1) >> 1].h + Dgrb2[(i - p1) >> 1].h + Dgrb2[(i + m1) >> 1].h)
                 + gquinc[2] * (Dgrb2[(i - v2) >> 1].h + Dgrb2[(i - 2) >> 1].h + Dgrb2[(i + 2) >> 1].h + Dgrb2[(i + v2) >> 1].h)
                 + gquinc[3] * (Dgrb2[(i - m2) >> 1].h + Dgrb2[(i + p2) >> 1].h + Dgrb2[(i - p2) >> 1].h + Dgrb2[(i + m2) >> 1].h));
        const float gvarv
            = epssq
              + (gquinc[0] * Dgrb2[i >> 1].v + gquinc[1] * (Dgrb2[(i - m1) >> 1].v + Dgrb2[(i + p1) >> 1].v + Dgrb2[(i - p1) >> 1].v + Dgrb2[(i + m1) >> 1].v)
                 + gquinc[2] * (Dgrb2[(i - v2) >> 1].v + Dgrb2[(i - 2) >> 1].v + Dgrb2[(i + 2) >> 1].v + Dgrb2[(i + v2) >> 1].v)
                 + gquinc[3] * (Dgrb2[(i - m2) >> 1].v + Dgrb2[(i + p2) >> 1].v + Dgrb2[(i - p2) >> 1].v + Dgrb2[(i + m2) >> 1].v));
        Dgrb0[i >> 1] = (hcd[i] * gvarv + vcd[i] * gvarh) / (gvarv + gvarh);
        rgbgreen[i] = cfa[i] + Dgrb0[i >> 1];
      }
      END_LOOP
    }
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- diagonal gradients, :957-981 (delp/delm/Dgrbsq1* take over cddiffsq / delm / their own planes) ------------
    for(int rr = 6 + y8; rr < rr1 - 6; rr += RG8)
    {
      const int cc = 6 + 2 * x80;
      if(cc < cc1 - 6)
      {
        const int i = rr * TS + cc;
        if((fc(rr, 2, f) & 1) == 0)
        {
          delp[i >> 1] = fabsf(cfa[i + p1] - cfa[i - p1]);
          delm[i >> 1] = fabsf(cfa[i + m1] - cfa[i - m1]);
          Dgrbsq1p[i >> 1] = (SQ(cfa[i + 1] - cfa[i + 1 - p1]) + SQ(cfa[i + 1] - cfa[i + 1 + p1]));
          Dgrbsq1m[i >> 1] = (SQ(cfa[i + 1] - cfa[i + 1 - m1]) + SQ(cfa[i + 1] - cfa[i + 1 + m1]));
        }
        else
        {
          Dgrbsq1p[i >> 1] = (SQ(cfa[i] - cfa[i - p1]) + SQ(cfa[i] - cfa[i + p1]));
          Dgrbsq1m[i >> 1] = (SQ(cfa[i] - cfa[i - m1]) + SQ(cfa[i] - cfa[i + m1]));
          delp[i >> 1] = fabsf(cfa[i + 1 + p1] - cfa[i + 1 - p1]);
          delm[i >> 1] = fabsf(cfa[i + 1 + m1] - cfa[i + 1 - m1]);
        }
      }
    }
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- diagonal interpolation of the opposite colour, :986-1104 (rbm/rbp take over vcd, pmwt takes delhvsqsum) ----
    SITE_LOOP(8)
    const int j = i >> 1;
    const float crse = XMUL2(cfa[i + m1]) / (eps + cfa[i] + (cfa[i + m2]));
    const float crnw = XMUL2(cfa[i - m1]) / (eps + cfa[i] + (cfa[i - m2]));
    const float crne = XMUL2(cfa[i + p1]) / (eps + cfa[i] + (cfa[i + p2]));
    const float crsw = XMUL2(cfa[i - p1]) / (eps + cfa[i] + (cfa[i - p2]));
    const float rbse = (fabsf(1.f - crse) < arthresh) ? cfa[i] * crse : (cfa[i + m1]) + XDIV2(cfa[i] - cfa[i + m2]);
    const float rbnw = (fabsf(1.f - crnw) < arthresh) ? cfa[i] * crnw : (cfa[i - m1]) + XDIV2(cfa[i] - cfa[i - m2]);
    const float rbne = (fabsf(1.f - crne) < arthresh) ? cfa[i] * crne : (cfa[i + p1]) + XDIV2(cfa[i] - cfa[i + p2]);
    const float rbsw = (fabsf(1.f - crsw) < arthresh) ? cfa[i] * crsw : (cfa[i - p1]) + XDIV2(cfa[i] - cfa[i - p2]);
    const float wtse = eps + delm[j] + delm[(i + m1) >> 1] + delm[(i + m2) >> 1];
    const float wtnw = eps + delm[j] + delm[(i - m1) >> 1] + delm[(i - m2) >> 1];
    const float wtne = eps + delp[j] + delp[(i + p1) >> 1] + delp[(i + p2) >> 1];
    const float wtsw = eps + delp[j] + delp[(i - p1) >> 1] + delp[(i - p2) >> 1];
    float rm = (wtse * rbnw + wtnw * rbse) / (wtse + wtnw);
    float rp = (wtne * rbsw + wtsw * rbne) / (wtne + wtsw);
    const float rbvarm
        = epssq
          + (gausseven[0] * (Dgrbsq1m[(i - v1) >> 1] + Dgrbsq1m[(i - 1) >> 1] + Dgrbsq1m[(i + 1) >> 1] + Dgrbsq1m[(i + v1) >> 1])
             + gausseven[1]
                   * (Dgrbsq1m[(i - v2 - 1) >> 1] + Dgrbsq1m[(i - v2 + 1) >> 1] + Dgrbsq1m[(i - 2 - v1) >> 1] + Dgrbsq1m[(i + 2 - v1) >> 1]
                      + Dgrbsq1m[(i - 2 + v1) >> 1] + Dgrbsq1m[(i + 2 + v1) >> 1] + Dgrbsq1m[(i + v2 - 1) >> 1] + Dgrbsq1m[(i + v2 + 1) >> 1]));
    const float pw = rbvarm
                     / ((epssq
                         + (gausseven[0] * (Dgrbsq1p[(i - v1) >> 1] + Dgrbsq1p[(i - 1) >> 1] + Dgrbsq1p[(i + 1) >> 1] + Dgrbsq1p[(i + v1) >> 1])
                            + gausseven[1]
                                  * (Dgrbsq1p[(i - v2 - 1) >> 1] + Dgrbsq1p[(i - v2 + 1) >> 1] + Dgrbsq1p[(i - 2 - v1) >> 1] + Dgrbsq1p[(i + 2 - v1) >> 1]
                                     + Dgrbsq1p[(i - 2 + v1) >> 1] + Dgrbsq1p[(i + 2 + v1) >> 1] + Dgrbsq1p[(i + v2 - 1) >> 1]
                                     + Dgrbsq1p[(i + v2 + 1) >> 1])))
                        + rbvarm);
    if(rp < cfa[i])
    {
      if(XMUL2(rp) < cfa[i])
        rp = ULIMF(rp, cfa[i - p1], cfa[i + p1]);
      else
      {
        const float pwt = XMUL2(cfa[i] - rp) / (eps + rp + cfa[i]);
        rp = pwt * rp + (1.f - pwt) * ULIMF(rp, cfa[i - p1], cfa[i + p1]);
      }
    }
    if(rm < cfa[i])
    {
      if(XMUL2(rm) < cfa[i])
        rm = ULIMF(rm, cfa[i - m1], cfa[i + m1]);
      else
      {
        const float mwt = XMUL2(cfa[i] - rm) / (eps + rm + cfa[i]);
        rm = mwt * rm + (1.f - mwt) * ULIMF(rm, cfa[i - m1], cfa[i + m1]);
      }
    }
    if(rp > clip_pt) rp = ULIMF(rp, cfa[i - p1], cfa[i + p1]);
    if(rm > clip_pt) rm = ULIMF(rm, cfa[i - m1], cfa[i + m1]);
    rbm[j] = rm;
    rbp[j] = rp;
    pmwt[j] = pw;
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- pmwt refined in place, row after row (:1111-1118); then R+B (:1120-1121) ---------------------------------
    stage_in(s_half, pmwt, tid);
    __syncthreads();
    if(tid < ROW_T)
      for(int rr = 10; rr < rr1 - 10; rr++)
      {
        const int i = rr * TS + 10 + (fc(rr, 2, f) & 1) + 2 * tid;
        if(tid < TSH && i < rr * TS + cc1 - 10)
        {
          const float pmwtalt = XDIV4(s_half[(i - m1) >> 1] + s_half[(i + p1) >> 1] + s_half[(i - p1) >> 1] + s_half[(i + m1) >> 1]);
          if(fabsf(0.5f - s_half[i >> 1]) < fabsf(0.5f - pmwtalt)) s_half[i >> 1] = pmwtalt;
        }
        row_barrier();
      }
    __syncthreads();
    stage_out(pmwt, s_half, tid);
    __syncthreads();
    AMAZE_PROF_MARK(); // pmwt rows done
    SITE_LOOP(10)
    const int j = i >> 1;
    rbint[j] = XDIV2(cfa[i] + rbm[j] * (1.f - pmwt[j]) + rbp[j] * pmwt[j]);
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- green re-interpolated where the diagonal direction discriminates better, :1127-1241 ----------------------
    SITE_LOOP(12)
    const int j = i >> 1;
    if(!(fabsf(0.5f - pmwt[i >> 1]) < fabsf(0.5f - hvwt[i >> 1])))
    {
      const float cru = (float)((double)cfa[i - v1] * 2.0 / (double)(eps + rbint[j] + rbint[(j - v1)]));
      const float crd = (float)((double)cfa[i + v1] * 2.0 / (double)(eps + rbint[j] + rbint[(j + v1)]));
      const float crl = (float)((double)cfa[i - 1] * 2.0 / (double)(eps + rbint[j] + rbint[(j - 1)]));
      const float crr = (float)((double)cfa[i + 1] * 2.0 / (double)(eps + rbint[j] + rbint[(j + 1)]));
      const float gu = (fabsf(1.f - cru) < arthresh) ? rbint[j] * cru : cfa[i - v1] + XDIV2(rbint[j] - rbint[(j - v1)]);
      const float gd = (fabsf(1.f - crd) < arthresh) ? rbint[j] * crd : cfa[i + v1] + XDIV2(rbint[j] - rbint[(j + v1)]);
      const float gl = (fabsf(1.f - crl) < arthresh) ? rbint[j] * crl : cfa[i - 1] + XDIV2(rbint[j] - rbint[(j - 1)]);
      const float gr = (fabsf(1.f - crr) < arthresh) ? rbint[j] * crr : cfa[i + 1] + XDIV2(rbint[j] - rbint[(j + 1)]);
      float Gintv = (dirwts0[i - v1] * gd + dirwts0[i + v1] * gu) / (dirwts0[i + v1] + dirwts0[i - v1]);
      float Ginth = (dirwts1[i - 1] * gr + dirwts1[i + 1] * gl) / (dirwts1[i - 1] + dirwts1[i + 1]);
      if(Gintv < rbint[j])
      {
        if(2 * Gintv < rbint[j])
          Gintv = ULIMF(Gintv, cfa[i - v1], cfa[i + v1]);
        else
        {
          const float vwt = (float)(2.0 * (double)(rbint[j] - Gintv) / (double)(eps + Gintv + rbint[j]));
          Gintv = vwt * Gintv + (1.f - vwt) * ULIMF(Gintv, cfa[i - v1], cfa[i + v1]);
        }
      }
      if(Ginth < rbint[j])
      {
        if(2 * Ginth < rbint[j])
          Ginth = ULIMF(Ginth, cfa[i - 1], cfa[i + 1]);
        else
        {
          const float hwt = (float)(2.0 * (double)(rbint[j] - Ginth) / (double)(eps + Ginth + rbint[j]));
          Ginth = hwt * Ginth + (1.f - hwt) * ULIMF(Ginth, cfa[i - 1], cfa[i + 1]);
        }
      }
      if(Ginth > clip_pt) Ginth = ULIMF(Ginth, cfa[i - 1], cfa[i + 1]);
      if(Gintv > clip_pt) Gintv = ULIMF(Gintv, cfa[i - v1], cfa[i + v1]);
      const float g = Ginth * (1.f - hvwt[j]) + Gintv * hvwt[j];
      rgbgreen[i] = g;
      Dgrb0[i >> 1] = g - cfa[i];
    }
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- chroma: split G-B out of G-R (:1247-1253) ------------------------------------------------------------------
    for(int rr = 13 - a.ey + 2 * y8; rr < rr1 - 12; rr += 2 * RG8)
    {
      const int j = ((rr * TS + 13 - a.ex) >> 1) + x80;
      if(j < ((rr * TS + cc1 - 12) >> 1))
      {
        Dgrb1[j] = Dgrb0[j];
        Dgrb0[j] = 0;
      }
    }
    __syncthreads();
    AMAZE_PROF_MARK();
    // ---- ... and interpolate each at the other colour's sites from its diagonal neighbours (:1255-1289) -------------
    SITE_LOOP(14)
    const int c = 1 - fc(rr, cc, f) / 2;
    float *const D = c ? Dgrb1 : Dgrb0;
    const float wtnw = 1.f / (eps + fabsf(D[(i - m1) >> 1] - D[(i + m1) >> 1]) + fabsf(D[(i - m1) >> 1] - D[(i - m3) >> 1]) + fabsf(D[(i + m1) >> 1] - D[(i - m3) >> 1]));
    const float wtne = 1.f / (eps + fabsf(D[(i + p1) >> 1] - D[(i - p1) >> 1]) + fabsf(D[(i + p1) >> 1] - D[(i + p3) >> 1]) + fabsf(D[(i - p1) >> 1] - D[(i + p3) >> 1]));
    const float wtsw = 1.f / (eps + fabsf(D[(i - p1) >> 1] - D[(i + p1) >> 1]) + fabsf(D[(i - p1) >> 1] - D[(i + m3) >> 1]) + fabsf(D[(i + p1) >> 1] - D[(i - p3) >> 1]));
    const float wtse = 1.f / (eps + fabsf(D[(i + m1) >> 1] - D[(i - m1) >> 1]) + fabsf(D[(i + m1) >> 1] - D[(i - p3) >> 1]) + fabsf(D[(i - m1) >> 1] - D[(i + m3) >> 1]));
    D[i >> 1] = (wtnw * (1.325f * D[(i - m1) >> 1] - 0.175f * D[(i - m3) >> 1] - 0.075f * D[(i - m1 - 2) >> 1] - 0.075f * D[(i - m1 - v2) >> 1])
                 + wtne * (1.325f * D[(i + p1) >> 1] - 0.175f * D[(i + p3) >> 1] - 0.075f * D[(i + p1 + 2) >> 1] - 0.075f * D[(i + p1 + v2) >> 1])
                 + wtsw * (1.325f * D[(i - p1) >> 1] - 0.175f * D[(i - p3) >> 1] - 0.075f * D[(i - p1 - 2) >> 1] - 0.075f * D[(i - p1 - v2) >> 1])
                 + wtse * (1.325f * D[(i + m1) >> 1] - 0.175f * D[(i + m3) >> 1] - 0.075f * D[(i + m1 + 2) >> 1] - 0.075f * D[(i + m1 + v2) >> 1]))
                / (wtnw + wtne + wtsw + wtse);
    END_LOOP
    __syncthreads();

    AMAZE_PROF_MARK();
    // ---- output, :1291-1407: alpha is not written by the reference; 0 here ------------------------------------------
    FULL_LOOP(16)
    const int row = rr + top, col = cc + left;
    if(col < width && row < height)
    {
      const bool at_green = (((fc(rr, 2, f) & 1) == 1) ^ (((cc - 16) & 1) != 0));
      float r, b;
      if(at_green)
      {
        const float temp = 1.f / (hvwt[(i - v1) >> 1] + 2.f - hvwt[(i + 1) >> 1] - hvwt[(i - 1) >> 1] + hvwt[(i + v1) >> 1]);
        r = clampnan(rgbgreen[i]
                         - ((hvwt[(i - v1) >> 1]) * Dgrb0[(i - v1) >> 1] + (1.f - hvwt[(i + 1) >> 1]) * Dgrb0[(i + 1) >> 1]
                            + (1.f - hvwt[(i - 1) >> 1]) * Dgrb0[(i - 1) >> 1] + (hvwt[(i + v1) >> 1]) * Dgrb0[(i + v1) >> 1])
                               * temp,
                     0.0f, 1.0f);
        b = clampnan(rgbgreen[i]
                         - ((hvwt[(i - v1) >> 1]) * Dgrb1[(i - v1) >> 1] + (1.f - hvwt[(i + 1) >> 1]) * Dgrb1[(i + 1) >> 1]
                            + (1.f - hvwt[(i - 1) >> 1]) * Dgrb1[(i - 1) >> 1] + (hvwt[(i + v1) >> 1]) * Dgrb1[(i + v1) >> 1])
                               * temp,
                     0.0f, 1.0f);
      }
      else
      {
        r = clampnan(rgbgreen[i] - Dgrb0[i >> 1], 0.0f, 1.0f);
        b = clampnan(rgbgreen[i] - Dgrb1[i >> 1], 0.0f, 1.0f);
      }
      __stcs(reinterpret_cast<float4 *>(a.out + 4 * ((size_t)row * width + col)), make_float4(r, clampnan(rgbgreen[i], 0.0f, 1.0f), b, 0.0f));
    }
    END_LOOP
    AMAZE_PROF_MARK();
  }
}
} // namespace

namespace b200
{
int sm_count();
// amaze_demosaic_RT(), amaze.cc:181-1419.  `filters` already carries the ROI phase.
int amaze_demosaic_dev(const float *d_in, float *d_out, int width, int height, uint32_t filters, const float processed_maximum[3], cudaStream_t stream)
{
  if(width < 1 || height < 1) return B200_OK;
  // the mirrored border reads rows / columns up to 32 (:363,:414): smaller frames are out-of-bounds reads in the reference
  if(width < 33 || height < 33) return fail(B200_ERR_UNSUPPORTED, "AMaZE: frames under 33 px a side are undefined in the reference");
  // the sweeps below take the colour of a site from its row and column parity
  for(int r = 0; r < 8; r++)
    for(int c = 0; c < 2; c++)
      if(b200_fc(r, c, filters) != b200_fc(r & 1, c, filters))
        return fail(B200_ERR_UNSUPPORTED, "AMaZE: filters 0x%08x is not a 2x2 Bayer pattern", filters);
  amaze_args_t a;
  a.in = d_in;
  a.out = d_out;
  a.width = width;
  a.height = height;
  a.filters = filters;
  a.clip_pt = fminf(processed_maximum[0], fminf(processed_maximum[1], processed_maximum[2]));
  a.clip_pt8 = 0.8f * a.clip_pt;
  // tiles: top = -16 + k*128 < height, left likewise (:334-336)
  a.ntx = (width + 16 + (TS - 32) - 1) / (TS - 32);
  const int nty = (height + 16 + (TS - 32) - 1) / (TS - 32);
  a.ntiles = a.ntx * nty;
  // (ey, ex): offset of the R site in a Bayer quartet, :206-234
  if(b200_fc(0, 0, filters) == 1)
  {
    if(b200_fc(0, 1, filters) == 0)
    {
      a.ey = 0;
      a.ex = 1;
    }
    else
    {
      a.ey = 1;
      a.ex = 0;
    }
  }
  else if(b200_fc(0, 0, filters) == 0)
  {
    a.ey = 0;
    a.ex = 0;
  }
  else
  {
    a.ey = 1;
    a.ex = 1;
  }
  // persistent CTAs: as many as are resident at once (register-limited), each with its own scratch region
  static std::atomic<int> per_sm[16] = {}; // per device, 0 = not known yet; two threads may both find it, the same way
  int dev = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  int resident = per_sm[dev & 15].load(std::memory_order_acquire);
  if(!resident)
  {
    B200_CUDA_TRY(cudaFuncSetAttribute(amaze_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HALF));
    int n = 0;
    B200_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, amaze_tiles_kernel, NT, HALF));
    resident = n < 1 ? 1 : n;
    per_sm[dev & 15].store(resident, std::memory_order_release);
  }
  int grid = resident * sm_count();
  if(grid > a.ntiles) grid = a.ntiles;
  void *scr = nullptr;
  int rc = scratch(SLOT_TMP2, (size_t)grid * SCRATCH_STRIDE, &scr);
  if(rc) return rc;
  a.scratch = (char *)scr;
  amaze_tiles_kernel<<<grid, NT, HALF, stream>>>(a);
  B200_CUDA_TRY(cudaGetLastError());
  return B200_OK;
}
} // namespace b200

#ifdef B200_AMAZE_PROF
extern "C" int b200_amaze_prof(unsigned long long *out, int n, int reset)
{
  unsigned long long z[40] = { 0 };
  if(out && cudaMemcpyFromSymbol(out, g_amaze_prof, sizeof(unsigned long long) * (n < 40 ? n : 40)) != cudaSuccess) return 1;
  if(reset && cudaMemcpyToSymbol(g_amaze_prof, z, sizeof(z)) != cudaSuccess) return 1;
  return 0;
}
#endif
