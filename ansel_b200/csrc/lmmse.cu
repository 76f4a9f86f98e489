// LMMSE demosaic (L. Zhang, X. Wu; RawTherapee's implementation as tiled for darktable) for B200 / sm_100a.
//
// What the reference computes: src/iop/demosaic/lmmse.c lmmse_demosaic :136-576 (limf :67-70, median3f :72-75, median9f :77-121,
// calc_gamma :123-135); the two gamma tables it works in: iop/demosaic.c:1208-1213 (double precision exp / log on the host).
// What shapes the kernel:
//   * the reference walks tiles of 136x136 (128 of input + a margin of 4; 8 more on every side overlap the neighbours, 112 kept) on six
//     planes it zeroes ONCE per thread and carries from tile to tile.  A tile reads places it never writes (the two outermost rows /
//     columns of the difference planes, row / column 0 of the median planes, everything behind a short last tile), so in the reference
//     about a tenth of the pixels -- the tile seams and the frame's rim -- depend on which tile the thread ran before
//     (tests/test_cpu_lmmse.py measures it).  Here every tile starts from zeroed planes: a tile is a function of its input alone.
//     Parity contract: bit-identical to oracle/restate/lmmse_oracle.c in that mode (carry = 0); the same oracle with the planes carried
//     through the serial raster walk is bit-identical to the reference's lines compiled without OpenMP;
//   * one CTA per tile at a time, twelve stages with a __syncthreads between them, every stage one thread per site: the in-place updates
//     of the reference (bilinear red / blue, the median rebuild, the three refinement sweeps) each read only what earlier stages wrote
//     (checked thread by thread in both orders on the CPU);
//   * the six planes of a tile (444 KB) live in per-CTA scratch in global memory: 148 CTAs x 444 KB = 66 MB, L2 resident.
// Algorithmic bytes: 20 B/px (SURVEY.md 8d).
#ifndef B200_KERNELS_ON_CPU // tests/emul compiles the stages of this file with g++ to check them against the oracle without a GPU
#include "runtime.h"
#include <atomic>
#include <mutex>
#endif
#include <math.h>
#include <string.h>

namespace
{
constexpr int GRP = 136, BORDER = 4, OVERLAP = 8, TILESIZE = GRP - 2 * BORDER, TILEVALID = TILESIZE - 2 * OVERLAP, NP = GRP * GRP;
constexpr int LM_NT = 1024;

struct lm_args_t
{
  const float *in;
  float4 *out;
  float *scratch;                   // 6 * NP floats per CTA
  const float *gamma_in, *gamma_out; // 65536 floats each
  int width, height, nv, nh, medians, refine;
  unsigned filters;
  float scaler, revscaler, h0, h1, h2, h3, h4;
};
struct lm_tile_t
{
  int tv, th, rowStart, colStart, tileRows, tileCols, last_rr, last_cc, ccmin, ccmax, rrmin, rrmax;
};

__device__ __forceinline__ int lm_fc(int row, int col, unsigned f) { return (f >> ((((row << 1) & 14) + (col & 1)) << 1)) & 3; }
__device__ __forceinline__ float lm_limf(float x, float mn, float mx) { return fmaxf(mn, fminf(x, mx)); }
__device__ __forceinline__ float lm_median3(float x0, float x1, float x2) { return fmaxf(fminf(x0, x1), fminf(x2, fmaxf(x0, x1))); }
// :77-121, the network as the reference wrote it
__device__ __forceinline__ float lm_median9(float a0, float a1, float a2, float a3, float a4, float a5, float a6, float a7, float a8)
{
  float t;
  t = fminf(a1, a2); a2 = fmaxf(a1, a2); a1 = t;
  t = fminf(a4, a5); a5 = fmaxf(a4, a5); a4 = t;
  t = fminf(a7, a8); a8 = fmaxf(a7, a8); a7 = t;
  t = fminf(a0, a1); a1 = fmaxf(a0, a1); a0 = t;
  t = fminf(a3, a4); a4 = fmaxf(a3, a4); a3 = t;
  t = fminf(a6, a7); a7 = fmaxf(a6, a7); a6 = t;
  t = fminf(a1, a2); a2 = fmaxf(a1, a2); a1 = t;
  t = fminf(a4, a5); a5 = fminf(a4, a5); a4 = t; // :101: both the minimum
  t = fminf(a7, a8); a8 = fmaxf(a7, a8);
  a3 = fmaxf(a0, a3);
  a5 = fminf(a5, a8);
  a7 = fmaxf(a4, t);
  t = fminf(a4, t);
  a6 = fmaxf(a3, a6);
  a4 = fmaxf(a1, t);
  a2 = fminf(a2, a5);
  a4 = fminf(a4, a7);
  t = fminf(a4, a2);
  a2 = fmaxf(a4, a2);
  a4 = fmaxf(a6, t);
  return fminf(a4, a2);
}
__device__ __forceinline__ float lm_gamma(float val, const float *table)
{ // calc_gamma, :123-135
  const float index = val * 65535.0f;
  if(index < 0.0f) return 0.0f;
  if(index > 65534.99f) return 1.0f;
  const int idx = (int)index;
  const float diff = index - (float)idx;
  const float p1 = __ldg(table + idx);
  const float p2 = __ldg(table + idx + 1) - p1;
  return p1 + p2 * diff;
}
__device__ __forceinline__ float lm_sq(float x) { return x * x; }
__device__ __forceinline__ float lm_div(float a, float b)
{ // IEEE division, opaque to nvcc's x / c -> x * (1 / c) rewrite under -ftz=true (labglue.cu: divc)
#ifdef B200_KERNELS_ON_CPU
  return a / b;
#else
  float q;
  asm("div.rn.ftz.f32 %0, %1, %2;" : "=f"(q) : "f"(a), "f"(b));
  return q;
#endif
}

__device__ __forceinline__ lm_tile_t lm_tile_of(const lm_args_t &a, int t)
{
  lm_tile_t T;
  T.tv = t / a.nh;
  T.th = t - T.tv * a.nh;
  T.rowStart = T.tv * TILEVALID;
  T.colStart = T.th * TILEVALID;
  T.tileRows = min(T.rowStart + TILESIZE, a.height) - T.rowStart;
  T.tileCols = min(T.colStart + TILESIZE, a.width) - T.colStart;
  T.last_rr = T.tileRows + 2 * BORDER;
  T.last_cc = T.tileCols + 2 * BORDER;
  T.ccmin = T.th == 0 ? 6 : 0; // :365-370
  T.ccmax = T.last_cc - (T.th == a.nh - 1 ? 6 : 0);
  T.rrmin = T.tv == 0 ? 6 : 0;
  T.rrmax = T.last_rr - (T.tv == a.nv - 1 ? 6 : 0);
  return T;
}

// stage 0: the planes cleared, the gamma-encoded mosaic into plane 5 (:191-200)
__device__ void lm_load(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  for(int i = tid; i < 6 * NP; i += nt) Q[i] = 0.0f;
}
__device__ void lm_encode(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  for(int i = tid; i < T.tileRows * T.tileCols; i += nt)
  {
    const int r = i / T.tileCols, c = i - r * T.tileCols;
    Q[5 * NP + (r + BORDER) * GRP + c + BORDER] = lm_gamma(a.revscaler * __ldg(a.in + (size_t)(T.rowStart + r) * a.width + T.colStart + c), a.gamma_in);
  }
}
// stage 1: G - R(B) along rows (plane 0) and columns (plane 1), :202-236
__device__ void lm_differences(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.last_rr - 4, nc = T.last_cc - 4;
  constexpr int w1 = GRP, w2 = 2 * GRP;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int rr = 2 + i / nc, cc = 2 + i % nc;
    const float *cfa = Q + 5 * NP + rr * GRP + cc;
    float h, v;
    if(((cc - 2) & 1) == (lm_fc(rr, 2, a.filters) & 1))
    { // red / blue site
      const float v0 = 0.0625f * (cfa[-w1 - 1] + cfa[-w1 + 1] + cfa[w1 - 1] + cfa[w1 + 1]) + 0.25f * cfa[0];
      h = -0.25f * (cfa[-2] + cfa[2]) + 0.5f * (cfa[-1] + cfa[0] + cfa[1]);
      const float Y0 = v0 + 0.5f * h;
      h = (cfa[0] > 1.75f * Y0) ? lm_median3(h, cfa[-1], cfa[1]) : lm_limf(h, 0.0f, 1.0f);
      h -= cfa[0];
      v = -0.25f * (cfa[-w2] + cfa[w2]) + 0.5f * (cfa[-w1] + cfa[0] + cfa[w1]);
      const float Y1 = v0 + 0.5f * v;
      v = (cfa[0] > 1.75f * Y1) ? lm_median3(v, cfa[-w1], cfa[w1]) : lm_limf(v, 0.0f, 1.0f);
      v -= cfa[0];
    }
    else
    { // green site
      h = 0.25f * (cfa[-2] + cfa[2]) - 0.5f * (cfa[-1] + cfa[0] + cfa[1]);
      v = 0.25f * (cfa[-w2] + cfa[w2]) - 0.5f * (cfa[-w1] + cfa[0] + cfa[w1]);
      h = lm_limf(h, -1.0f, 0.0f) + cfa[0];
      v = lm_limf(v, -1.0f, 0.0f) + cfa[0];
    }
    Q[rr * GRP + cc] = h;
    Q[NP + rr * GRP + cc] = v;
  }
}
// stage 2: their low pass into planes 2 and 3, :238-250
__device__ void lm_lowpass(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.last_rr - 8, nc = T.last_cc - 8;
  constexpr int w1 = GRP, w2 = 2 * GRP, w3 = 3 * GRP, w4 = 4 * GRP;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int p = (4 + i / nc) * GRP + 4 + i % nc;
    const float *hd = Q + p, *vd = Q + NP + p;
    Q[2 * NP + p] = a.h0 * hd[0] + a.h1 * (hd[-1] + hd[1]) + a.h2 * (hd[-2] + hd[2]) + a.h3 * (hd[-3] + hd[3]) + a.h4 * (hd[-4] + hd[4]);
    Q[3 * NP + p] = a.h0 * vd[0] + a.h1 * (vd[-w1] + vd[w1]) + a.h2 * (vd[-w2] + vd[w2]) + a.h3 * (vd[-w3] + vd[w3]) + a.h4 * (vd[-w4] + vd[w4]);
  }
}
// the variance-weighted estimate along one direction, :258-283
__device__ __forceinline__ void lm_estimate(const float *lp, const float *df, int s, float &x, float &v)
{
  float p[9];
#pragma unroll
  for(int k = 0; k < 9; k++) p[k] = lp[(k - 4) * s];
  const float mu = lm_div(p[0] + p[1] + p[2] + p[3] + p[4] + p[5] + p[6] + p[7] + p[8], 9.0f);
  float vx = 1e-7f;
#pragma unroll
  for(int k = 0; k < 9; k++) vx += lm_sq(p[k] - mu);
#pragma unroll
  for(int k = 0; k < 9; k++) p[k] -= df[(k - 4) * s];
  float vn = 1e-7f;
#pragma unroll
  for(int k = 0; k < 9; k++) vn += lm_sq(p[k]);
  x = (df[0] * vx + lp[0] * vn) / (vx + vn);
  v = vx * vn / (vx + vn);
}
// stage 3: the interpolated G - R(B) at red / blue sites into plane 4, :252-314
__device__ void lm_interpolate(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.last_rr - 8, nc = (T.last_cc - 8 + 1) / 2;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int rr = 4 + i / nc, cc = 4 + (lm_fc(rr, 4, a.filters) & 1) + 2 * (i % nc);
    if(cc >= T.last_cc - 4) continue;
    const int p = rr * GRP + cc;
    float xh, vh, xv, vv;
    lm_estimate(Q + 2 * NP + p, Q + p, 1, xh, vh);
    lm_estimate(Q + 3 * NP + p, Q + NP + p, GRP, xv, vv);
    Q[4 * NP + p] = (xh * vv + xv * vh) / (vh + vv);
  }
}
// stage 4: the colour planes: the mosaic in its own plane, green at red / blue sites, zero outside the frame (:316-336)
__device__ void lm_colours(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  for(int i = tid; i < T.last_rr * T.last_cc; i += nt)
  {
    const int rr = i / T.last_cc, cc = i - rr * T.last_cc, p = rr * GRP + cc;
    const int row_in = T.rowStart - BORDER + rr, col_in = T.colStart - BORDER + cc;
    const int c = lm_fc(rr, cc, a.filters);
    const bool inside = row_in >= 0 && row_in < a.height && col_in >= 0 && col_in < a.width;
    const float own = inside ? Q[5 * NP + p] : 0.0f;
    const float green = inside ? own + Q[4 * NP + p] : 0.0f; // plane 4 is read before plane 1 is written: other sites
    Q[c * NP + p] = own;
    if(c != 1) Q[NP + p] = green;
  }
}
// stage 5: red and blue at green sites from the colour differences of the row / column neighbours (:338-352)
__device__ void lm_rb_at_green(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.last_rr - 2, nc = (T.last_cc - 2 + 1) / 2;
  constexpr int w1 = GRP;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int rr = 1 + i / nc, cc = 1 + (lm_fc(rr, 2, a.filters) & 1) + 2 * (i % nc);
    if(cc >= T.last_cc - 1) continue;
    const int c = lm_fc(rr, cc + 1, a.filters), p = rr * GRP + cc;
    const float *g = Q + NP + p;
    float *q = Q + c * NP + p;
    q[0] = g[0] + 0.5f * (q[-1] - g[-1] + q[1] - g[1]);
    q = Q + (2 - c) * NP + p;
    q[0] = g[0] + 0.5f * (q[-w1] - g[-w1] + q[w1] - g[w1]);
  }
}
// stage 6: the opposite colour at red / blue sites from the four green neighbours' (:354-363)
__device__ void lm_rb_at_rb(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.last_rr - 2, nc = (T.last_cc - 2 + 1) / 2;
  constexpr int w1 = GRP;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int rr = 1 + i / nc, cc = 1 + (lm_fc(rr, 1, a.filters) & 1) + 2 * (i % nc);
    if(cc >= T.last_cc - 1) continue;
    const int c = 2 - lm_fc(rr, cc, a.filters), p = rr * GRP + cc;
    const float *g = Q + NP + p;
    float *q = Q + c * NP + p;
    q[0] = g[0] + 0.25f * (q[-w1] - g[-w1] + q[-1] - g[-1] + q[1] - g[1] + q[w1] - g[w1]);
  }
}
// stage 7a: 3x3 medians of R - G into plane 3 and of B - G into plane 4 (:377-397)
__device__ void lm_medians(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.last_rr - 2, nc = T.last_cc - 2;
  constexpr int w1 = GRP;
  for(int i = tid; i < 2 * nr * nc; i += nt)
  {
    const int k = i / (nr * nc), j = i - k * (nr * nc), p = (1 + j / nc) * GRP + 1 + j % nc;
    const float *q = Q + (2 * k) * NP + p, *g = Q + NP + p;
    Q[(3 + k) * NP + p] = lm_median9(q[-w1 - 1] - g[-w1 - 1], q[-w1] - g[-w1], q[-w1 + 1] - g[-w1 + 1], q[-1] - g[-1], q[0] - g[0], q[1] - g[1],
                                     q[w1 - 1] - g[w1 - 1], q[w1] - g[w1], q[w1 + 1] - g[w1 + 1]);
  }
}
// stage 7b: every site rebuilt from green and the medians (:399-477: the row walked in pairs from ccmin, a trailing single site with the
// pair's first operation: the operation of a site is that of its parity)
__device__ void lm_rebuild(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.rrmax - 1 - T.rrmin, nc = T.ccmax - T.ccmin;
  if(nr <= 0 || nc <= 0) return;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int rr = T.rrmin + i / nc, cc = T.ccmin + i % nc, p = rr * GRP + cc;
    const int c0 = lm_fc(rr, 0, a.filters), c1 = lm_fc(rr, 1, a.filters);
    const bool first = ((cc - T.ccmin) & 1) == 0;
    if((c0 == 1) == first)
    {
      const float g = Q[NP + p];
      Q[p] = g + Q[3 * NP + p];
      Q[2 * NP + p] = g + Q[4 * NP + p];
    }
    else
    {
      const int c = c0 == 1 ? 2 - c1 : 2 - c0, d = c + 3 - (c == 0 ? 0 : 1);
      Q[c * NP + p] = Q[NP + p] + Q[d * NP + p];
      Q[NP + p] = 0.5f * (Q[p] - Q[3 * NP + p] + Q[2 * NP + p] - Q[4 * NP + p]);
    }
  }
}
// stage 8: the mosaic back into its own plane (:480-489)
__device__ void lm_restore(const lm_args_t &a, const lm_tile_t &T, float *Q, int tid, int nt)
{
  const int nr = T.last_rr - 8, nc = T.last_cc - 8;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int rr = 4 + i / nc, cc = 4 + i % nc, p = rr * GRP + cc;
    Q[lm_fc(rr, cc, a.filters) * NP + p] = Q[5 * NP + p];
  }
}
// stage 9: the three sweeps of a refinement step (:494-545); which = 0 green at red / blue sites, 1 red and blue at green sites, 2 the
// opposite colour at red / blue sites
__device__ void lm_refine(const lm_args_t &a, const lm_tile_t &T, float *Q, int which, int tid, int nt)
{
  const int nr = T.rrmax - 2 - (T.rrmin + 2), nc = (T.ccmax - 2 - (T.ccmin + 2) + 1) / 2;
  if(nr <= 0 || nc <= 0) return;
  constexpr int w1 = GRP, w2 = 2 * GRP;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int rr = T.rrmin + 2 + i / nc;
    const int par = which == 1 ? (lm_fc(rr, 3, a.filters) & 1) : (lm_fc(rr, 2, a.filters) & 1);
    const int cc = T.ccmin + 2 + par + 2 * (i % nc);
    if(cc >= T.ccmax - 2) continue;
    const int p = rr * GRP + cc;
    float *g = Q + NP + p;
    if(which == 0)
    {
      const float *q = Q + lm_fc(rr, cc, a.filters) * NP + p;
      const float dL = 1.0f / (1.0f + fabsf(q[-2] - q[0]) + fabsf(g[1] - g[-1])), dR = 1.0f / (1.0f + fabsf(q[2] - q[0]) + fabsf(g[1] - g[-1]));
      const float dU = 1.0f / (1.0f + fabsf(q[-w2] - q[0]) + fabsf(g[w1] - g[-w1])), dD = 1.0f / (1.0f + fabsf(q[w2] - q[0]) + fabsf(g[w1] - g[-w1]));
      g[0] = (q[0] + ((g[-1] - q[-1]) * dL + (g[1] - q[1]) * dR + (g[-w1] - q[-w1]) * dU + (g[w1] - q[w1]) * dD) / (dL + dR + dU + dD));
    }
    else if(which == 1)
    {
      int c = lm_fc(rr, cc + 1, a.filters);
#pragma unroll
      for(int k = 0; k < 2; k++, c = 2 - c)
      {
        float *q = Q + c * NP + p;
        const float dL = 1.0f / (1.0f + fabsf(g[-2] - g[0]) + fabsf(q[1] - q[-1])), dR = 1.0f / (1.0f + fabsf(g[2] - g[0]) + fabsf(q[1] - q[-1]));
        const float dU = 1.0f / (1.0f + fabsf(g[-w2] - g[0]) + fabsf(q[w1] - q[-w1])), dD = 1.0f / (1.0f + fabsf(g[w2] - g[0]) + fabsf(q[w1] - q[-w1]));
        q[0] = (g[0] - ((g[-1] - q[-1]) * dL + (g[1] - q[1]) * dR + (g[-w1] - q[-w1]) * dU + (g[w1] - q[w1]) * dD) / (dL + dR + dU + dD));
      }
    }
    else
    {
      const int c = 2 - lm_fc(rr, cc, a.filters);
      float *q = Q + c * NP + p;
      const float *e = Q + (2 - c) * NP + p;
      const float dL = 1.0f / (1.0f + fabsf(e[-2] - e[0]) + fabsf(g[1] - g[-1])), dR = 1.0f / (1.0f + fabsf(e[2] - e[0]) + fabsf(g[1] - g[-1]));
      const float dU = 1.0f / (1.0f + fabsf(e[-w2] - e[0]) + fabsf(g[w1] - g[-w1])), dD = 1.0f / (1.0f + fabsf(e[w2] - e[0]) + fabsf(g[w1] - g[-w1]));
      q[0] = (g[0] - ((g[-1] - q[-1]) * dL + (g[1] - q[1]) * dR + (g[-w1] - q[-w1]) * dU + (g[w1] - q[w1]) * dD) / (dL + dR + dU + dD));
    }
  }
}
// stage 10: the kept part of the tile, decoded (:548-570)
__device__ void lm_store(const lm_args_t &a, const lm_tile_t &T, const float *Q, int tid, int nt)
{
  const int rowEnd = T.rowStart + T.tileRows, colEnd = T.colStart + T.tileCols;
  const int first_v = T.rowStart + (T.tv == 0 ? 0 : OVERLAP), last_v = rowEnd - (T.tv == a.nv - 1 ? 0 : OVERLAP);
  const int first_h = T.colStart + (T.th == 0 ? 0 : OVERLAP), last_h = colEnd - (T.th == a.nh - 1 ? 0 : OVERLAP);
  const int nr = last_v - first_v, nc = last_h - first_h;
  if(nr <= 0 || nc <= 0) return;
  for(int i = tid; i < nr * nc; i += nt)
  {
    const int row = first_v + i / nc, col = first_h + i % nc;
    const int p = (row - T.rowStart + BORDER) * GRP + col - T.colStart + BORDER;
    a.out[(size_t)row * a.width + col] = make_float4(a.scaler * lm_gamma(Q[p], a.gamma_out), a.scaler * lm_gamma(Q[NP + p], a.gamma_out),
                                                       a.scaler * lm_gamma(Q[2 * NP + p], a.gamma_out), 0.0f);
  }
}

#ifndef B200_KERNELS_ON_CPU
__global__ void __launch_bounds__(LM_NT, 1) lmmse_tiles_kernel(const __grid_constant__ lm_args_t a)
{
  float *const Q = a.scratch + (size_t)blockIdx.x * 6 * NP;
  const int tid = threadIdx.x;
  for(int t = blockIdx.x; t < a.nv * a.nh; t += gridDim.x)
  {
    const lm_tile_t T = lm_tile_of(a, t);
    lm_load(a, T, Q, tid, LM_NT);
    __syncthreads();
    lm_encode(a, T, Q, tid, LM_NT);
    __syncthreads();
    lm_differences(a, T, Q, tid, LM_NT);
    __syncthreads();
    lm_lowpass(a, T, Q, tid, LM_NT);
    __syncthreads();
    lm_interpolate(a, T, Q, tid, LM_NT);
    __syncthreads();
    lm_colours(a, T, Q, tid, LM_NT);
    __syncthreads();
    lm_rb_at_green(a, T, Q, tid, LM_NT);
    __syncthreads();
    lm_rb_at_rb(a, T, Q, tid, LM_NT);
    __syncthreads();
    for(int pass = 0; pass < a.medians; pass++)
    {
      lm_medians(a, T, Q, tid, LM_NT);
      __syncthreads();
      lm_rebuild(a, T, Q, tid, LM_NT);
      __syncthreads();
    }
    lm_restore(a, T, Q, tid, LM_NT);
    __syncthreads();
    for(int step = 0; step < a.refine; step++)
      for(int which = 0; which < 3; which++)
      {
        lm_refine(a, T, Q, which, tid, LM_NT);
        __syncthreads();
      }
    lm_store(a, T, Q, tid, LM_NT);
    __syncthreads();
  }
}
#endif

// the plan: what lmmse_demosaic() sets up before its tile loop, :139-162
void lm_plan(lm_args_t &a, int width, int height, unsigned filters, int mode, const float processed_maximum[3])
{
  memset(&a, 0, sizeof(a));
  a.width = width;
  a.height = height;
  a.filters = filters;
  float h0 = 1.0f, h1 = expf(-1.0f / 8.0f), h2 = expf(-4.0f / 8.0f), h3 = expf(-9.0f / 8.0f), h4 = expf(-16.0f / 8.0f);
  const float hs = h0 + 2.0f * (h1 + h2 + h3 + h4);
  a.h0 = h0 / hs;
  a.h1 = h1 / hs;
  a.h2 = h2 / hs;
  a.h3 = h3 / hs;
  a.h4 = h4 / hs;
  a.medians = mode < 2 ? mode : 3;
  a.refine = mode > 2 ? mode - 2 : 0;
  a.scaler = fmaxf(processed_maximum[0], fmaxf(processed_maximum[1], processed_maximum[2]));
  a.revscaler = 1.0f / a.scaler;
  a.nv = 1 + (height - 2 * OVERLAP - 1) / TILEVALID;
  a.nh = 1 + (width - 2 * OVERLAP - 1) / TILEVALID;
}
// iop/demosaic.c:1208-1213: the gamma the method works in and its inverse, 65536 samples each, in double precision on the host
void lm_gamma_tables(float *gamma_in, float *gamma_out)
{
  for(int j = 0; j < 65536; j++)
  {
    const double x = (double)j / 65535.0;
    gamma_in[j] = (x <= 0.001867) ? x * 17.0 : 1.044445 * exp(log(x) / 2.4) - 0.044445;
    gamma_out[j] = (x <= 0.031746) ? x / 17.0 : exp(log((x + 0.044445) / 1.044445) * 2.4);
  }
}
} // namespace

#ifndef B200_KERNELS_ON_CPU
namespace b200
{
// lmmse_demosaic(), lmmse.c:136-576.  mode = dt_iop_demosaic_lmmse_t (data->lmmse_refine), filters with the ROI phase folded in.
int lmmse_demosaic_dev(const float *d_in, float *d_out, int width, int height, uint32_t filters, int mode, const float processed_maximum[3], cudaStream_t stream)
{
  if(width < 16 || height < 16) return B200_OK; // "too small area": the reference returns with the output untouched (:140-144)
  if(mode < 0 || mode > 4) return fail(B200_ERR_ARG, "LMMSE: refine mode %d", mode);
  for(int r = 0; r < 8; r++)
    for(int c = 0; c < 2; c++)
      if(b200_fc(r, c, filters) != b200_fc(r & 1, c, filters)) return fail(B200_ERR_UNSUPPORTED, "LMMSE: filters 0x%08x is not a 2x2 Bayer pattern", filters);
  int dev = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  // per device: gamma_in, gamma_out.  Made once under the lock and published only when uploaded, so no thread launches on
  // tables still being filled.
  static std::atomic<float *> d_tables[16] = {};
  static std::mutex tables_mu;
  float *tables = d_tables[dev & 15].load(std::memory_order_acquire);
  if(!tables)
  {
    std::lock_guard<std::mutex> lock(tables_mu);
    tables = d_tables[dev & 15].load(std::memory_order_acquire); // another thread may have made them meanwhile
    if(!tables)
    {
      float *h = (float *)malloc(2 * 65536 * sizeof(float));
      if(!h) return fail(B200_ERR_ARG, "LMMSE: out of host memory");
      lm_gamma_tables(h, h + 65536);
      float *d = nullptr;
      cudaError_t e = cudaMalloc(&d, 2 * 65536 * sizeof(float));
      if(e == cudaSuccess) e = cudaMemcpyAsync(d, h, 2 * 65536 * sizeof(float), cudaMemcpyHostToDevice, stream);
      if(e == cudaSuccess) e = cudaStreamSynchronize(stream); // complete before another thread's stream may read them
      free(h);
      if(e != cudaSuccess)
      {
        if(d) cudaFree(d);
        return fail(B200_ERR_CUDA, "LMMSE: gamma tables: %s", cudaGetErrorString(e));
      }
      tables = d;
      d_tables[dev & 15].store(tables, std::memory_order_release);
    }
  }
  lm_args_t a;
  lm_plan(a, width, height, filters, mode, processed_maximum);
  a.in = d_in;
  a.out = (float4 *)d_out;
  a.gamma_in = tables;
  a.gamma_out = tables + 65536;
  int grid = sm_count();
  if(grid > a.nv * a.nh) grid = a.nv * a.nh;
  void *scr = nullptr;
  int rc = scratch(SLOT_TMP2, (size_t)grid * 6 * NP * sizeof(float), &scr);
  if(rc) return rc;
  a.scratch = (float *)scr;
  lmmse_tiles_kernel<<<grid, LM_NT, 0, stream>>>(a);
  B200_CUDA_TRY(cudaGetLastError());
  return B200_OK;
}
} // namespace b200
#endif
