// Frank Markesteijn's demosaicer for X-Trans sensors, one and three passes, for B200 / sm_100a.
//
// What the reference computes: src/iop/demosaic/markesteijn.c xtrans_markesteijn_interpolate :47-521 with passes == 1 (the default
// demosaicer of every X-Trans frame, iop/demosaic.c:1085) and passes == 3 (eight directions, a border of 17, two more rounds that
// recompute green from the closer interpolated values).  Parity contract: bit-identical to that source under C float semantics
// (oracle/restate/markesteijn_oracle.c, pinned against the lines compiled in place).
// What shapes the kernel:
//   * the reference works in tiles of 122x122 with a border of 12, mirrored beyond the frame; every stage is local, but the first
//     one (bounds of green at the red/blue pairs, :199-246) depends on where a tile starts, so the tile grid is kept: one CTA
//     walks whole reference tiles, stage after stage, a __syncthreads between stages;
//   * that first stage is a loop that changes its own row counter to hop between the rows of a vertical pair and lets the last
//     visit of a pixel win.  Its control flow depends on the position and size of the tile only -- sixteen classes at most per
//     frame -- so the host replays it once per class (mk_walk) and ships, for every red/blue pixel, the pixel whose green
//     hexagon opened the run that wrote it last.  What the data decides (a run whose maximum came out as 0.0f starts over at its
//     second pixel) is decided in the kernel;
//   * everything else is one thread per pixel: four directional greens, red/blue at the solitary greens (a six-step recurrence
//     per pixel, in registers), red at blue and blue at red, the 2x2 green blocks (planes 0 and 1 only: the reference's loop
//     stops there with four directions), squared YPbPr differences, 3x3 homogeneity counts, 5x5 sums of those (the reference
//     rolls them in uint8 arithmetic: same sums), the average of the most homogeneous directions.
// Scratch per resident CTA, in global memory (L2): directions x 3 channels + one derivative plane per direction of 122x122 floats
// (952 KB with four directions, 1.9 MB with eight; the homogeneity counts, 14.9 KB per direction, live in shared memory).  Planes are split by direction and channel so that a
// warp reads consecutive floats.  Algorithmic bytes: 20 B/px (SURVEY.md 8d).
#ifndef B200_KERNELS_ON_CPU // tests/emul compiles the stages of this file with g++ to check them against the oracle without a GPU
#include "runtime.h"
#endif
#include <float.h>
#include <string.h>
#include <vector>
#include <atomic>

namespace
{
constexpr int TS = 122, NPX = TS * TS;
constexpr int MK_NT = 1024;
constexpr int MK_MAX_CLASSES = 20; // (first row, three phases, last row) x (three phases, last column)
// what the number of passes decides, :64, :106, :305, :357, :376, :419-452
template <int PASSES> struct mk_geo
{
  static constexpr int NDIR = PASSES > 1 ? 8 : 4, PAD = PASSES > 1 ? 17 : 12, STEP = TS - 2 * PAD;
  static constexpr int PLANES = 4 * NDIR; // colour planes (direction * 3 + channel), then one derivative plane per direction
  static constexpr int PAD_SG = PASSES > 1 ? 5 : 6, PAD_RB = PASSES > 1 ? 5 : 6, PAD_G22 = PASSES > 1 ? 4 : 8, PAD_YUV = PASSES > 1 ? 13 : 8;
};

struct mk_args_t
{
  const float *in;
  float4 *out;
  float *scratch;     // mk_geo::PLANES * NPX floats per CTA
  const short *start; // [class][NPX]: the record of the walk
  int width, height, ntx, ntiles, pad, step;
  int sgrow, sgcol;
  short hex[3][3][8];
  uint8_t xt[36];     // the sensor's pattern seen from the region's origin: xt[r][c] = xtrans[(r + roi.y) % 6][(c + roi.x) % 6]
  uint8_t cls_row[6], cls_col[6]; // class of a full tile by the phase of its origin; the last tile row / column: cls_last_*
  int cls_last_row, cls_last_col, cls_first_row, n_col_classes; // the first tile row is its own class: (row - sgrow) % 3 is negative above the frame
};

struct mk_tile_t
{
  int top, left, nrow, ncol, cls;
};

__host__ __device__ inline int mk_fc(const uint8_t *xt, int row, int col) { return xt[((row + 600) % 6) * 6 + (col + 600) % 6]; }
__device__ __forceinline__ const short *mk_hex(const mk_args_t &a, int row, int col) { return a.hex[(row + 600) % 3][(col + 600) % 3]; }
__device__ __forceinline__ int mk_mirror(int n, int size) { return n >= size ? 2 * size - n - 2 : (n < 0 ? -n : n); } // TRANSLATE, :158
__device__ __forceinline__ float mk_sqr(float x) { return x * x; }
__device__ __forceinline__ float mk_div(float a, float b)
{ // IEEE division, opaque to nvcc's x / c -> x * (1 / c) rewrite under -ftz=true (labglue.cu: divc); halving is exact either way
#ifdef B200_KERNELS_ON_CPU
  return a / b;
#else
  float q;
  asm("div.rn.ftz.f32 %0, %1, %2;" : "=f"(q) : "f"(a), "f"(b));
  return q;
#endif
}
__device__ __forceinline__ float mk_clamps(float v, float l, float h) { return v > l ? (v < h ? v : h) : l; } // CLAMPS, math/math.h:78

__device__ __forceinline__ mk_tile_t mk_tile_of(const mk_args_t &a, int t)
{
  mk_tile_t T;
  const int ty = t / a.ntx, tx = t - ty * a.ntx;
  T.top = -a.pad + ty * a.step;
  T.left = -a.pad + tx * a.step;
  T.nrow = min(TS, a.height + a.pad - T.top);
  T.ncol = min(TS, a.width + a.pad - T.left);
  const int rc = ty == 0 ? a.cls_first_row : (T.nrow == TS ? a.cls_row[(T.top + 600) % 6] : a.cls_last_row), cc = T.ncol == TS ? a.cls_col[(T.left + 600) % 6] : a.cls_last_col;
  T.cls = rc * a.n_col_classes + cc;
  return T;
}

// ---- stage 0, :139-186: the tile, mirrored beyond the frame, the same in all four directions -------------------------------
__device__ void mk_load(const mk_args_t &a, const mk_tile_t &T, float *P, int tid, int nt)
{
  for(int idx = tid; idx < T.nrow * T.ncol; idx += nt)
  {
    const int r = idx / T.ncol, c = idx - r * T.ncol, row = T.top + r, col = T.left + c;
    const int f = mk_fc(a.xt, row, col);
    float v;
    if(col >= 0 && row >= 0 && col < a.width && row < a.height)
      v = __ldg(a.in + (size_t)a.width * row + col);
    else
    {
      const int cy = mk_mirror(row, a.height), cx = mk_mirror(col, a.width);
      if(f == mk_fc(a.xt, cy, cx))
        v = __ldg(a.in + (size_t)a.width * cy + cx);
      else
      { // the mirror pixel has another colour: the mean of that colour over the mirrored 3x3
        float sum = 0.0f;
        int count = 0;
        for(int y = row - 1; y <= row + 1; y++)
          for(int x = col - 1; x <= col + 1; x++)
          {
            const int yy = mk_mirror(y, a.height), xx = mk_mirror(x, a.width);
            if(mk_fc(a.xt, yy, xx) == f)
            {
              sum += __ldg(a.in + (size_t)a.width * yy + xx);
              count++;
            }
          }
        v = sum / (float)count;
      }
    }
    const int p = r * TS + c;
#pragma unroll
    for(int d = 0; d < 4; d++)
    {
      P[(d * 3 + 0) * NPX + p] = f == 0 ? v : 0.0f;
      P[(d * 3 + 1) * NPX + p] = f == 1 ? v : 0.0f;
      P[(d * 3 + 2) * NPX + p] = f == 2 ? v : 0.0f;
    }
  }
}

// ---- stage 1, :199-271: bounds of green from the record of the walk, then green along the four directions --------------------
__device__ __forceinline__ void mk_minmax6(const float *G, const short *hex, float &mn, float &mx)
{
#pragma unroll
  for(int c = 0; c < 6; c++)
  {
    const float v = G[hex[c]];
    if(mn > v) mn = v;
    if(mx < v) mx = v;
  }
}
// the bounds of green of a red/blue pixel p (row, col), :203-231, from the record of the walk; G: plane 0, green
__device__ __forceinline__ void mk_bounds(const mk_args_t &a, const mk_tile_t &T, const float *G, const short *start, int p, const short *hex, float &mn, float &mx)
{
  mn = FLT_MAX;
  mx = 0.0f;
  const int s = start[p];
  if(s >= 0)
  {
    const int sr = s / TS, sc = s - sr * TS;
    mk_minmax6(G + s, mk_hex(a, T.top + sr, T.left + sc), mn, mx);
    if(s != p && mx == 0.0f) mk_minmax6(G + p, hex, mn, mx); // the loop's marker of a new pair: the second pixel goes on by itself
  }
}
__device__ void mk_green(const mk_args_t &a, const mk_tile_t &T, float *P, int tid, int nt)
{
  const int nr = T.nrow - 6, nc = T.ncol - 6;
  if(nr <= 0 || nc <= 0) return;
  const short *const start = a.start + (size_t)T.cls * NPX;
  const float *const G = P + 1 * NPX; // plane 0, green: the native greens
  for(int idx = tid; idx < nr * nc; idx += nt)
  {
    const int r = 3 + idx / nc, c = 3 + idx % nc, row = T.top + r, col = T.left + c;
    const int f = mk_fc(a.xt, row, col);
    if(f == 1) continue;
    const int p = r * TS + c;
    const short *const hex = mk_hex(a, row, col);
    float mn, mx;
    mk_bounds(a, T, G, start, p, hex, mn, mx);
    const float *const N = P + f * NPX + p; // plane 0, the pixel's own colour: natives
    const float *const g = G + p;
    float color[4];
    color[0] = 0.6796875f * (g[hex[1]] + g[hex[0]]) - 0.1796875f * (g[2 * hex[1]] + g[2 * hex[0]]);
    color[1] = 0.87109375f * g[hex[3]] + g[hex[2]] * 0.13f + 0.359375f * (N[0] - N[-hex[2]]);
#pragma unroll
    for(int k = 0; k < 2; k++)
      color[2 + k] = 0.640625f * g[hex[4 + k]] + 0.359375f * g[-2 * hex[4 + k]] + 0.12890625f * (2 * N[0] - N[3 * hex[4 + k]] - N[-3 * hex[4 + k]]);
    const int flip = !((row - a.sgrow) % 3);
#pragma unroll
    for(int k = 0; k < 4; k++) P[((k ^ flip) * 3 + 1) * NPX + p] = mk_clamps(color[k], mn, mx);
  }
}

// ---- stage 2, :304-354: red and blue at the solitary greens ---------------------------------------------------------------
// P: the first of the four direction planes the pass works on (planes 0-3 in the first pass, 4-7 afterwards); G0: plane 0's green
__device__ void mk_solitary(const mk_args_t &a, const mk_tile_t &T, float *P, int pad, int tid, int nt)
{
  const int mrow = T.top + T.nrow, mcol = T.left + T.ncol;
  const int row0 = (T.top - a.sgrow + pad + 2) / 3 * 3 + a.sgrow, col0 = (T.left - a.sgcol + pad + 2) / 3 * 3 + a.sgcol;
  const int nr = row0 < mrow - pad ? (mrow - pad - row0 + 2) / 3 : 0, nc = col0 < mcol - pad ? (mcol - pad - col0 + 2) / 3 : 0;
  for(int idx = tid; idx < nr * nc; idx += nt)
  {
    const int row = row0 + 3 * (idx / nc), col = col0 + 3 * (idx % nc);
    const int p = (row - T.top) * TS + (col - T.left);
    int h = mk_fc(a.xt, row, col + 1);
    float diff[6] = { 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f };
    float color[2][6];
    int plane = 0;
#pragma unroll
    for(int d = 0; d < 6; d++)
    {
      const int i = (d & 1) ? TS : 1;
      const float *const Gp = P + (plane * 3 + 1) * NPX + p;
#pragma unroll
      for(int c = 0; c < 2; c++, h ^= 2)
      {
        const int o = i << c;
        const float *const Hp = P + (plane * 3 + h) * NPX + p;
        const float g = 2 * Gp[0] - Gp[o] - Gp[-o];
        color[h != 0][d] = g + Hp[o] + Hp[-o];
        if(d > 1) diff[d] += mk_sqr(Gp[o] - Gp[-o] - Hp[o] + Hp[-o]) + mk_sqr(g);
      }
      if(d < 2 || (d & 1))
      {
        const int d_out = d - ((d > 1) && (diff[d - 1] < diff[d]));
        P[(plane * 3 + 0) * NPX + p] = color[0][d_out] / 2.f;
        P[(plane * 3 + 2) * NPX + p] = color[1][d_out] / 2.f;
        plane++;
      }
      h ^= 2;
    }
  }
}

// ---- stage 3, :356-373: red at the blue pixels, blue at the red ones ----------------------------------------------------------
__device__ void mk_red_blue(const mk_args_t &a, const mk_tile_t &T, float *P, int pad, int tid, int nt)
{
  const int nr = T.nrow - 2 * pad, nc = T.ncol - 2 * pad;
  if(nr <= 0 || nc <= 0) return;
  for(int idx = tid; idx < nr * nc; idx += nt)
  {
    const int r = pad + idx / nc, c0 = pad + idx % nc, row = T.top + r, col = T.left + c0;
    const int f = 2 - mk_fc(a.xt, row, col);
    if(f == 1) continue;
    const int p = r * TS + c0;
    const int c = (row - a.sgrow) % 3 ? TS : 1;
    const int h = 3 * (c ^ TS ^ 1);
#pragma unroll
    for(int d = 0; d < 4; d++)
    {
      const float *const Gp = P + (d * 3 + 1) * NPX + p;
      float *const Fp = P + (d * 3 + f) * NPX + p;
      const int i = d > 1 || ((d ^ c) & 1) || ((fabsf(Gp[0] - Gp[c]) + fabsf(Gp[0] - Gp[-c])) < 2.f * (fabsf(Gp[0] - Gp[h]) + fabsf(Gp[0] - Gp[-h]))) ? c : h;
      Fp[0] = (Fp[i] + Fp[-i] + 2.f * Gp[0] - Gp[i] - Gp[-i]) / 2.f;
    }
  }
}

// ---- stage 4, :375-399: red and blue in the 2x2 blocks of green: NK = directions / 2 planes (the loop `d += 2` over the directions) ----
template <int NK> __device__ void mk_green_blocks(const mk_args_t &a, const mk_tile_t &T, float *P, int pad, int tid, int nt)
{
  const int nr = T.nrow - 2 * pad, nc = T.ncol - 2 * pad;
  if(nr <= 0 || nc <= 0) return;
  for(int idx = tid; idx < nr * nc; idx += nt)
  {
    const int r = pad + idx / nc, c0 = pad + idx % nc, row = T.top + r, col = T.left + c0;
    if(!((row - a.sgrow) % 3) || !((col - a.sgcol) % 3)) continue;
    const int p = r * TS + c0;
    const short *const hex = mk_hex(a, row, col);
#pragma unroll
    for(int k = 0; k < NK; k++)
    {
      const int ha = hex[2 * k], hb = hex[2 * k + 1];
      const float *const Gp = P + (k * 3 + 1) * NPX + p;
      if(ha + hb)
      {
        const float g = 3.f * Gp[0] - 2.f * Gp[ha] - Gp[hb];
#pragma unroll
        for(int ch = 0; ch < 4; ch += 2)
        {
          float *const Cp = P + (k * 3 + ch) * NPX + p;
          Cp[0] = mk_div(g + 2.f * Cp[ha] + Cp[hb], 3.f);
        }
      }
      else
      {
        const float g = 2.f * Gp[0] - Gp[ha] - Gp[hb];
#pragma unroll
        for(int ch = 0; ch < 4; ch += 2)
        {
          float *const Cp = P + (k * 3 + ch) * NPX + p;
          Cp[0] = (g + Cp[ha] + Cp[hb]) / 2.f;
        }
      }
    }
  }
}

// ---- stage 5, :417-448: squared differences of Y, Pb, Pr along each direction --------------------------------------------------
struct mk_yuv_t
{
  float y, u, v;
};
__device__ __forceinline__ mk_yuv_t mk_yuv(const float *R, const float *G, const float *B, int q)
{
  mk_yuv_t t;
  const float r = R[q], g = G[q], b = B[q];
  t.y = 0.2627f * r + 0.6780f * g + 0.0593f * b;
  t.u = (b - t.y) * 0.56433f;
  t.v = (r - t.y) * 0.67815f;
  return t;
}
template <int PASSES> __device__ void mk_derivatives(const mk_args_t &a, const mk_tile_t &T, float *P, int tid, int nt)
{
  using geo = mk_geo<PASSES>;
  constexpr int pad = geo::PAD_YUV + 1;
  const int nr = T.nrow - 2 * pad, nc = T.ncol - 2 * pad;
  if(nr <= 0 || nc <= 0) return;
  for(int idx = tid; idx < geo::NDIR * nr * nc; idx += nt)
  {
    const int d = idx / (nr * nc), k = idx - d * (nr * nc);
    const int p = (pad + k / nc) * TS + pad + k % nc;
    const int dd = d & 3, f = dd == 0 ? 1 : (dd == 1 ? TS : (dd == 2 ? TS + 1 : TS - 1));
    const float *const R = P + (d * 3 + 0) * NPX, *const G = R + NPX, *const B = G + NPX;
    const mk_yuv_t c = mk_yuv(R, G, B, p), hi = mk_yuv(R, G, B, p + f), lo = mk_yuv(R, G, B, p - f);
    P[(3 * geo::NDIR + d) * NPX + p] = mk_sqr(2 * c.y - hi.y - lo.y) + mk_sqr(2 * c.u - hi.u - lo.u) + mk_sqr(2 * c.v - hi.v - lo.v);
  }
}

// ---- stage 6, :450-464: homogeneity counts ----------------------------------------------------------------------------------
template <int PASSES> __device__ void mk_homogeneity(const mk_args_t &a, const mk_tile_t &T, const float *P, uint8_t *homo, int tid, int nt)
{
  using geo = mk_geo<PASSES>;
  constexpr int pad = geo::PAD_YUV + 2, NDIR = geo::NDIR;
  const int nr = T.nrow - 2 * pad, nc = T.ncol - 2 * pad;
  if(nr <= 0 || nc <= 0) return;
  const float *const D = P + 3 * NDIR * NPX;
  for(int idx = tid; idx < nr * nc; idx += nt)
  {
    const int p = (pad + idx / nc) * TS + pad + idx % nc;
    float tr = FLT_MAX;
#pragma unroll
    for(int d = 0; d < NDIR; d++)
      if(tr > D[d * NPX + p]) tr = D[d * NPX + p];
    tr *= 8;
#pragma unroll
    for(int d = 0; d < NDIR; d++)
    {
      int n = 0;
#pragma unroll
      for(int v = -1; v <= 1; v++)
#pragma unroll
        for(int h = -1; h <= 1; h++) n += (D[d * NPX + p + v * TS + h] <= tr) ? 1 : 0;
      homo[d * NPX + p] = (uint8_t)n;
    }
  }
}

// ---- stage 7, :466-515: 5x5 sums of the counts, the average of the most homogeneous directions --------------------------------
template <int PASSES> __device__ void mk_average(const mk_args_t &a, const mk_tile_t &T, const float *P, const uint8_t *homo, int tid, int nt)
{
  using geo = mk_geo<PASSES>;
  constexpr int PAD = geo::PAD, NDIR = geo::NDIR;
  const int nr = T.nrow - 2 * PAD, nc = T.ncol - 2 * PAD;
  if(nr <= 0 || nc <= 0) return;
  for(int idx = tid; idx < nr * nc; idx += nt)
  {
    const int r = PAD + idx / nc, c = PAD + idx % nc, p = r * TS + c;
    int hm[NDIR], maxval = 0;
#pragma unroll
    for(int d = 0; d < NDIR; d++)
    {
      int s = 0;
#pragma unroll
      for(int v = -2; v <= 2; v++)
#pragma unroll
        for(int h = -2; h <= 2; h++) s += homo[d * NPX + p + v * TS + h];
      hm[d] = s; // 225 at most: the reference's uint8
      maxval = max(maxval, s);
    }
    maxval -= maxval >> 3;
#pragma unroll
    for(int d = 0; d < NDIR - 4; d++)
    { // :497-503: of a direction and its second-round twin the less homogeneous one drops out
      if(hm[d] < hm[d + 4])
        hm[d] = 0;
      else if(hm[d] > hm[d + 4])
        hm[d + 4] = 0;
    }
    float avg[4] = { 0.0f, 0.0f, 0.0f, 0.0f };
#pragma unroll
    for(int d = 0; d < NDIR; d++)
      if(hm[d] >= maxval)
      {
        avg[0] += P[(d * 3 + 0) * NPX + p];
        avg[1] += P[(d * 3 + 1) * NPX + p];
        avg[2] += P[(d * 3 + 2) * NPX + p];
        avg[3] += 1.0f;
      }
    float *const o = reinterpret_cast<float *>(a.out + (size_t)a.width * (r + T.top) + (c + T.left));
    o[0] = avg[0] / avg[3];
    o[1] = avg[1] / avg[3];
    o[2] = avg[2] / avg[3]; // lane 3 is not a result of the reference
  }
}

// ---- the rounds after the first (three passes): planes 0-3 copied to 4-7 (:275-281), then green again from the closer interpolated values,
// :284-302 (P: planes 4-7; G0: plane 0's green for the bounds).  The pixels it reads are green ones, the pixels it writes are not.
__device__ void mk_copy_planes(float *P, int tid, int nt)
{
  for(int idx = tid; idx < 12 * NPX; idx += nt) P[12 * NPX + idx] = P[idx];
}
__device__ void mk_recalc_green(const mk_args_t &a, const mk_tile_t &T, float *P, const float *G0, int tid, int nt)
{
  const int nr = T.nrow - 12, nc = T.ncol - 12;
  if(nr <= 0 || nc <= 0) return;
  const short *const start = a.start + (size_t)T.cls * NPX;
  for(int idx = tid; idx < nr * nc; idx += nt)
  {
    const int r = 6 + idx / nc, c = 6 + idx % nc, row = T.top + r, col = T.left + c;
    const int f = mk_fc(a.xt, row, col);
    if(f == 1) continue;
    const int p = r * TS + c;
    const short *const hex = mk_hex(a, row, col);
    float mn, mx;
    mk_bounds(a, T, G0, start, p, hex, mn, mx);
    const int flip = !((row - a.sgrow) % 3);
#pragma unroll
    for(int d = 3; d < 6; d++)
    {
      const int pl = (d - 2) ^ flip;
      float *const Gp = P + (pl * 3 + 1) * NPX + p;
      const float *const Fp = P + (pl * 3 + f) * NPX + p;
      const int h = hex[d];
      const float val = Gp[-2 * h] + 2 * Gp[h] - Fp[-2 * h] - 2 * Fp[h] + 3 * Fp[0];
      Gp[0] = mk_clamps(mk_div(val, 3.0f), mn, mx);
    }
  }
}

#ifndef B200_KERNELS_ON_CPU
template <int PASSES> __global__ void __launch_bounds__(MK_NT, 1) markesteijn_tiles_kernel(const __grid_constant__ mk_args_t a)
{
  using geo = mk_geo<PASSES>;
  extern __shared__ uint8_t mk_homo[];
  float *const P = a.scratch + (size_t)blockIdx.x * geo::PLANES * NPX;
  const int tid = threadIdx.x;
  for(int t = blockIdx.x; t < a.ntiles; t += gridDim.x)
  {
    const mk_tile_t T = mk_tile_of(a, t);
    mk_load(a, T, P, tid, MK_NT);
    __syncthreads();
    mk_green(a, T, P, tid, MK_NT);
    __syncthreads();
    for(int pass = 0; pass < PASSES; pass++)
    {
      float *const Pp = pass ? P + 12 * NPX : P;
      if(pass == 1)
      {
        mk_copy_planes(P, tid, MK_NT);
        __syncthreads();
      }
      if(pass)
      {
        mk_recalc_green(a, T, Pp, P + NPX, tid, MK_NT);
        __syncthreads();
      }
      mk_solitary(a, T, Pp, geo::PAD_SG, tid, MK_NT);
      __syncthreads();
      mk_red_blue(a, T, Pp, geo::PAD_RB, tid, MK_NT);
      __syncthreads();
      mk_green_blocks<geo::NDIR / 2>(a, T, Pp, geo::PAD_G22, tid, MK_NT);
      __syncthreads();
    }
    mk_derivatives<PASSES>(a, T, P, tid, MK_NT);
    __syncthreads();
    mk_homogeneity<PASSES>(a, T, P, mk_homo, tid, MK_NT);
    __syncthreads();
    mk_average<PASSES>(a, T, P, mk_homo, tid, MK_NT);
    __syncthreads();
  }
}
#endif

// ---- host: the hexagons (:79-103), the walk (:199-246), the classes of tiles ------------------------------------------------
void mk_hexagons(mk_args_t &a)
{
  static const short orth[12] = { 1, 0, 0, 1, -1, 0, 0, -1, 1, 0, 0, 1 };
  static const short patt[2][16] = { { 0, 1, 0, -1, 2, 0, -1, 0, 1, 1, 1, -1, 0, 0, 0, 0 }, { 0, 1, 0, -2, 1, 0, -2, 0, 1, 1, -2, -2, 1, -1, -1, 1 } };
  a.sgrow = a.sgcol = 0;
  memset(a.hex, 0, sizeof(a.hex));
  for(int row = 0; row < 3; row++)
    for(int col = 0; col < 3; col++)
    {
      const int g = mk_fc(a.xt, row, col) == 1;
      int ng = 0;
      for(int d = 0; d < 10; d += 2)
      {
        ng = mk_fc(a.xt, row + orth[d], col + orth[d + 2]) == 1 ? 0 : ng + 1;
        if(ng == 4)
        {
          a.sgrow = row;
          a.sgcol = col;
        }
        if(ng == g + 1)
          for(int c = 0; c < 8; c++)
          {
            const int v = orth[d] * patt[g][c * 2] + orth[d + 1] * patt[g][c * 2 + 1];
            const int h = orth[d + 2] * patt[g][c * 2] + orth[d + 3] * patt[g][c * 2 + 1];
            a.hex[row][col][c ^ (g * 2 & d)] = (short)(h + v * TS);
          }
      }
    }
}

// the loop of :199-246 over a tile at (top, left) of nrow x ncol pixels, control flow only: start[p] = the pixel whose hexagon opened
// the run that wrote pixel p last, -1 = never written
void mk_walk(short *start, const uint8_t *xt, int sgrow, int top, int left, int nrow, int ncol)
{
  const int mrow = top + nrow, mcol = left + ncol;
  for(int k = 0; k < NPX; k++) start[k] = -1;
  for(int row = top + 3; row < mrow - 3; row++)
  {
    int open = -1;
    for(int col = left + 3; col < mcol - 3; col++)
    {
      if(mk_fc(xt, row, col) == 1)
      {
        open = -1;
        continue;
      }
      const int p = (row - top) * TS + (col - left);
      if(open < 0) open = p;
      start[p] = (short)open;
      switch((row - sgrow) % 3)
      {
        case 1:
          if(row < mrow - 4) row++, col--;
          break;
        case 2:
          open = -1;
          if((col += 2) < mcol - 4 && row > top + 3) row--;
      }
    }
  }
}

// tiles (top = -pad + k * step < height - pad, left likewise: pad 12, step 98 with one pass, 17 and 88 with three) and their classes: full
// tiles by the phase of their origin (three of them: 98 = 2 and 88 = 4 mod 6), the last row / column by its size; one record of the walk per class.  Nonzero: too many classes.
int mk_build_classes(mk_args_t &a, std::vector<short> &maps)
{
  const int PAD = a.pad, STEP = a.step;
  a.ntx = (a.width + STEP - 1) / STEP;
  const int nty = (a.height + STEP - 1) / STEP;
  a.ntiles = a.ntx * nty;
  std::vector<int> row_top, row_n, col_left, col_n;
  // first_own: the tile at the negative origin is a class of its own (the walk takes (row - sgrow) % 3 with C's sign: the rows above
  // the frame never hop)
  auto classes = [&](int n_tiles, int size, uint8_t *by_phase, int &last, int *first, std::vector<int> &origin, std::vector<int> &extent) {
    for(int k = 0; k < 6; k++) by_phase[k] = 0;
    last = 0;
    for(int k = 0; k < n_tiles; k++)
    {
      const int o = -PAD + k * STEP, n = (o + TS < size + PAD) ? TS : size + PAD - o;
      int found = -1;
      for(size_t j = (first ? 1 : 0); j < origin.size() && k > 0; j++)
        if(extent[j] == n && (origin[j] + 600) % 6 == (o + 600) % 6) found = (int)j;
      if(found < 0)
      {
        origin.push_back(o);
        extent.push_back(n);
        found = (int)origin.size() - 1;
      }
      if(first && k == 0)
        *first = found;
      else if(n == TS)
        by_phase[(o + 600) % 6] = (uint8_t)found;
      else
        last = found;
    }
  };
  classes(nty, a.height, a.cls_row, a.cls_last_row, &a.cls_first_row, row_top, row_n);
  classes(a.ntx, a.width, a.cls_col, a.cls_last_col, nullptr, col_left, col_n);
  a.n_col_classes = (int)col_left.size();
  const size_t n_cls = row_top.size() * col_left.size();
  if(n_cls > MK_MAX_CLASSES) return 1;
  maps.resize(n_cls * NPX);
  for(size_t i = 0; i < row_top.size(); i++)
    for(size_t j = 0; j < col_left.size(); j++)
      mk_walk(maps.data() + (i * col_left.size() + j) * NPX, a.xt, a.sgrow, row_top[i], col_left[j], row_n[i], col_n[j]);
  return 0;
}

#ifndef B200_KERNELS_ON_CPU
struct mk_plan_t
{ // what depends on the geometry only: built once per (frame size, origin, pattern), kept on the device
  int width = 0, height = 0, rx = 0, ry = 0, dev = -1, passes = 0; // dev < 0: matches no call
  uint8_t xtrans[36] = { 0 };
  mk_args_t a;
  short *d_start = nullptr;
  cudaEvent_t used = nullptr; // recorded after every launch that reads d_start, on the stream it went to

  cudaError_t release()
  { // waits for the last launch that read the maps, on whichever stream it went to, then frees them
    cudaError_t e = used ? cudaEventSynchronize(used) : cudaSuccess;
    if(d_start && e == cudaSuccess) e = cudaFree(d_start);
    if(used) cudaEventDestroy(used);
    *this = mk_plan_t();
    return e;
  }
};
struct mk_plans_t
{ // per calling thread, as the device scratch is (runtime.cu): two geometries (the preview and the full pipe), replaced in turn
  mk_plan_t plan[2];
  int next = 0;
  ~mk_plans_t()
  {
    if(!b200::runtime_alive()) return;
    int cur = 0;
    cudaGetDevice(&cur);
    for(auto &p : plan)
      if(p.d_start || p.used)
      {
        cudaSetDevice(p.dev < 0 ? cur : p.dev);
        p.release();
      }
    cudaSetDevice(cur);
  }
};
thread_local mk_plans_t tls_plans;

template <int PASSES> int mk_launch(mk_args_t &a, int dev, cudaStream_t stream)
{
  using geo = mk_geo<PASSES>;
  static std::atomic<bool> attr_set[16] = {}; // per device; setting it twice from two threads is harmless
  const int smem = geo::NDIR * NPX;
  if(!attr_set[dev & 15].load(std::memory_order_acquire))
  {
    B200_CUDA_TRY(cudaFuncSetAttribute(markesteijn_tiles_kernel<PASSES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set[dev & 15].store(true, std::memory_order_release);
  }
  int grid = b200::sm_count();
  if(grid > a.ntiles) grid = a.ntiles;
  void *scr = nullptr;
  int rc = b200::scratch(b200::SLOT_TMP2, (size_t)grid * geo::PLANES * NPX * sizeof(float), &scr);
  if(rc) return rc;
  a.scratch = (float *)scr;
  markesteijn_tiles_kernel<PASSES><<<grid, MK_NT, smem, stream>>>(a);
  B200_CUDA_TRY(cudaGetLastError());
  return B200_OK;
}
#endif
} // namespace

#ifndef B200_KERNELS_ON_CPU
namespace b200
{
// xtrans_markesteijn_interpolate(), markesteijn.c:47-521, passes == 1 or 3.  (x0, y0): origin of the region on the sensor.
int markesteijn_demosaic_dev(const float *d_in, float *d_out, int width, int height, int x0, int y0, const uint8_t xtrans[6][6], int passes, cudaStream_t stream)
{
  if(passes != 1 && passes != 3) return fail(B200_ERR_ARG, "Markesteijn: %d passes", passes);
  { // the mirrored border (:158, TRANSLATE) reads row / column `pad` and 2 * size - (size + pad - 1) - 2: smaller frames are out-of-bounds reads
    // in the reference
    const int pad = passes == 1 ? mk_geo<1>::PAD : mk_geo<3>::PAD;
    if(width > 0 && height > 0 && (width <= pad || height <= pad))
      return fail(B200_ERR_UNSUPPORTED, "Markesteijn: frames of %d px or less a side are undefined in the reference with %d pass(es)", pad, passes);
  }
  if(width < 1 || height < 1) return B200_OK;
  int dev = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  mk_plan_t *plan = nullptr;
  for(auto &q : tls_plans.plan)
    if(q.d_start && q.dev == dev && q.passes == passes && q.width == width && q.height == height && q.rx == x0 && q.ry == y0 && !memcmp(q.xtrans, xtrans, 36)) plan = &q;
  if(!plan)
  {
    plan = &tls_plans.plan[tls_plans.next];
    tls_plans.next ^= 1;
    // a frame queued on another of this thread's streams may still read the maps being replaced: release() waits for it
    B200_CUDA_TRY(plan->release());
    B200_CUDA_TRY(cudaEventCreateWithFlags(&plan->used, cudaEventDisableTiming));
    mk_args_t &a = plan->a;
    memset(&a, 0, sizeof(a));
    a.width = width;
    a.height = height;
    a.pad = passes == 1 ? mk_geo<1>::PAD : mk_geo<3>::PAD;
    a.step = passes == 1 ? mk_geo<1>::STEP : mk_geo<3>::STEP;
    for(int r = 0; r < 6; r++)
      for(int c = 0; c < 6; c++) a.xt[r * 6 + c] = xtrans[(r + y0 + 600) % 6][(c + x0 + 600) % 6];
    mk_hexagons(a);
    std::vector<short> maps;
    if(mk_build_classes(a, maps)) return fail(B200_ERR_ARG, "Markesteijn: more than %d classes of tiles", MK_MAX_CLASSES);
    B200_CUDA_TRY(cudaMalloc(&plan->d_start, maps.size() * sizeof(short)));
    B200_CUDA_TRY(cudaMemcpyAsync(plan->d_start, maps.data(), maps.size() * sizeof(short), cudaMemcpyHostToDevice, stream));
    B200_CUDA_TRY(cudaStreamSynchronize(stream)); // `maps` leaves scope
    a.start = plan->d_start;
    plan->width = width;
    plan->height = height;
    plan->rx = x0;
    plan->ry = y0;
    plan->passes = passes;
    memcpy(plan->xtrans, xtrans, 36);
    plan->dev = dev; // complete: from here on the plan matches
  }
  mk_args_t a = plan->a;
  a.in = d_in;
  a.out = (float4 *)d_out;
  const int rc = passes == 1 ? mk_launch<1>(a, dev, stream) : mk_launch<3>(a, dev, stream);
  if(rc) return rc;
  B200_CUDA_TRY(cudaEventRecord(plan->used, stream));
  return B200_OK;
}
} // namespace b200
#endif
