// RCD (Ratio-Corrected Demosaicing 2.3) for B200 / sm_100a.
//
// What the reference computes: src/iop/demosaic/rcd.c:274-564 (tile walk) and :91-272 (frame-edge
// ring).  Parity contract: bit-identical to that source evaluated with C-standard float
// semantics (oracle/restate/rcd_oracle.c, pinned against oracle/_ref/libref_strict.so).
// Consequences that shape this kernel:
//   * the reference's result depends on its own 112x112 / 94x94 tile grid (the zero VH_Dir ring at
//     tile-local rows/cols < 4 leaks into kept pixels), so one CTA processes exactly one
//     reference tile, entirely in shared memory;
//   * fabs() in the reference is the double function: gradient sums are accumulated in FP64 and
//     rounded once (B200 has full-rate-enough FP64; this is not B300);
//   * no FMA contraction, IEEE division, FTZ on (the reference sets FTZ|DAZ, rcd.c:300): the
//     library is compiled with --fmad=false -ftz=true -prec-div=true.
//
// Shared-memory planes per tile, all with a row pitch of 56 floats:
//   cfaE cfaO   raw values at even / odd columns          vhE vhO   VH_Dir at even / odd columns
//   grb   green at red/blue sites (rgb[1] there; equals cfa until step 3.1 writes it)
//   pq    low-pass, later PQ_Dir -- the reference aliases them too (rcd.c:314)
//   pd    P_CDiff_Hpf, later "crb" = the opposite colour at red/blue sites (rgb[2-FC])
//   qd    Q_CDiff_Hpf
// = 8 regions of 6272 floats + 16 floats of padding each = 201,216 B -> one CTA per SM.
// The half-width planes of the reference are addressed with flat_index/2 (rcd.c:396,444,453,464) =
// row*56 + (col>>1); the full planes are split by column parity so that they use the SAME index.  Red/blue-
// site loops (lane stride = 2 columns) then walk every plane with stride 1, and full-width loops put even
// lanes in the E plane and odd lanes in the O plane, whose base is 16 banks further: no bank conflicts
// (the interleaved layout paid +49 % shared-memory wavefronts, profiles/r01_rcd_tiles_ncu.md).
// rgb[0]/rgb[2] at green sites are only ever consumed by the output loop, so step 4.3 is fused
// into the store and evaluated for kept pixels only.
//
// HBM traffic per tile: 112*112*4 B read (1.42x over-read from the 18-px overlap, served by L2),
// 94*94*16 B written.  Algorithmic bytes: 20 B/px (SURVEY.md 8d).
#include "runtime.h"
#include <atomic>

namespace
{
constexpr int T = 112;     // RCD_TILESIZE   rcd.c:53-55
constexpr int KEEP = 94;   // RCD_TILEVALID  rcd.c:75
constexpr int RING = 9;    // RCD_BORDER     rcd.c:73
constexpr int EDGE = 6;    // RCD_MARGIN     rcd.c:74
constexpr int H = T / 2;   // width of a half plane row
#ifndef RCD_RG
#define RCD_RG 8
#endif
#ifndef RCD_UNROLL
#define RCD_UNROLL 1
#endif
#define RCD_PRAGMA(x) _Pragma(#x)
#define RCD_UNROLL_LOOP(n) RCD_PRAGMA(unroll n)
constexpr int RG = RCD_RG; // row groups: NT = RG x 112 columns, or 2*RG x 56 site columns
constexpr int NT = RG * T; // threads per CTA
constexpr int HP = T * H;       // floats in one half plane
constexpr int RS = HP + 16;     // region stride: consecutive regions sit 16 banks apart
constexpr int SMEM_FLOATS = 8 * RS;

constexpr float kEps = 1e-5f;    // rcd.c:81
constexpr float kEpsSq = 1e-10f; // rcd.c:82

struct rcd_args_t
{
  const float *in;
  float *out;
  int width, height;
  uint32_t filters;
  float scaler, revscaler;
  int nv, nh;
};

__device__ __forceinline__ int fc(int row, int col, uint32_t f)
{
  return (int)((f >> (((((unsigned)row << 1) & 14u) + ((unsigned)col & 1u)) << 1)) & 3u);
}
__device__ __forceinline__ float sq(float v) { return v * v; }
__device__ __forceinline__ float mixf(float a, float b, float c) { return a * (b - c) + c; } // iop/demosaic.c:250-257
// squared 7-tap high-pass of rcd.c:360-386,442-449 from its taps at -3..3
__device__ __forceinline__ float hpf2v(float m3, float m2, float m1, float c0, float p1, float p2, float p3)
{
  return sq((m3 - m1 - p1 + p3) - 3.0f * (m2 + p2) + 6.0f * c0);
}
__device__ __forceinline__ float refine(float centre, float nb)
{
  return (fabsf(0.5f - centre) < fabsf(0.5f - nb)) ? nb : centre;
}
// |a - b| widened to double, the way `fabs(float - float)` reads in C
__device__ __forceinline__ double dabs(float a, float b) { return (double)fabsf(a - b); }

__global__ void __launch_bounds__(NT, 1) rcd_tiles_kernel(const rcd_args_t a)
{
  extern __shared__ __align__(16) float smem[];
  float *const cfa = smem;          // E plane at +0, O plane at +RS
  float *const vh = smem + 2 * RS;  // likewise
  float *const grb = smem + 4 * RS;
  float *const pq = smem + 5 * RS;
  float *const pd = smem + 6 * RS;
  float *const qd = smem + 7 * RS;
  float *const crb = pd;
  // scratch views used only during step 1 (grb/pq and pd/qd are idle then): E/O planes like cfa
  float *const vsq = grb; // squared vertical high-pass
  float *const hsq = pd;  // squared horizontal high-pass

  const int tid = threadIdx.x;
  const int tv = blockIdx.x / a.nh, th = blockIdx.x - tv * a.nh;
  const int row0 = tv * KEEP, col0 = th * KEEP;
  const int tr = min(T, a.height - row0), tc = min(T, a.width - col0);
  const uint32_t f = a.filters;

  // thread -> (column, row group) maps; no integer division by runtime values anywhere below
  const int x112 = tid % T, y4 = tid / T; // RG row groups over full-width domains
  const int x56 = tid % H, y8 = tid / H;  // 2*RG row groups over every-second-column domains
  // full-width domains: element (r, x112) of a split plane sits at fb + r*56; its left/right neighbours
  // x-1, x+1, x-3, x+3 at fo + r*56 + {0, 1, -1, 2}; x-2, x+2 at fb + r*56 -+ 1
  const int fpx = x112 & 1;
  const int fb = fpx * RS + (x112 >> 1);
  const int fo = (1 - fpx) * RS + (x112 >> 1) + fpx - 1;

  // ---- step 0: load, clamp, normalise (rcd.c:343-351) ---------------------------------------
  // All of a thread's loads are issued before anything else, so the tile costs one DRAM/L2 round trip, and that
  // round trip is spent clearing shared memory: the reference's never-written scratch is defined as zero.
  {
    constexpr int NR = T / RG;
    static_assert(NR * RG == T, "row groups must divide the tile");
    float v[NR];
    const float *src = a.in + (size_t)(row0 + y4) * a.width + col0 + x112;
    const size_t pitch = (size_t)RG * a.width;
#pragma unroll
    for(int k = 0; k < NR; k++) v[k] = (x112 < tc && y4 + k * RG < tr) ? __ldg(src + k * pitch) : 0.0f;
    {
      float4 *p = reinterpret_cast<float4 *>(smem);
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      for(int k = tid; k < SMEM_FLOATS / 4; k += NT) p[k] = z;
    }
    __syncthreads();
#pragma unroll
    for(int k = 0; k < NR; k++)
      if(x112 < tc && y4 + k * RG < tr) cfa[fb + (y4 + k * RG) * H] = fmaxf(0.0f, v[k]) * a.revscaler;
  }
  __syncthreads();

  // ---- step 1: squared V/H high-pass, then direction strength (rcd.c:353-390) ----------------
  for(int r = 3 + y4; r < tr - 3; r += RG)
  {
    const float *c = cfa + fb + r * H, *o = cfa + fo + r * H;
    if(x112 >= 4 && x112 < tc - 4) vsq[fb + r * H] = hpf2v(c[-3 * H], c[-2 * H], c[-H], c[0], c[H], c[2 * H], c[3 * H]);
    if(r >= 4 && r < tr - 4 && x112 >= 3 && x112 < tc - 3) hsq[fb + r * H] = hpf2v(o[-1], c[-1], o[0], c[0], o[1], c[1], o[2]);
  }
  __syncthreads();
  for(int r = 4 + y4; r < tr - 4; r += RG)
    if(x112 >= 4 && x112 < tc - 4)
    {
      const int i = fb + r * H, j = fo + r * H;
      const float vs = fmaxf(kEpsSq, vsq[i - H] + vsq[i] + vsq[i + H]);
      const float hs = fmaxf(kEpsSq, hsq[j] + hsq[i] + hsq[j + 1]);
      vh[i] = vs / (vs + hs);
    }
  __syncthreads();
  // give the borrowed planes back: zero, then green-at-red/blue starts out as the raw value
  {
    float4 *p = reinterpret_cast<float4 *>(grb); // grb, pq, pd, qd (and their padding) are contiguous
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for(int k = tid; k < 4 * RS / 4; k += NT) p[k] = z;
  }
  __syncthreads();
  for(int r = y8; r < tr; r += 2 * RG)
  {
    const int p = fc(r, 0, f) & 1;
    if(p + 2 * x56 < tc) grb[r * H + x56] = cfa[p * RS + r * H + x56];
  }

  // Red/blue site (r, c), c = base + p + 2*x56 with p = the column parity of those sites in row r:
  //   h  = r*56 + (c>>1)   index in every half plane and inside a split plane
  //   sb = p*RS + h        same-parity plane: (r+dr, c+2k) at sb + 56*dr + k
  //   ob = (1-p)*RS + h + p - 1   other plane: c-1, c+1, c-3, c+3 at ob + {0, 1, -1, 2} (+ 56*dr)
  //   half-plane neighbours: (c-1)>>1 = h + p - 1, (c+1)>>1 = h + p

  // ---- step 2.1: low-pass at red/blue sites (rcd.c:394-402) ----------------------------------
  for(int r = 2 + y8; r < tr - 2; r += 2 * RG)
  {
    const int p = fc(r, 0, f) & 1;
    if(2 + p + 2 * x56 < tc - 2)
    {
      const int h = r * H + 1 + x56;
      const float *s = cfa + p * RS + h, *o = cfa + (1 - p) * RS + h + p - 1;
      pq[h] = s[0] + 0.5f * (s[-H] + s[H] + o[0] + o[1]) + 0.25f * (o[-H] + o[1 - H] + o[H] + o[1 + H]);
    }
  }
  __syncthreads();

  // ---- step 3.1: green at red/blue sites (rcd.c:406-437) -------------------------------------
  RCD_UNROLL_LOOP(RCD_UNROLL)
  for(int r = 4 + y8; r < tr - 4; r += 2 * RG)
  {
    const int p = fc(r, 0, f) & 1;
    if(4 + p + 2 * x56 < tc - 4)
    {
      const int h = r * H + 2 + x56;
      const float *s = cfa + p * RS + h, *o = cfa + (1 - p) * RS + h + p - 1;
      const float x = s[0];
      const float u1 = s[-H], u2 = s[-2 * H], u3 = s[-3 * H], u4 = s[-4 * H];
      const float d1 = s[H], d2 = s[2 * H], d3 = s[3 * H], d4 = s[4 * H];
      const float l1 = o[0], l2 = s[-1], l3 = o[-1], l4 = s[-2];
      const float r1 = o[1], r2 = s[1], r3 = o[2], r4 = s[2];
      const double ud = dabs(u1, d1), lr = dabs(l1, r1);
      const float gn = (float)((double)kEps + ud + dabs(x, u2) + dabs(u1, u3) + dabs(u2, u4));
      const float gs = (float)((double)kEps + ud + dabs(x, d2) + dabs(d1, d3) + dabs(d2, d4));
      const float gw = (float)((double)kEps + lr + dabs(x, l2) + dabs(l1, l3) + dabs(l2, l4));
      const float ge = (float)((double)kEps + lr + dabs(x, r2) + dabs(r1, r3) + dabs(r2, r4));

      const float l = pq[h], ll = l + l;
      const float en = u1 * ll / (kEps + l + pq[h - 2 * H]);
      const float es = d1 * ll / (kEps + l + pq[h + 2 * H]);
      const float ew = l1 * ll / (kEps + l + pq[h - 1]);
      const float ee = r1 * ll / (kEps + l + pq[h + 1]);

      const float ev = (gs * en + gn * es) / (gn + gs);
      const float eh = (gw * ee + ge * ew) / (ge + gw);
      const float *vo = vh + (1 - p) * RS + h + p - 1; // the four diagonal neighbours are of the other parity
      const float nb = 0.25f * (vo[-H] + vo[1 - H] + vo[H] + vo[1 + H]);
      grb[h] = mixf(refine(vh[p * RS + h], nb), eh, ev);
    }
  }

  // ---- step 4.0: squared diagonal high-pass at every second column from 3 (rcd.c:442-449) -----
  // site (r, c), c = 3 + 2*x56 odd, m = c>>1: (r+k, c+k) is in the O plane for even k, the E plane for odd k,
  // at column index m + ((k+1)>>1); (r+k, c-k) at m + ((1-k)>>1)
  for(int r = 3 + y8; r < tr - 3; r += 2 * RG)
  {
    if(3 + 2 * x56 < tc - 3)
    {
      const int h = r * H + 1 + x56;
      const float *e = cfa + h, *o = cfa + RS + h;
      const float c0 = o[0];
      pd[h] = hpf2v(e[-3 * H - 1], o[-2 * H - 1], e[-H], c0, e[H + 1], o[2 * H + 1], e[3 * H + 2]);
      qd[h] = hpf2v(e[-3 * H + 2], o[-2 * H + 1], e[-H + 1], c0, e[H], o[2 * H - 1], e[3 * H - 1]);
    }
  }
  __syncthreads();

  // ---- step 4.1: P/Q direction strength, overwriting the low-pass (rcd.c:451-459) ------------
  for(int r = 4 + y8; r < tr - 4; r += 2 * RG)
  {
    const int p = fc(r, 0, f) & 1;
    if(4 + p + 2 * x56 < tc - 4)
    {
      const int h = r * H + 2 + x56, hu = h - H + p - 1, hd = h + H + p - 1;
      const float ps = fmaxf(kEpsSq, pd[hu] + pd[h] + pd[hd + 1]);
      const float qs = fmaxf(kEpsSq, qd[hu + 1] + qd[h] + qd[hd]);
      pq[h] = ps / (ps + qs);
    }
  }
  __syncthreads();
  // pd becomes crb: the opposite colour at red/blue sites, zero where step 4.2 never writes
  {
    float4 *p = reinterpret_cast<float4 *>(crb);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for(int k = tid; k < HP / 4; k += NT) p[k] = z;
  }
  __syncthreads();

  // ---- step 4.2: opposite colour at red/blue sites (rcd.c:462-491) ---------------------------
  // rgb[c] at the diagonal neighbours is that site's own raw value, i.e. cfa.
  RCD_UNROLL_LOOP(RCD_UNROLL)
  for(int r = 4 + y8; r < tr - 4; r += 2 * RG)
  {
    const int p = fc(r, 0, f) & 1;
    if(4 + p + 2 * x56 < tc - 4)
    {
      const int h = r * H + 2 + x56, hu = h - H + p - 1, hd = h + H + p - 1;
      const float nb = 0.25f * (pq[hu] + pq[hu + 1] + pq[hd] + pq[hd + 1]);
      const float disc = refine(pq[h], nb);

      const float *o = cfa + (1 - p) * RS + h + p - 1;
      const float cnw = o[-H], cne = o[1 - H], csw = o[H], cse = o[1 + H];
      const float g = grb[h];
      const double d_nwse = dabs(cnw, cse), d_nesw = dabs(cne, csw);
      const float gnw = (float)((double)kEps + d_nwse + dabs(cnw, o[-3 * H - 1]) + dabs(g, grb[h - 2 * H - 1]));
      const float gne = (float)((double)kEps + d_nesw + dabs(cne, o[-3 * H + 2]) + dabs(g, grb[h - 2 * H + 1]));
      const float gsw = (float)((double)kEps + d_nesw + dabs(csw, o[3 * H - 1]) + dabs(g, grb[h + 2 * H - 1]));
      const float gse = (float)((double)kEps + d_nwse + dabs(cse, o[3 * H + 2]) + dabs(g, grb[h + 2 * H + 1]));

      const float dnw = cnw - grb[hu], dne = cne - grb[hu + 1];
      const float dsw = csw - grb[hd], dse = cse - grb[hd + 1];
      const float ep = (gnw * dse + gse * dnw) / (gnw + gse);
      const float eq = (gne * dsw + gsw * dne) / (gne + gsw);
      crb[h] = g + mixf(disc, eq, ep);
    }
  }
  __syncthreads();

  // ---- step 4.3 fused with the store of the kept interior (rcd.c:494-554) --------------------
  const int ra = (tv == 0 ? EDGE : RING), rb = tr - (tv == a.nv - 1 ? EDGE : RING);
  const int ca = (th == 0 ? EDGE : RING), cb = tc - (th == a.nh - 1 ? EDGE : RING);
  RCD_UNROLL_LOOP(RCD_UNROLL)
  for(int r = ra + y8; r < rb; r += 2 * RG)
  {
    const int rbpar = fc(r, 0, f) & 1; // column parity of the red/blue sites in this row
    const int native = fc(r, rbpar, f); // 0 or 2: the colour those sites carry
    const int h = r * H + x56;          // both sites of this thread's column pair share it
    // --- the red/blue site of this thread's column pair
    {
      const int c = 2 * x56 + rbpar;
      if(c >= ca && c < cb)
      {
        float px[3];
        px[native] = cfa[rbpar * RS + h];
        px[1] = grb[h];
        px[2 - native] = crb[h];
        float4 o = make_float4(a.scaler * fmaxf(0.0f, px[0]), a.scaler * fmaxf(0.0f, px[1]),
                               a.scaler * fmaxf(0.0f, px[2]), 0.0f);
        __stcs(reinterpret_cast<float4 *>(a.out + 4 * ((size_t)(row0 + r) * a.width + col0 + c)), o);
      }
    }
    // --- the green site: red and blue from the four cardinal neighbours
    {
      const int q = 1 - rbpar, c = 2 * x56 + q;
      if(c >= ca && c < cb)
      {
        const float *s = cfa + q * RS + h;               // the site and its same-column / +-2 column neighbours
        const float *vo = vh + (1 - q) * RS + h + q - 1; // VH_Dir at the diagonal neighbours
        const float nb = 0.25f * (vo[-H] + vo[1 - H] + vo[H] + vo[1 + H]);
        const float disc = refine(vh[q * RS + h], nb);
        const float g = s[0];
        const float n1 = (float)((double)kEps + dabs(g, s[-2 * H]));
        const float s1 = (float)((double)kEps + dabs(g, s[2 * H]));
        const float w1 = (float)((double)kEps + dabs(g, s[-1]));
        const float e1 = (float)((double)kEps + dabs(g, s[1]));
        const int hl = h + q - 1; // half index of the left neighbour; the right one is hl + 1
        const float gu = grb[h - H], gd = grb[h + H], gl = grb[hl], gr = grb[hl + 1];

        // Vertical neighbours carry colour `vcol` natively, horizontal ones carry `native`.
        // rgb[k] at a site of the other colour is crb there; at its own colour it is cfa.  Both planes have
        // a 56-float row pitch, so one base pointer per direction serves either.
        const int vcol = 2 - native;
        float px[3];
        px[1] = g;
#pragma unroll
        for(int k = 0; k <= 2; k += 2)
        {
          const float *const pv = (k == vcol) ? s : (crb + h);                                   // (r+-1, c), (r+-3, c)
          const float *const ph = (k == native) ? (cfa + (1 - q) * RS + hl) : (crb + hl);         // c-1, c+1, c-3, c+3 at {0, 1, -1, 2}
          const float cu1 = pv[-H], cd1 = pv[H], cu3 = pv[-3 * H], cd3 = pv[3 * H];
          const float cl1 = ph[0], cr1 = ph[1], cl3 = ph[-1], cr3 = ph[2];
          const float sn = fabsf(cu1 - cd1), ew = fabsf(cl1 - cr1);
          const float gn = (float)((double)(n1 + sn) + dabs(cu1, cu3));
          const float gs = (float)((double)(s1 + sn) + dabs(cd1, cd3));
          const float gw = (float)((double)(w1 + ew) + dabs(cl1, cl3));
          const float ge = (float)((double)(e1 + ew) + dabs(cr1, cr3));
          const float dn = cu1 - gu, ds = cd1 - gd, dw = cl1 - gl, de = cr1 - gr;
          const float ev = (gn * ds + gs * dn) / (gn + gs);
          const float eh = (ge * dw + gw * de) / (ge + gw);
          px[k] = g + mixf(disc, eh, ev);
        }
        float4 o = make_float4(a.scaler * fmaxf(0.0f, px[0]), a.scaler * fmaxf(0.0f, px[1]),
                               a.scaler * fmaxf(0.0f, px[2]), 0.0f);
        __stcs(reinterpret_cast<float4 *>(a.out + 4 * ((size_t)(row0 + r) * a.width + col0 + c)), o);
      }
    }
  }
}

// ---- frame-edge ring: rcd_ppg_border(), rcd.c:91-272, one thread per ring pixel --------------
// The reference makes three in-place sweeps; per pixel at frame distance d they amount to
//   d < 3      non-native channels = mean of that colour over the clipped 3x3 neighbourhood
//   3 <= d < 9 green at red/blue sites from the PPG gradient test
//   1 <= d < 6 red/blue from the neighbours' native value and green
// and only d < 6 survives the tile stores.  Everything is recomputed from the mosaic, so the
// kernel has no ordering constraints (see oracle/restate/rcd_oracle.c ring_pixel()).
struct ring_t
{
  const float *in;
  int w, h;
  uint32_t f;
};
__device__ __forceinline__ int ring_dist(const ring_t &q, int r, int c)
{
  return min(min(r, c), min(q.h - 1 - r, q.w - 1 - c));
}
__device__ __forceinline__ float ring_raw(const ring_t &q, int r, int c)
{
  return fmaxf(0.0f, __ldg(q.in + (size_t)r * q.w + c));
}
__device__ float ring_mean(const ring_t &q, int r, int c, int k)
{
  if(k == fc(r, c, q.f)) return ring_raw(q, r, c);
  float sum = 0.0f, cnt = 0.0f;
  for(int y = r - 1; y != r + 2; y++)
    for(int x = c - 1; x != c + 2; x++)
      if(y >= 0 && x >= 0 && y < q.h && x < q.w && fc(y, x, q.f) == k)
      {
        sum += ring_raw(q, y, x);
        cnt += 1.0f;
      }
  return cnt > 0.0f ? sum / cnt : ring_raw(q, r, c);
}
__device__ float ring_green(const ring_t &q, int r, int c)
{
  if(ring_dist(q, r, c) < 3) return ring_mean(q, r, c, 1);
  const int s = fc(r, c, q.f);
  const float pc = ring_raw(q, r, c);
  if(!(s == 0 || s == 2)) return pc;
  const float ym = ring_raw(q, r - 1, c), ym2 = ring_raw(q, r - 2, c), ym3 = ring_raw(q, r - 3, c);
  const float yp = ring_raw(q, r + 1, c), yp2 = ring_raw(q, r + 2, c), yp3 = ring_raw(q, r + 3, c);
  const float xm = ring_raw(q, r, c - 1), xm2 = ring_raw(q, r, c - 2), xm3 = ring_raw(q, r, c - 3);
  const float xp = ring_raw(q, r, c + 1), xp2 = ring_raw(q, r, c + 2), xp3 = ring_raw(q, r, c + 3);
  const float guessx = (xm + pc + xp) * 2.0f - xp2 - xm2;
  const float diffx = (fabsf(xm2 - pc) + fabsf(xp2 - pc) + fabsf(xm - xp)) * 3.0f + (fabsf(xp3 - xp) + fabsf(xm3 - xm)) * 2.0f;
  const float guessy = (ym + pc + yp) * 2.0f - yp2 - ym2;
  const float diffy = (fabsf(ym2 - pc) + fabsf(yp2 - pc) + fabsf(ym - yp)) * 3.0f + (fabsf(yp3 - yp) + fabsf(ym3 - ym)) * 2.0f;
  if(diffx > diffy) return fmaxf(fminf(guessy * .25f, fmaxf(ym, yp)), fminf(ym, yp));
  return fmaxf(fminf(guessx * .25f, fmaxf(xm, xp)), fminf(xm, xp));
}
__device__ __forceinline__ float ring_chan(const ring_t &q, int r, int c, int k)
{
  return ring_dist(q, r, c) < 3 ? ring_mean(q, r, c, k) : ring_raw(q, r, c);
}

__global__ void __launch_bounds__(128) rcd_ring_kernel(const float *in, float *out, int width, int height, uint32_t filters)
{
  // ring pixels in a fixed enumeration: EDGE full rows on top, EDGE at the bottom, then the two
  // EDGE-wide side bands of the rows in between
  const long long n_top = (long long)EDGE * width * 2;
  const long long n_side = (long long)(height - 2 * EDGE) * EDGE * 2;
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if(k >= n_top + n_side) return;
  int r, c;
  if(k < n_top)
  {
    r = (int)(k / width);
    c = (int)(k - (long long)r * width);
    if(r >= EDGE) r = height - 2 * EDGE + r;
  }
  else
  {
    const long long j = k - n_top;
    r = EDGE + (int)(j / (2 * EDGE));
    c = (int)(j - (long long)(r - EDGE) * (2 * EDGE));
    if(c >= EDGE) c = width - 2 * EDGE + c;
  }
  const ring_t q = { in, width, height, filters };
  const int d = ring_dist(q, r, c);
  const int s = fc(r, c, filters);
  float px[3];
  if(d < 3)
  {
    px[0] = ring_mean(q, r, c, 0);
    px[2] = ring_mean(q, r, c, 2);
  }
  else
  {
    px[0] = px[2] = 0.0f;
    if(s == 0 || s == 2) px[s] = ring_raw(q, r, c);
  }
  px[1] = ring_green(q, r, c);
  if(d >= 1)
  {
    const float g = px[1];
    if(s & 1)
    {
      const float gt = ring_green(q, r - 1, c), gb = ring_green(q, r + 1, c);
      const float gl = ring_green(q, r, c - 1), gr = ring_green(q, r, c + 1);
      if(fc(r, c + 1, filters) == 0)
      {
        px[2] = (ring_chan(q, r - 1, c, 2) + ring_chan(q, r + 1, c, 2) + 2.0f * g - gt - gb) * .5f;
        px[0] = (ring_chan(q, r, c - 1, 0) + ring_chan(q, r, c + 1, 0) + 2.0f * g - gl - gr) * .5f;
      }
      else
      {
        px[0] = (ring_chan(q, r - 1, c, 0) + ring_chan(q, r + 1, c, 0) + 2.0f * g - gt - gb) * .5f;
        px[2] = (ring_chan(q, r, c - 1, 2) + ring_chan(q, r, c + 1, 2) + 2.0f * g - gl - gr) * .5f;
      }
    }
    else
    {
      const int k2 = (s == 0) ? 2 : 0;
      const float tl = ring_chan(q, r - 1, c - 1, k2), tr = ring_chan(q, r - 1, c + 1, k2);
      const float bl = ring_chan(q, r + 1, c - 1, k2), br = ring_chan(q, r + 1, c + 1, k2);
      const float gtl = ring_green(q, r - 1, c - 1), gtr = ring_green(q, r - 1, c + 1);
      const float gbl = ring_green(q, r + 1, c - 1), gbr = ring_green(q, r + 1, c + 1);
      const float diff1 = fabsf(tl - br) + fabsf(gtl - g) + fabsf(gbr - g);
      const float guess1 = tl + br + 2.0f * g - gtl - gbr;
      const float diff2 = fabsf(tr - bl) + fabsf(gtr - g) + fabsf(gbl - g);
      const float guess2 = tr + bl + 2.0f * g - gtr - gbl;
      float v;
      if(diff1 > diff2)
        v = guess2 * .5f;
      else if(diff1 < diff2)
        v = guess1 * .5f;
      else
        v = (guess1 + guess2) * .25f;
      px[k2] = v;
    }
  }
  // alpha: the reference leaves the outer 3 px as it found them; 0 is what a zeroed cacheline gives
  *reinterpret_cast<float4 *>(out + 4 * ((size_t)r * width + c)) = make_float4(px[0], px[1], px[2], 0.0f);
}

bool standard_bayer(uint32_t f)
{
  // 2x2-periodic, greens on one diagonal, red and blue on the other
  for(int r = 0; r < 8; r++)
    for(int c = 0; c < 2; c++)
      if(b200_fc(r, c, f) != b200_fc(r & 1, c, f)) return false;
  const int a = b200_fc(0, 0, f), b = b200_fc(0, 1, f), c = b200_fc(1, 0, f), d = b200_fc(1, 1, f);
  if(a == 1 && d == 1) return (b == 0 && c == 2) || (b == 2 && c == 0);
  if(b == 1 && c == 1) return (a == 0 && d == 2) || (a == 2 && d == 0);
  return false;
}
} // namespace

namespace b200
{
// rcd_demosaic(), rcd.c:274-564.  `filters` already carries the ROI phase.
int rcd_demosaic_dev(const float *d_in, float *d_out, int width, int height, uint32_t filters,
                     const float processed_maximum[3], cudaStream_t stream)
{
  if(width < 16 || height < 16) return B200_OK; // "too small area": the reference returns with the output untouched (rcd.c:280-284)
  if(!standard_bayer(filters))
    return fail(B200_ERR_UNSUPPORTED, "RCD: filters 0x%08x is not a 2x2 Bayer pattern", filters);

  static std::atomic<bool> attr_set[16] = {}; // per device; setting it twice from two threads is harmless
  int dev = 0;
  B200_CUDA_TRY(cudaGetDevice(&dev));
  const int smem_bytes = SMEM_FLOATS * (int)sizeof(float);
  if(!attr_set[dev & 15].load(std::memory_order_acquire))
  {
    B200_CUDA_TRY(cudaFuncSetAttribute(rcd_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    attr_set[dev & 15].store(true, std::memory_order_release);
  }

  const long long ring_px = 2LL * EDGE * width + 2LL * EDGE * (height - 2 * EDGE);
  rcd_ring_kernel<<<(unsigned)((ring_px + 127) / 128), 128, 0, stream>>>(d_in, d_out, width, height, filters);
  B200_CUDA_TRY(cudaGetLastError());

  rcd_args_t a;
  a.in = d_in;
  a.out = d_out;
  a.width = width;
  a.height = height;
  a.filters = filters;
  a.scaler = fmaxf(processed_maximum[0], fmaxf(processed_maximum[1], processed_maximum[2]));
  a.revscaler = 1.0f / a.scaler;
  a.nv = 1 + (height - 2 * RING - 1) / KEEP;
  a.nh = 1 + (width - 2 * RING - 1) / KEEP;
  {
    timed_launch timed(TIMED_RCD, stream);
    rcd_tiles_kernel<<<(unsigned)(a.nv * a.nh), NT, smem_bytes, stream>>>(a);
  }
  B200_CUDA_TRY(cudaGetLastError());
  return B200_OK;
}
} // namespace b200
