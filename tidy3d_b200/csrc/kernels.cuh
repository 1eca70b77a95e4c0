// Device kernels of the B200 mode solver (sm_100a).  All kernels are batched: blockIdx.z (or .y for
// the 1-D kernels) is the problem index inside a batch of same-shaped eigenproblems.
//
// Vector layout: a "batched vector" is [B][2][nx][ny] (Ex then Ey, y fastest), scalar type T (double
// or cplx).  Coefficient fields are [B or 1][nf][nx][ny] of type C (double or cplx).  The 1-D
// difference coefficients are [B][4][n] of type T per axis (f0, f1, b0, bm).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

namespace b200ms {

// ------------------------------------------------------------------------------------------------
// scalar helpers
// ------------------------------------------------------------------------------------------------
struct __align__(16) cplx {
  double re, im;
};
#define HD __host__ __device__ __forceinline__
HD cplx mk(double r, double i) { cplx c; c.re = r; c.im = i; return c; }
HD cplx operator+(cplx a, cplx b) { return mk(a.re + b.re, a.im + b.im); }
HD cplx operator-(cplx a, cplx b) { return mk(a.re - b.re, a.im - b.im); }
HD cplx operator-(cplx a) { return mk(-a.re, -a.im); }
HD cplx operator*(cplx a, cplx b) { return mk(a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re); }
HD cplx operator*(double a, cplx b) { return mk(a * b.re, a * b.im); }
HD cplx operator*(cplx a, double b) { return mk(a.re * b, a.im * b); }
HD cplx &operator+=(cplx &a, cplx b) { a.re += b.re; a.im += b.im; return a; }
HD cplx &operator-=(cplx &a, cplx b) { a.re -= b.re; a.im -= b.im; return a; }
HD double cj(double a) { return a; }
HD cplx cj(cplx a) { return mk(a.re, -a.im); }
HD double recip(double a) { return 1.0 / a; }
HD cplx recip(cplx a) { double d = 1.0 / (a.re * a.re + a.im * a.im); return mk(a.re * d, -a.im * d); }
HD double abs2(double a) { return a * a; }
HD double abs2(cplx a) { return a.re * a.re + a.im * a.im; }
// single-precision twins (multigrid preconditioner in fp32)
struct __align__(8) cplxf {
  float re, im;
};
HD cplxf mkf(float r, float i) { cplxf c; c.re = r; c.im = i; return c; }
HD cplxf operator+(cplxf a, cplxf b) { return mkf(a.re + b.re, a.im + b.im); }
HD cplxf operator-(cplxf a, cplxf b) { return mkf(a.re - b.re, a.im - b.im); }
HD cplxf operator-(cplxf a) { return mkf(-a.re, -a.im); }
HD cplxf operator*(cplxf a, cplxf b) { return mkf(a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re); }
HD cplxf operator*(float a, cplxf b) { return mkf(a * b.re, a * b.im); }
HD cplxf operator*(cplxf a, float b) { return mkf(a.re * b, a.im * b); }
HD cplxf operator*(double a, cplxf b) { return mkf((float)a * b.re, (float)a * b.im); }
HD cplxf &operator+=(cplxf &a, cplxf b) { a.re += b.re; a.im += b.im; return a; }
HD cplxf &operator-=(cplxf &a, cplxf b) { a.re -= b.re; a.im -= b.im; return a; }
HD float cj(float a) { return a; }
HD cplxf cj(cplxf a) { return mkf(a.re, -a.im); }
HD float recip(float a) { return 1.0f / a; }
HD cplxf recip(cplxf a) { float d = 1.0f / (a.re * a.re + a.im * a.im); return mkf(a.re * d, -a.im * d); }
HD double abs2(float a) { return (double)a * a; }
HD double abs2(cplxf a) { return (double)a.re * a.re + (double)a.im * a.im; }
HD double real_part(double a) { return a; }
HD double real_part(cplx a) { return a.re; }
HD double real_part(float a) { return a; }
HD double real_part(cplxf a) { return a.re; }
// precision conversion between the Krylov (fp64) and multigrid (fp32) vector types
HD void convert(double s, double &d) { d = s; }
HD void convert(double s, float &d) { d = (float)s; }
HD void convert(float s, double &d) { d = s; }
HD void convert(float s, float &d) { d = s; }
HD void convert(cplx s, cplx &d) { d = s; }
HD void convert(cplx s, cplxf &d) { d = mkf((float)s.re, (float)s.im); }
HD void convert(cplxf s, cplx &d) { d = mk(s.re, s.im); }
HD void convert(cplxf s, cplxf &d) { d = s; }

// real scalar type matching a vector element type (transfer weights are converted to it once per thread: with double
// weights the fp32 transfer kernels were instruction-bound on F2F conversions and DFMAs, profiles/r02_restrict_ncu.txt)
template <typename T> struct RealOf { using type = double; };
template <> struct RealOf<float> { using type = float; };
template <> struct RealOf<cplxf> { using type = float; };

template <typename T> HD T zero_of();
template <> HD float zero_of<float>() { return 0.0f; }
template <> HD cplxf zero_of<cplxf>() { return mkf(0.0f, 0.0f); }
template <> HD double zero_of<double>() { return 0.0; }
template <> HD cplx zero_of<cplx>() { return mk(0.0, 0.0); }
template <typename T> HD T from_real(double r);
template <> HD float from_real<float>(double r) { return (float)r; }
template <> HD cplxf from_real<cplxf>(double r) { return mkf((float)r, 0.0f); }
template <> HD double from_real<double>(double r) { return r; }
template <> HD cplx from_real<cplx>(double r) { return mk(r, 0.0); }
// conversions between storage types (real <- complex drops the imaginary part)
template <typename T> HD T cast_to(cplx v);
template <> HD double cast_to<double>(cplx v) { return v.re; }
template <> HD cplx cast_to<cplx>(cplx v) { return v; }
HD cplx to_cplx(double v) { return mk(v, 0.0); }
HD cplx to_cplx(cplx v) { return v; }
// any of the four vector scalar types <-> double-complex (small dense work is always done in cplx)
HD cplx to_cplx_any(double v) { return mk(v, 0.0); }
HD cplx to_cplx_any(float v) { return mk((double)v, 0.0); }
HD cplx to_cplx_any(cplx v) { return v; }
HD cplx to_cplx_any(cplxf v) { return mk((double)v.re, (double)v.im); }
template <typename U> HD U from_cplx_any(cplx v);
template <> HD double from_cplx_any<double>(cplx v) { return v.re; }
template <> HD float from_cplx_any<float>(cplx v) { return (float)v.re; }
template <> HD cplx from_cplx_any<cplx>(cplx v) { return v; }
template <> HD cplxf from_cplx_any<cplxf>(cplx v) { return mkf((float)v.re, (float)v.im); }

template <typename T> __device__ __forceinline__ T ldg(const T *p) { return *p; }
template <> __device__ __forceinline__ double ldg<double>(const double *p) { return __ldg(p); }
template <> __device__ __forceinline__ cplx ldg<cplx>(const cplx *p) {
  double2 v = __ldg(reinterpret_cast<const double2 *>(p));
  return mk(v.x, v.y);
}

template <> __device__ __forceinline__ float ldg<float>(const float *p) { return __ldg(p); }
template <> __device__ __forceinline__ cplxf ldg<cplxf>(const cplxf *p) {
  float2 v = __ldg(reinterpret_cast<const float2 *>(p));
  return mkf(v.x, v.y);
}
__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ cplx warp_sum(cplx v) { return mk(warp_sum(v.re), warp_sum(v.im)); }
__device__ __forceinline__ cplxf warp_sum(cplxf v) { return mkf(warp_sum(v.re), warp_sum(v.im)); }

// y = a .* b element-wise;  fill
template <typename T>
__global__ void __launch_bounds__(256) mul_kernel(size_t total, const T *a, const T *b, T *y) {
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < total; e += stride) y[e] = ldg(a + e) * ldg(b + e);
}
template <typename T>
__global__ void __launch_bounds__(256) fill_kernel(size_t total, T v, T *y) {
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < total; e += stride) y[e] = v;
}

// dst = (D) src, element-wise over a batched vector
template <typename S, typename D>
__global__ void __launch_bounds__(256) convert_kernel(size_t total, const S *src, D *dst) {
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < total; e += stride) {
    D d;
    convert(src[e], d);
    dst[e] = d;
  }
}

// ------------------------------------------------------------------------------------------------
// fused curl-curl stencil
// ------------------------------------------------------------------------------------------------
// _D: stored omega/diag.  _D0: two sweeps from a zero guess in one pass, x' = x0 + dinv (rhs - (A-sigma) x0) with x0 = dinv rhs formed
// while the rows are loaded (replaces the separate dinv*rhs product kernel and the x read of the first sweep)
enum { MODE_APPLY = 0, MODE_RESID = 1, MODE_JACOBI = 2, MODE_JACOBI_D = 3, MODE_JACOBI_D0 = 4 };

template <typename T, typename C>
struct StencilArgs {
  int nx, ny;
  const T *x;        // [B][2][N] input vector
  const T *rhs;      // [B][2][N] (RESID / JACOBI)
  T *y;              // [B][2][N] output
  const C *fields;   // exx, eyy, iez, (mxx, myy, imz)   [field_bstride*b + k*N]
  size_t field_bstride;
  const T *cx;       // [B][4][nx]
  const T *cy;       // [B][4][ny]
  const T *sigma;    // [B]
  double omega;      // Jacobi damping
  const T *dinv;     // [B][2][N] omega / diag(A - sigma) (MODE_JACOBI_D)
};

template <typename T> struct Tile;
template <> struct Tile<double> { static constexpr int TX = 8, TY = 64; };
template <> struct Tile<cplx> { static constexpr int TX = 8, TY = 32; };
template <> struct Tile<float> { static constexpr int TX = 8, TY = 64; };
template <> struct Tile<cplxf> { static constexpr int TX = 8, TY = 64; };

// y = (A - sigma) x                       MODE_APPLY
// y = rhs - (A - sigma) x                 MODE_RESID
// y = x + omega * D^-1 (rhs - (A-sigma)x) MODE_JACOBI   (D = diag(A) - sigma, recomputed on the fly)
//
// A v for v = [Ex; Ey] in the radius-1 form (DESIGN.md section 3):
//   t = imz * (Dxf v2 - Dyf v1)                      (Hz sites)
//   u = -iez * (Dxb (exx v1) + Dyb (eyy v2))         (Ez sites)
//   p1 = Dxf u + myy * (Dyb t - exx v1),  p2 = Dyf u - mxx * (Dxb t + eyy v2)
// which equals P.Q of tidy3d/plugins/mode/solver.py:479-490 (the Dxb Dyb - Dyb Dxb terms cancel).
// One CTA computes a TX x TY tile: the halo of v, exx*v1, eyy*v2 is staged in shared memory, then
// u and t on the (TX+1) x (TY+1) dual tiles, then the outputs.
template <typename T, typename C, int MODE, bool HAS_MU>
__global__ void __launch_bounds__(256) stencil_kernel(StencilArgs<T, C> a) {
  constexpr int TX = Tile<T>::TX, TY = Tile<T>::TY;
  constexpr int RY = 256 / TY;       // thread rows
  constexpr int PER = TX / RY;       // output rows per thread
  constexpr int HW = TY + 2, HH = TX + 2;
  __shared__ T sV1[HH][HW], sV2[HH][HW], sA[HH][HW], sB[HH][HW];
  __shared__ T sU[TX + 1][TY + 1], sT[TX + 1][TY + 1];
  __shared__ C sIez[(MODE == MODE_JACOBI) ? TX + 1 : 1][(MODE == MODE_JACOBI) ? TY + 1 : 1];
  __shared__ C sImz[(MODE == MODE_JACOBI && HAS_MU) ? TX + 1 : 1][(MODE == MODE_JACOBI && HAS_MU) ? TY + 1 : 1];
  __shared__ T sCx[4][HH + 1], sCy[4][HW + 1];

  const int nx = a.nx, ny = a.ny;
  const size_t N = (size_t)nx * ny;
  const int b = blockIdx.z;
  const int i0 = blockIdx.y * TX, j0 = blockIdx.x * TY;
  const int tid = threadIdx.y * TY + threadIdx.x;
  const T *x1 = a.x + (size_t)b * 2 * N, *x2 = x1 + N;
  const C *fb = a.fields + a.field_bstride * b;
  const C *exx = fb, *eyy = fb + N, *iez = fb + 2 * N;
  const C *mxx = fb + 3 * N, *myy = fb + 4 * N, *imz = fb + 5 * N;
  const T *cx = a.cx + (size_t)b * 4 * nx, *cy = a.cy + (size_t)b * 4 * ny;

  // 1-D coefficients for rows i0-1 .. i0+TX+1 and columns j0-1 .. j0+TY+1 (zero outside the grid)
  for (int k = tid; k < 4 * (HH + 1); k += 256) {
    int w = k / (HH + 1), r = k % (HH + 1), gi = i0 - 1 + r;
    sCx[w][r] = (gi >= 0 && gi < nx) ? ldg(cx + (size_t)w * nx + gi) : zero_of<T>();
  }
  for (int k = tid; k < 4 * (HW + 1); k += 256) {
    int w = k / (HW + 1), c = k % (HW + 1), gj = j0 - 1 + c;
    sCy[w][c] = (gj >= 0 && gj < ny) ? ldg(cy + (size_t)w * ny + gj) : zero_of<T>();
  }
  // halo of v and eps*v
  for (int k = tid; k < HH * HW; k += 256) {
    int r = k / HW, c = k % HW, gi = i0 - 1 + r, gj = j0 - 1 + c;
    T v1 = zero_of<T>(), v2 = zero_of<T>(), pa = zero_of<T>(), pb = zero_of<T>();
    if (gi >= 0 && gi < nx && gj >= 0 && gj < ny) {
      size_t g = (size_t)gi * ny + gj;
      v1 = ldg(x1 + g);
      v2 = ldg(x2 + g);
      pa = ldg(exx + g) * v1;
      pb = ldg(eyy + g) * v2;
    }
    sV1[r][c] = v1; sV2[r][c] = v2; sA[r][c] = pa; sB[r][c] = pb;
  }
  __syncthreads();
  // dual tiles: u at (i0+r, j0+c), t at (i0-1+r, j0-1+c), r in [0,TX], c in [0,TY]
  for (int k = tid; k < (TX + 1) * (TY + 1); k += 256) {
    int r = k / (TY + 1), c = k % (TY + 1);
    {
      int gi = i0 + r, gj = j0 + c;
      T u = zero_of<T>();
      C ie = C();
      if (gi < nx && gj < ny) {
        ie = ldg(iez + (size_t)gi * ny + gj);
        T acc = sCx[2][r + 1] * sA[r + 1][c + 1] + sCx[3][r + 1] * sA[r][c + 1] +
                sCy[2][c + 1] * sB[r + 1][c + 1] + sCy[3][c + 1] * sB[r + 1][c];
        u = -(ie * acc);
      }
      sU[r][c] = u;
      if (MODE == MODE_JACOBI) sIez[r][c] = ie;
    }
    {
      int gi = i0 - 1 + r, gj = j0 - 1 + c;
      T t = zero_of<T>();
      C im = C();
      if (gi >= 0 && gi < nx && gj >= 0 && gj < ny) {
        T acc = sCx[0][r] * sV2[r][c] + sCx[1][r] * sV2[r + 1][c] - sCy[0][c] * sV1[r][c] - sCy[1][c] * sV1[r][c + 1];
        if (HAS_MU) {
          im = ldg(imz + (size_t)gi * ny + gj);
          t = im * acc;
        } else {
          t = acc;
        }
      }
      sT[r][c] = t;
      if (MODE == MODE_JACOBI && HAS_MU) sImz[r][c] = im;
    }
  }
  __syncthreads();
  const T sg = ldg(a.sigma + b);
  T *y1 = a.y + (size_t)b * 2 * N, *y2 = y1 + N;
  const T *r1 = (MODE != MODE_APPLY) ? a.rhs + (size_t)b * 2 * N : nullptr;
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const int r = threadIdx.y + q * RY, c = threadIdx.x;
    const int gi = i0 + r, gj = j0 + c;
    if (gi >= nx || gj >= ny) continue;
    const size_t g = (size_t)gi * ny + gj;
    const T u00 = sU[r][c], u10 = sU[r + 1][c], u01 = sU[r][c + 1];
    const T t00 = sT[r + 1][c + 1], t0m = sT[r + 1][c], tm0 = sT[r][c + 1];
    const T pa = sA[r + 1][c + 1], pb = sB[r + 1][c + 1];
    const T v1 = sV1[r + 1][c + 1], v2 = sV2[r + 1][c + 1];
    const T xf0 = sCx[0][r + 1], xf1 = sCx[1][r + 1], xb0 = sCx[2][r + 1], xbm = sCx[3][r + 1];
    const T yf0 = sCy[0][c + 1], yf1 = sCy[1][c + 1], yb0 = sCy[2][c + 1], ybm = sCy[3][c + 1];
    T p1 = xf0 * u00 + xf1 * u10;
    T p2 = yf0 * u00 + yf1 * u01;
    T c1 = yb0 * t00 + ybm * t0m - pa;
    T c2 = xb0 * t00 + xbm * tm0 + pb;
    C mx = C(), my = C();
    if (HAS_MU) {
      mx = ldg(mxx + g);
      my = ldg(myy + g);
      p1 += my * c1;
      p2 -= mx * c2;
    } else {
      p1 += c1;
      p2 -= c2;
    }
    T o1 = p1 - sg * v1, o2 = p2 - sg * v2;
    if (MODE == MODE_APPLY) {
      y1[g] = o1;
      y2[g] = o2;
    } else if (MODE == MODE_RESID) {
      y1[g] = ldg(r1 + g) - o1;
      y2[g] = ldg(r1 + N + g) - o2;
    } else {
      const C ex = ldg(exx + g), ey = ldg(eyy + g);
      const T xbm_n = sCx[3][r + 2], ybm_n = sCy[3][c + 2];  // xbm[i+1], ybm[j+1]
      const T xf1_p = sCx[1][r], yf1_p = sCy[1][c];          // xf1[i-1], yf1[j-1]
      T s1 = sIez[r][c] * (xf0 * xb0) + sIez[r + 1][c] * (xf1 * xbm_n);
      T s2 = sIez[r][c] * (yf0 * yb0) + sIez[r][c + 1] * (yf1 * ybm_n);
      T d1, d2;
      if (HAS_MU) {
        T m1 = sImz[r + 1][c + 1] * (yb0 * yf0) + sImz[r + 1][c] * (ybm * yf1_p);
        T m2 = sImz[r + 1][c + 1] * (xb0 * xf0) + sImz[r][c + 1] * (xbm * xf1_p);
        d1 = -(ex * s1) - my * m1 - (my * ex) * from_real<T>(1.0) - sg;
        d2 = -(ey * s2) - mx * m2 - (mx * ey) * from_real<T>(1.0) - sg;
      } else {
        T m1 = yb0 * yf0 + ybm * yf1_p;
        T m2 = xb0 * xf0 + xbm * xf1_p;
        d1 = -(ex * s1) - m1 - ex * from_real<T>(1.0) - sg;
        d2 = -(ey * s2) - m2 - ey * from_real<T>(1.0) - sg;
      }
      y1[g] = v1 + a.omega * (recip(d1) * (ldg(r1 + g) - o1));
      y2[g] = v2 + a.omega * (recip(d2) * (ldg(r1 + N + g) - o2));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Marching variant of the fused stencil (the production kernel on grids with nx >= 32).
// One thread per grid column (y index), 128 columns per CTA of which the inner 126 produce output; the
// CTA marches over TXR rows.  Own-column neighbours (i-1, i+1) live in registers; the four values each
// cell needs from its y-neighbours (eyy*v2 and v1 for u/t, then u and t themselves) are exchanged
// through double-buffered shared-memory rows, one __syncthreads per row.  Per cell: 5 (+3 with mu)
// coalesced global loads, 4 shared stores + 4 shared loads, ~35 fp64 FMAs, 2 global stores.
// Software pipeline per iteration k (row index):
//   step 0  row k+2 arrives from the prefetch registers; loads of row k+3 are issued
//   step 1  publish b[k+2], v1[k+2]
//   step 2  u[k+1], t[k+1] from registers + neighbours published in iteration k-1; publish them
//   step 3  outputs of row k from u[k], u[k+1], t[k], t[k-1] (registers) and u[k][j+1], t[k][j-1]
// ------------------------------------------------------------------------------------------------
constexpr int kMarchCols = 128, kMarchOut = 126;

// Measured alternatives (bench.py --stencil-only, 32 x 512^2): a two-deep software prefetch (89 registers) ran the fp64
// apply at 126 us and forcing 8 CTAs/SM through __launch_bounds__ (64 registers, small spills) at 131 us, against
// 108 us for this one-deep version at 72 registers; occupancy and register pressure trade off right here.
template <typename T, typename C, int MODE, bool HAS_MU, int TXR>
__global__ void __launch_bounds__(kMarchCols) stencil_march_kernel(StencilArgs<T, C> a) {
  constexpr bool JAC = (MODE == MODE_JACOBI);
  __shared__ T sB[2][kMarchCols + 2], sV[2][kMarchCols + 2], sU[2][kMarchCols + 2], sTt[2][kMarchCols + 2];
  __shared__ C sIe[JAC ? 2 : 1][JAC ? kMarchCols + 2 : 1];
  __shared__ C sIm[(JAC && HAS_MU) ? 2 : 1][(JAC && HAS_MU) ? kMarchCols + 2 : 1];
  __shared__ T sX[4][TXR + 6];

  const int nx = a.nx, ny = a.ny;
  const size_t N = (size_t)nx * ny;
  const int b = blockIdx.z;
  const int c = threadIdx.x;
  const int gj = (int)blockIdx.x * kMarchOut - 1 + c;
  const int i0 = blockIdx.y * TXR;
  const int iend = (i0 + TXR < nx) ? i0 + TXR : nx;
  const bool colv = (gj >= 0 && gj < ny);
  const bool outc = colv && c >= 1 && c <= kMarchOut;
  const T *x1 = a.x + (size_t)b * 2 * N, *x2 = x1 + N;
  const C *fb = a.fields + a.field_bstride * b;
  const C *exx = fb, *eyy = fb + N, *iez = fb + 2 * N;
  const C *mxx = fb + 3 * N, *myy = fb + 4 * N, *imz = fb + 5 * N;
  const T *cx = a.cx + (size_t)b * 4 * nx, *cy = a.cy + (size_t)b * 4 * ny;
  const T zT = zero_of<T>();

  for (int q = c; q < 4 * (TXR + 6); q += kMarchCols) {
    const int w = q / (TXR + 6), r = q % (TXR + 6), gi = i0 - 3 + r;
    sX[w][r] = (gi >= 0 && gi < nx) ? ldg(cx + (size_t)w * nx + gi) : zT;
  }
  for (int s = 0; s < 2; ++s) {
    sB[s][c + 1] = zT; sV[s][c + 1] = zT; sU[s][c + 1] = zT; sTt[s][c + 1] = zT;
    if (JAC) sIe[s][c + 1] = C();
    if (JAC && HAS_MU) sIm[s][c + 1] = C();
  }
  if (c < 2) {
    for (int s = 0; s < 2; ++s) {
      const int e = c == 0 ? 0 : kMarchCols + 1;
      sB[s][e] = zT; sV[s][e] = zT; sU[s][e] = zT; sTt[s][e] = zT;
      if (JAC) sIe[s][e] = C();
      if (JAC && HAS_MU) sIm[s][e] = C();
    }
  }
  T yf0 = zT, yf1 = zT, yb0 = zT, ybm = zT, ybm_n = zT, yf1_p = zT;
  if (colv) {
    yf0 = ldg(cy + gj); yf1 = ldg(cy + ny + gj); yb0 = ldg(cy + 2 * ny + gj); ybm = ldg(cy + 3 * ny + gj);
    if (JAC) {
      if (gj + 1 < ny) ybm_n = ldg(cy + 3 * ny + gj + 1);
      if (gj > 0) yf1_p = ldg(cy + ny + gj - 1);
    }
  }
  const T sg = ldg(a.sigma + b);
  T *y1 = a.y + (size_t)b * 2 * N, *y2 = y1 + N;
  const T *r1 = (MODE != MODE_APPLY) ? a.rhs + (size_t)b * 2 * N : nullptr;
  const T *dv0 = (MODE == MODE_JACOBI_D || MODE == MODE_JACOBI_D0) ? a.dinv + (size_t)b * 2 * N : nullptr;
  constexpr bool DSTORED = (MODE == MODE_JACOBI_D || MODE == MODE_JACOBI_D0);

  // prefetch registers (raw row), rows k+2 / k+1 / k
  T pv1 = zT, pv2 = zT;
  C pex = C(), pey = C(), pie = C(), pim = C(), pmx = C(), pmy = C();
  T a1 = zT, b1 = zT, v11 = zT, v21 = zT, a0 = zT, b0 = zT, v10 = zT, v20 = zT;
  C ie1 = C(), ie0 = C(), im1 = C(), im0 = C(), imm = C(), mx1 = C(), my1 = C(), mx0 = C(), my0 = C();
  C ex1 = C(), ey1 = C(), ex0 = C(), ey0 = C();
  T u0 = zT, t0 = zT, tm = zT;
  T nr1 = zT, nr2 = zT, nd1 = zT, nd2 = zT;

  auto load_row = [&](int gi) {
    pv1 = zT; pv2 = zT; pex = C(); pey = C(); pie = C();
    if (HAS_MU) { pim = C(); pmx = C(); pmy = C(); }
    if (colv && gi >= 0 && gi < nx && gi >= i0 - 1 && gi <= i0 + TXR) {
      const size_t g = (size_t)gi * ny + gj;
      if (MODE == MODE_JACOBI_D0) {  // x0 = dinv * rhs formed on the fly
        pv1 = ldg(dv0 + g) * ldg(r1 + g);
        pv2 = ldg(dv0 + N + g) * ldg(r1 + N + g);
      } else {
        pv1 = ldg(x1 + g); pv2 = ldg(x2 + g);
      }
      pex = ldg(exx + g); pey = ldg(eyy + g); pie = ldg(iez + g);
      if (HAS_MU) { pim = ldg(imz + g); pmx = ldg(mxx + g); pmy = ldg(myy + g); }
    }
  };
  load_row(i0 - 1);
  __syncthreads();

  for (int k = i0 - 3; k < iend; ++k) {
    const int s = k & 1, sp = s ^ 1;
    const int xr = k - (i0 - 3);  // index of row k in sX
    // step 0: row k+2 out of the prefetch registers, then prefetch row k+3 (and rhs of row k+1)
    const T v12 = pv1, v22 = pv2;
    const T a2 = pex * pv1, b2 = pey * pv2;
    const C ie2 = pie, im2 = pim, mx2 = pmx, my2 = pmy, ex2 = pex, ey2 = pey;
    load_row(k + 3);
    T cr1 = nr1, cr2 = nr2, cd1 = nd1, cd2 = nd2;
    if (MODE != MODE_APPLY) {
      nr1 = zT; nr2 = zT;
      if (outc && k + 1 >= i0 && k + 1 < iend) {
        const size_t g = (size_t)(k + 1) * ny + gj;
        nr1 = ldg(r1 + g); nr2 = ldg(r1 + N + g);
        if (DSTORED) { nd1 = ldg(dv0 + g); nd2 = ldg(dv0 + N + g); }
      }
    }
    // step 1
    sB[s][c + 1] = b2;
    sV[s][c + 1] = v12;
    // step 2: u[k+1], t[k+1]
    const T bl = sB[sp][c], v1r = sV[sp][c + 2];
    const T xf0n = sX[0][xr + 1], xf1n = sX[1][xr + 1], xb0n = sX[2][xr + 1], xbmn = sX[3][xr + 1];
    T u1 = -(ie1 * (xb0n * a1 + xbmn * a0 + yb0 * b1 + ybm * bl));
    T t1 = xf0n * v21 + xf1n * v22 - yf0 * v11 - yf1 * v1r;
    if (HAS_MU) t1 = im1 * t1;
    sU[s][c + 1] = u1;
    sTt[s][c + 1] = t1;
    if (JAC) sIe[s][c + 1] = ie1;
    if (JAC && HAS_MU) sIm[s][c + 1] = im1;
    // step 3: outputs of row k
    if (outc && k >= i0) {
      const T ur = sU[sp][c + 2], tl = sTt[sp][c];
      const T xf0 = sX[0][xr], xf1 = sX[1][xr], xb0 = sX[2][xr], xbm = sX[3][xr];
      T p1 = xf0 * u0 + xf1 * u1;
      T p2 = yf0 * u0 + yf1 * ur;
      const T c1 = yb0 * t0 + ybm * tl - a0;
      const T c2 = xb0 * t0 + xbm * tm + b0;
      if (HAS_MU) { p1 += my0 * c1; p2 -= mx0 * c2; } else { p1 += c1; p2 -= c2; }
      const T o1 = p1 - sg * v10, o2 = p2 - sg * v20;
      const size_t g = (size_t)k * ny + gj;
      if (MODE == MODE_APPLY) {
        y1[g] = o1; y2[g] = o2;
      } else if (MODE == MODE_RESID) {
        y1[g] = cr1 - o1; y2[g] = cr2 - o2;
      } else if (DSTORED) {
        y1[g] = v10 + cd1 * (cr1 - o1); y2[g] = v20 + cd2 * (cr2 - o2);
      } else {
        const T xbm_n = sX[3][xr + 1], xf1_p = sX[1][xr - 1 >= 0 ? xr - 1 : 0];
        const C ier = sIe[sp][c + 2];
        T s1 = ie0 * (xf0 * xb0) + ie1 * (xf1 * xbm_n);
        T s2 = ie0 * (yf0 * yb0) + ier * (yf1 * ybm_n);
        T d1, d2;
        if (HAS_MU) {
          const C iml = sIm[sp][c];
          T m1 = im0 * (yb0 * yf0) + iml * (ybm * yf1_p);
          T m2 = im0 * (xb0 * xf0) + imm * (xbm * xf1_p);
          d1 = -(ex0 * s1) - my0 * m1 - (my0 * ex0) * from_real<T>(1.0) - sg;
          d2 = -(ey0 * s2) - mx0 * m2 - (mx0 * ey0) * from_real<T>(1.0) - sg;
        } else {
          T m1 = yb0 * yf0 + ybm * yf1_p;
          T m2 = xb0 * xf0 + xbm * xf1_p;
          d1 = -(ex0 * s1) - m1 - ex0 * from_real<T>(1.0) - sg;
          d2 = -(ey0 * s2) - m2 - ey0 * from_real<T>(1.0) - sg;
        }
        y1[g] = v10 + a.omega * (recip(d1) * (cr1 - o1));
        y2[g] = v20 + a.omega * (recip(d2) * (cr2 - o2));
      }
    }
    // shift the register pipeline
    tm = t0; t0 = t1; u0 = u1;
    a0 = a1; b0 = b1; v10 = v11; v20 = v21; a1 = a2; b1 = b2; v11 = v12; v21 = v22;
    ie0 = ie1; ie1 = ie2;
    if (HAS_MU) { imm = im0; im0 = im1; im1 = im2; mx0 = mx1; my0 = my1; mx1 = mx2; my1 = my2; }
    if (JAC) { ex0 = ex1; ey0 = ey1; ex1 = ex2; ey1 = ey2; }
    __syncthreads();
  }
}

// y = omega * D^-1 rhs  (first Jacobi sweep from a zero guess; no halo needed)
template <typename T, typename C, bool HAS_MU>
__global__ void __launch_bounds__(256) jacobi0_kernel(StencilArgs<T, C> a) {
  const int nx = a.nx, ny = a.ny;
  const size_t N = (size_t)nx * ny;
  const int b = blockIdx.z;
  const int gj = blockIdx.x * 64 + threadIdx.x, gi = blockIdx.y * 4 + threadIdx.y;
  if (gi >= nx || gj >= ny) return;
  const size_t g = (size_t)gi * ny + gj;
  const C *fb = a.fields + a.field_bstride * b;
  const C *exx = fb, *eyy = fb + N, *iez = fb + 2 * N, *mxx = fb + 3 * N, *myy = fb + 4 * N, *imz = fb + 5 * N;
  const T *cx = a.cx + (size_t)b * 4 * nx, *cy = a.cy + (size_t)b * 4 * ny;
  const T z = zero_of<T>();
  const T xf0 = ldg(cx + gi), xf1 = ldg(cx + nx + gi), xb0 = ldg(cx + 2 * nx + gi), xbm = ldg(cx + 3 * nx + gi);
  const T yf0 = ldg(cy + gj), yf1 = ldg(cy + ny + gj), yb0 = ldg(cy + 2 * ny + gj), ybm = ldg(cy + 3 * ny + gj);
  const T xbm_n = gi + 1 < nx ? ldg(cx + 3 * nx + gi + 1) : z, ybm_n = gj + 1 < ny ? ldg(cy + 3 * ny + gj + 1) : z;
  const T xf1_p = gi > 0 ? ldg(cx + nx + gi - 1) : z, yf1_p = gj > 0 ? ldg(cy + ny + gj - 1) : z;
  const C ie00 = ldg(iez + g);
  const C ie10 = gi + 1 < nx ? ldg(iez + g + ny) : C();
  const C ie01 = gj + 1 < ny ? ldg(iez + g + 1) : C();
  const C ex = ldg(exx + g), ey = ldg(eyy + g);
  const T sg = ldg(a.sigma + b);
  T s1 = ie00 * (xf0 * xb0) + ie10 * (xf1 * xbm_n);
  T s2 = ie00 * (yf0 * yb0) + ie01 * (yf1 * ybm_n);
  T d1, d2;
  if (HAS_MU) {
    const C im00 = ldg(imz + g);
    const C im0m = gj > 0 ? ldg(imz + g - 1) : C();
    const C imm0 = gi > 0 ? ldg(imz + g - ny) : C();
    const C mx = ldg(mxx + g), my = ldg(myy + g);
    T m1 = im00 * (yb0 * yf0) + im0m * (ybm * yf1_p);
    T m2 = im00 * (xb0 * xf0) + imm0 * (xbm * xf1_p);
    d1 = -(ex * s1) - my * m1 - (my * ex) * from_real<T>(1.0) - sg;
    d2 = -(ey * s2) - mx * m2 - (mx * ey) * from_real<T>(1.0) - sg;
  } else {
    T m1 = yb0 * yf0 + ybm * yf1_p;
    T m2 = xb0 * xf0 + xbm * xf1_p;
    d1 = -(ex * s1) - m1 - ex * from_real<T>(1.0) - sg;
    d2 = -(ey * s2) - m2 - ey * from_real<T>(1.0) - sg;
  }
  const T *r1 = a.rhs + (size_t)b * 2 * N;
  T *y1 = a.y + (size_t)b * 2 * N;
  y1[g] = a.omega * (recip(d1) * ldg(r1 + g));
  y1[N + g] = a.omega * (recip(d2) * ldg(r1 + N + g));
}

// ------------------------------------------------------------------------------------------------
// grid transfer (tensor product of 1-D lists, see host_setup.hpp)
// ------------------------------------------------------------------------------------------------
// packed restriction list of one coarse index: up to four (fine index, weight) entries; unused entries repeat a valid index
// with weight zero, so the kernel needs no predicates
struct __align__(16) RList4 {
  int idx[4];
  float w[4];
};
struct Transfer1DDev {
  const int *p_i0, *p_i1;
  const double *p_w0, *p_w1;
  const int *r_ptr, *r_idx;
  const double *r_w;
  const float *p_w0f, *p_w1f;  // the prolongation weights in single precision (fp32 multigrid: no F2F per weight and thread)
  const RList4 *r4;            // packed restriction lists, nullptr when some coarse index has more than four entries
};
struct TransferArgs {
  int nxf, nyf, nxc, nyc;
  Transfer1DDev xn, xe, yn, ye;  // node / edge lists per axis
  int mask_x, mask_y;            // PEC min walls: zero Ey[0,:] (mask_x) and Ex[:,0] (mask_y)
};

// coarse[b][comp] = R fine[b][comp]   (Ex: x edge / y node, Ey: x node / y edge)
// Each thread produces one coarse value from an (up to) 4 x 4 patch of fine values.  The two 1-D lists of the thread
// (<= 4 entries each for the aggregations plan_hierarchy produces: aggregates of <= 3 cells, linear interpolation) are read
// into registers first and the 16 fine loads are issued together (predicated), instead of a doubly nested loop whose every
// term waits on an index load and then on a data load; longer lists fall back to the loop.
template <typename T>
__global__ void __launch_bounds__(256) restrict_kernel(TransferArgs a, const T *fine, T *coarse) {
  const int J = blockIdx.x * 64 + threadIdx.x, I = blockIdx.y * 4 + threadIdx.y;
  const int comp = blockIdx.z & 1, b = blockIdx.z >> 1;
  if (I >= a.nxc || J >= a.nyc) return;
  const Transfer1DDev &tx = comp == 0 ? a.xe : a.xn;
  const Transfer1DDev &ty = comp == 0 ? a.yn : a.ye;
  const size_t Nf = (size_t)a.nxf * a.nyf, Nc = (size_t)a.nxc * a.nyc;
  const T *f = fine + ((size_t)b * 2 + comp) * Nf;
  T acc = zero_of<T>();
  const int kx0 = __ldg(tx.r_ptr + I), kx1 = __ldg(tx.r_ptr + I + 1), ky0 = __ldg(ty.r_ptr + J), ky1 = __ldg(ty.r_ptr + J + 1);
  if (kx1 - kx0 <= 4 && ky1 - ky0 <= 4) {
    using R = typename RealOf<T>::type;
    int iy[4];
    const T *rowp[4];
    R wx[4], wy[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const bool vx = kx0 + q < kx1, vy = ky0 + q < ky1;
      rowp[q] = f + (size_t)(vx ? __ldg(tx.r_idx + kx0 + q) : 0) * a.nyf;
      wx[q] = vx ? (R)__ldg(tx.r_w + kx0 + q) : (R)0;
      iy[q] = vy ? __ldg(ty.r_idx + ky0 + q) : 0;
      wy[q] = vy ? (R)__ldg(ty.r_w + ky0 + q) : (R)0;
    }
    T v[4][4];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int q = 0; q < 4; ++q) v[p][q] = (kx0 + p < kx1 && ky0 + q < ky1) ? ldg(rowp[p] + iy[q]) : zero_of<T>();
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      T racc = zero_of<T>();
#pragma unroll
      for (int q = 0; q < 4; ++q) racc += wy[q] * v[p][q];
      acc += wx[p] * racc;
    }
  } else {
    for (int kx = kx0; kx < kx1; ++kx) {
      const double wxk = tx.r_w[kx];
      const T *row = f + (size_t)tx.r_idx[kx] * a.nyf;
      T racc = zero_of<T>();
      for (int ky = ky0; ky < ky1; ++ky) racc += ty.r_w[ky] * ldg(row + ty.r_idx[ky]);
      acc += wxk * racc;
    }
  }
  if ((comp == 0 && a.mask_y && J == 0 && a.nyc > 1) || (comp == 1 && a.mask_x && I == 0 && a.nxc > 1)) acc = zero_of<T>();
  coarse[((size_t)b * 2 + comp) * Nc + (size_t)I * a.nyc + J] = acc;
}

// Restriction from packed lists (fp32 multigrid).  ncu on restrict_kernel at 64 x 512^2 (profiles/r02_transfers_ncu.txt): 370
// thread instructions per coarse value, issue slots 71 % busy, DRAM at 1.2 TB/s -- the loads of the four list ranges, sixteen
// double -> float weight conversions and the per-term predicates, not the sixteen gathers, set the pace.  Here a coarse index'
// list is one 32-byte record (two 128-bit loads), the weights are fp32, unused entries carry weight zero and a valid index, and the
// sixteen gathers are unconditional.  Same summation order as restrict_kernel, so the results are identical.
template <typename T>
__global__ void __launch_bounds__(256) restrict4_kernel(TransferArgs a, const T *fine, T *coarse) {
  const int J = blockIdx.x * 64 + threadIdx.x, I = blockIdx.y * 4 + threadIdx.y;
  const int comp = blockIdx.z & 1, b = blockIdx.z >> 1;
  if (I >= a.nxc || J >= a.nyc) return;
  const Transfer1DDev &tx = comp == 0 ? a.xe : a.xn;
  const Transfer1DDev &ty = comp == 0 ? a.yn : a.ye;
  const size_t Nf = (size_t)a.nxf * a.nyf, Nc = (size_t)a.nxc * a.nyc;
  const T *f = fine + ((size_t)b * 2 + comp) * Nf;
  const int4 xi = __ldg(reinterpret_cast<const int4 *>(tx.r4 + I)), yi = __ldg(reinterpret_cast<const int4 *>(ty.r4 + J));
  const float4 xw = __ldg(reinterpret_cast<const float4 *>(tx.r4 + I) + 1), yw = __ldg(reinterpret_cast<const float4 *>(ty.r4 + J) + 1);
  const int ix[4] = {xi.x, xi.y, xi.z, xi.w}, iy[4] = {yi.x, yi.y, yi.z, yi.w};
  const float wx[4] = {xw.x, xw.y, xw.z, xw.w}, wy[4] = {yw.x, yw.y, yw.z, yw.w};
  T v[4][4];
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const T *row = f + (size_t)ix[p] * a.nyf;
#pragma unroll
    for (int q = 0; q < 4; ++q) v[p][q] = ldg(row + iy[q]);
  }
  T acc = zero_of<T>();
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    T racc = zero_of<T>();
#pragma unroll
    for (int q = 0; q < 4; ++q) racc += wy[q] * v[p][q];
    acc += wx[p] * racc;
  }
  if ((comp == 0 && a.mask_y && J == 0 && a.nyc > 1) || (comp == 1 && a.mask_x && I == 0 && a.nxc > 1)) acc = zero_of<T>();
  coarse[((size_t)b * 2 + comp) * Nc + (size_t)I * a.nyc + J] = acc;
}

// fine[b][comp] += P coarse[b][comp].  All index / weight loads and the four coarse loads are independent and issued
// before the read-modify-write of the fine value.
template <typename T>
__global__ void __launch_bounds__(256) prolong_add_kernel(TransferArgs a, const T *coarse, T *fine) {
  const int j = blockIdx.x * 64 + threadIdx.x, i = blockIdx.y * 4 + threadIdx.y;
  const int comp = blockIdx.z & 1, b = blockIdx.z >> 1;
  if (i >= a.nxf || j >= a.nyf) return;
  if ((comp == 0 && a.mask_y && j == 0 && a.nyf > 1) || (comp == 1 && a.mask_x && i == 0 && a.nxf > 1)) return;
  const Transfer1DDev &tx = comp == 0 ? a.xe : a.xn;
  const Transfer1DDev &ty = comp == 0 ? a.yn : a.ye;
  const size_t Nf = (size_t)a.nxf * a.nyf, Nc = (size_t)a.nxc * a.nyc;
  const T *c = coarse + ((size_t)b * 2 + comp) * Nc;
  T *f = fine + ((size_t)b * 2 + comp) * Nf + (size_t)i * a.nyf + j;
  const int I0 = __ldg(tx.p_i0 + i), I1 = __ldg(tx.p_i1 + i), J0 = __ldg(ty.p_i0 + j), J1 = __ldg(ty.p_i1 + j);
  using R = typename RealOf<T>::type;
  const R wx0 = (R)__ldg(tx.p_w0 + i), wx1 = (R)__ldg(tx.p_w1 + i), wy0 = (R)__ldg(ty.p_w0 + j), wy1 = (R)__ldg(ty.p_w1 + j);
  const T fv = *f;
  const T c00 = ldg(c + (size_t)I0 * a.nyc + J0), c01 = ldg(c + (size_t)I0 * a.nyc + J1);
  const T c10 = ldg(c + (size_t)I1 * a.nyc + J0), c11 = ldg(c + (size_t)I1 * a.nyc + J1);
  *f = fv + (wx0 * (wy0 * c00 + wy1 * c01) + wx1 * (wy0 * c10 + wy1 * c11));
}

// Four consecutive fine columns per thread: the x-lists and the two coarse row pointers are shared by the four outputs and
// the y-lists are read as 16-byte vectors; the one-output-per-thread version above is instruction-bound on the fine level
// (33.5 M outputs x ~60 instructions at 64 x 512^2).
// VEC (fp32 vectors, nyf % 4 == 0): the four fine values are read and written as one 128-bit access.  With scalar accesses every
// load / store instruction of a warp touches 4 of every 16 bytes over a 512-byte span, so each fine sector is visited by four load
// and four (partial-sector) store instructions.
template <typename T, bool VEC = false>
__global__ void __launch_bounds__(256) prolong_add4_kernel(TransferArgs a, const T *coarse, T *fine) {
  using R = typename RealOf<T>::type;
  const int j4 = blockIdx.x * 64 + threadIdx.x, i = blockIdx.y * 4 + threadIdx.y;
  const int comp = blockIdx.z & 1, b = blockIdx.z >> 1;
  const int j0 = 4 * j4;
  if (i >= a.nxf || j0 >= a.nyf) return;
  const bool row_masked = comp == 1 && a.mask_x && i == 0 && a.nxf > 1;
  if (row_masked) return;
  const Transfer1DDev &tx = comp == 0 ? a.xe : a.xn;
  const Transfer1DDev &ty = comp == 0 ? a.yn : a.ye;
  const size_t Nf = (size_t)a.nxf * a.nyf, Nc = (size_t)a.nxc * a.nyc;
  const T *c = coarse + ((size_t)b * 2 + comp) * Nc;
  const T *c0 = c + (size_t)__ldg(tx.p_i0 + i) * a.nyc, *c1 = c + (size_t)__ldg(tx.p_i1 + i) * a.nyc;
  const R wx0 = (R)__ldg(tx.p_w0 + i), wx1 = (R)__ldg(tx.p_w1 + i);
  T *f = fine + ((size_t)b * 2 + comp) * Nf + (size_t)i * a.nyf + j0;
  int J0[4], J1[4];
  R wy0[4], wy1[4];
  const int nq = min(4, a.nyf - j0);
  if (nq == 4) {
    const int4 q0 = __ldg(reinterpret_cast<const int4 *>(ty.p_i0 + j0)), q1 = __ldg(reinterpret_cast<const int4 *>(ty.p_i1 + j0));
    J0[0] = q0.x; J0[1] = q0.y; J0[2] = q0.z; J0[3] = q0.w;
    J1[0] = q1.x; J1[1] = q1.y; J1[2] = q1.z; J1[3] = q1.w;
    if constexpr (VEC && std::is_same<R, float>::value) {
      const float4 w0 = __ldg(reinterpret_cast<const float4 *>(ty.p_w0f + j0)), w1 = __ldg(reinterpret_cast<const float4 *>(ty.p_w1f + j0));
      wy0[0] = w0.x; wy0[1] = w0.y; wy0[2] = w0.z; wy0[3] = w0.w;
      wy1[0] = w1.x; wy1[1] = w1.y; wy1[2] = w1.z; wy1[3] = w1.w;
    } else {
      const double2 w0a = __ldg(reinterpret_cast<const double2 *>(ty.p_w0 + j0)), w0b = __ldg(reinterpret_cast<const double2 *>(ty.p_w0 + j0 + 2));
      const double2 w1a = __ldg(reinterpret_cast<const double2 *>(ty.p_w1 + j0)), w1b = __ldg(reinterpret_cast<const double2 *>(ty.p_w1 + j0 + 2));
      wy0[0] = (R)w0a.x; wy0[1] = (R)w0a.y; wy0[2] = (R)w0b.x; wy0[3] = (R)w0b.y;
      wy1[0] = (R)w1a.x; wy1[1] = (R)w1a.y; wy1[2] = (R)w1b.x; wy1[3] = (R)w1b.y;
    }
  } else {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = j0 + (q < nq ? q : 0);
      J0[q] = __ldg(ty.p_i0 + j); J1[q] = __ldg(ty.p_i1 + j);
      wy0[q] = (R)__ldg(ty.p_w0 + j); wy1[q] = (R)__ldg(ty.p_w1 + j);
    }
  }
  T fv[4], cv[4][4];
  if constexpr (VEC && std::is_same<T, float>::value) {
    if (nq == 4) {
      const float4 f4 = *reinterpret_cast<const float4 *>(f);
      fv[0] = f4.x; fv[1] = f4.y; fv[2] = f4.z; fv[3] = f4.w;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        cv[q][0] = ldg(c0 + J0[q]); cv[q][1] = ldg(c0 + J1[q]); cv[q][2] = ldg(c1 + J0[q]); cv[q][3] = ldg(c1 + J1[q]);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (comp == 0 && a.mask_y && j0 + q == 0 && a.nyf > 1) continue;
        fv[q] = fv[q] + (wx0 * (wy0[q] * cv[q][0] + wy1[q] * cv[q][1]) + wx1 * (wy0[q] * cv[q][2] + wy1[q] * cv[q][3]));
      }
      *reinterpret_cast<float4 *>(f) = make_float4(fv[0], fv[1], fv[2], fv[3]);
      return;
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (q < nq) {
      fv[q] = f[q];
      cv[q][0] = ldg(c0 + J0[q]); cv[q][1] = ldg(c0 + J1[q]); cv[q][2] = ldg(c1 + J0[q]); cv[q][3] = ldg(c1 + J1[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (q >= nq) continue;
    if (comp == 0 && a.mask_y && j0 + q == 0 && a.nyf > 1) continue;
    f[q] = fv[q] + (wx0 * (wy0[q] * cv[q][0] + wy1[q] * cv[q][1]) + wx1 * (wy0[q] * cv[q][2] + wy1[q] * cv[q][3]));
  }
}

// coefficient field restriction: out = R in (optionally on reciprocals: out = 1 / R (1 / in))
template <typename C>
__global__ void __launch_bounds__(256) restrict_field_kernel(int nxf, int nyf, int nxc, int nyc, Transfer1DDev tx,
                                                             Transfer1DDev ty, const C *in, size_t in_bstride, C *out,
                                                             size_t out_bstride, int reciprocal) {
  const int J = blockIdx.x * 64 + threadIdx.x, I = blockIdx.y * 4 + threadIdx.y, b = blockIdx.z;
  if (I >= nxc || J >= nyc) return;
  const C *f = in + in_bstride * b;
  C acc = C();
  for (int kx = tx.r_ptr[I]; kx < tx.r_ptr[I + 1]; ++kx) {
    const C *row = f + (size_t)tx.r_idx[kx] * nyf;
    C racc = C();
    for (int ky = ty.r_ptr[J]; ky < ty.r_ptr[J + 1]; ++ky) {
      C v = ldg(row + ty.r_idx[ky]);
      if (reciprocal) v = recip(v);
      racc += ty.r_w[ky] * v;
    }
    acc += tx.r_w[kx] * racc;
  }
  if (reciprocal) acc = recip(acc);
  out[out_bstride * b + (size_t)I * nyc + J] = acc;
}

// ------------------------------------------------------------------------------------------------
// batched Krylov vector kernels.  Basis vector i of problem b: V + i*vstride + b*len
// ------------------------------------------------------------------------------------------------
constexpr int kDotGroup = 8;
constexpr int kDotChunks = 64;  // partial sums per problem

// partial[b][chunk][i] = sum_{e in chunk} conj(V_i[b][e]) * w[b][e],  i in [i0, i0+nv)
template <typename T>
__global__ void __launch_bounds__(256) multidot_partial_kernel(const T *V, size_t vstride, size_t len, const T *w,
                                                               int nv, T *partial, int pstride) {
  const int b = blockIdx.y, chunk = blockIdx.x;
  const T *wb = w + (size_t)b * len;
  __shared__ T red[8][kDotGroup];
  const size_t per = (len + gridDim.x - 1) / gridDim.x;
  const size_t e0 = (size_t)chunk * per, e1 = (e0 + per < len) ? e0 + per : len;
  for (int g0 = 0; g0 < nv; g0 += kDotGroup) {
    const int ng = (nv - g0 < kDotGroup) ? nv - g0 : kDotGroup;
    T acc[kDotGroup];
#pragma unroll
    for (int k = 0; k < kDotGroup; ++k) acc[k] = zero_of<T>();
    for (size_t e = e0 + threadIdx.x; e < e1; e += 256) {
      const T we = ldg(wb + e);
#pragma unroll
      for (int k = 0; k < kDotGroup; ++k)
        if (k < ng) acc[k] += cj(ldg(V + (size_t)(g0 + k) * vstride + (size_t)b * len + e)) * we;
    }
#pragma unroll
    for (int k = 0; k < kDotGroup; ++k) {
      T v = warp_sum(acc[k]);
      if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < ng) {
      T s = zero_of<T>();
      for (int wv = 0; wv < 8; ++wv) s += red[wv][threadIdx.x];
      partial[((size_t)b * gridDim.x + chunk) * pstride + g0 + threadIdx.x] = s;
    }
    __syncthreads();
  }
}

// out[b][i] (+)= sum_chunk partial[b][chunk][i]
template <typename T>
__global__ void multidot_final_kernel(const T *partial, int nchunk, int pstride, int nv, T *out, int ostride,
                                      int accumulate) {
  const int b = blockIdx.x, i = threadIdx.x;
  if (i >= nv) return;
  T s = zero_of<T>();
  for (int c = 0; c < nchunk; ++c) s += partial[((size_t)b * nchunk + c) * pstride + i];
  if (accumulate) s += out[(size_t)b * ostride + i];
  out[(size_t)b * ostride + i] = s;
}

// w[b] += sign * sum_i coef[b][i] * V_i[b]
template <typename T>
__global__ void __launch_bounds__(256) multiaxpy_kernel(const T *V, size_t vstride, size_t len, const T *coef,
                                                        int cstride, int nv, double sign, T *w) {
  const int b = blockIdx.y;
  extern __shared__ unsigned char smem_raw[];
  T *sc = reinterpret_cast<T *>(smem_raw);
  for (int i = threadIdx.x; i < nv; i += 256) sc[i] = coef[(size_t)b * cstride + i];
  __syncthreads();
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < len; e += stride) {
    T acc = zero_of<T>();
    for (int i = 0; i < nv; ++i) acc += sc[i] * ldg(V + (size_t)i * vstride + (size_t)b * len + e);
    T *p = w + (size_t)b * len + e;
    *p = *p + sign * acc;
  }
}

// out_k[b] = sum_i Q[b][i][k] * V_i[b],  k in [0, nk); Q row-major [nv][qld]
template <typename T>
__global__ void __launch_bounds__(256) lincomb_kernel(const T *V, size_t vstride, size_t len, const T *Q, int nv,
                                                      int nk, int qld, T *out, size_t ostride) {
  const int b = blockIdx.y;
  extern __shared__ unsigned char smem_raw[];
  T *sq = reinterpret_cast<T *>(smem_raw);
  for (int i = threadIdx.x; i < nv * qld; i += 256) sq[i] = Q[(size_t)b * nv * qld + i];
  __syncthreads();
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < len; e += stride) {
    for (int k0 = 0; k0 < nk; k0 += 8) {
      T acc[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = zero_of<T>();
      for (int i = 0; i < nv; ++i) {
        const T v = ldg(V + (size_t)i * vstride + (size_t)b * len + e);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k0 + k < nk) acc[k] += sq[i * qld + k0 + k] * v;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k0 + k < nk) out[(size_t)(k0 + k) * ostride + (size_t)b * len + e] = acc[k];
    }
  }
}

// y[b] = alpha[b] * x[b]  with alpha = 1/sqrt(re(nrm2[b])) (guarded) when inv_sqrt, else alpha[b]
template <typename T>
__global__ void __launch_bounds__(256) scale_kernel(const T *x, T *y, size_t len, const T *alpha, int astride,
                                                    int inv_sqrt) {
  const int b = blockIdx.y;
  T al = alpha[(size_t)b * astride];
  if (inv_sqrt) {
    const double n2 = real_part(al);
    al = from_real<T>(n2 > 1e-60 ? rsqrt(n2) : 0.0);
  }
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < len; e += stride)
    y[(size_t)b * len + e] = al * ldg(x + (size_t)b * len + e);
}

// y = a*x + b*y (scalars shared by the batch)
template <typename T>
__global__ void __launch_bounds__(256) axpby_kernel(size_t total, double a, const T *x, double bcoef, T *y) {
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < total; e += stride) {
    T v = a * ldg(x + e);
    if (bcoef != 0.0) v = v + bcoef * y[e];
    y[e] = v;
  }
}

// dst[b][i] += src[b][i], i < n (tiny per-problem vectors)
template <typename T>
__global__ void add_small_kernel(T *dst, int dstride, const T *src, int sstride, int n) {
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[(size_t)b * dstride + i] = dst[(size_t)b * dstride + i] + src[(size_t)b * sstride + i];
}

// out[b] = max(0, h[b][nv] - sum_{i<nv} |h[b][i]|^2): squared norm of w after one Gram-Schmidt pass
template <typename T>
__global__ void pythagoras_kernel(const T *h, int hstride, int nv, T *out, int ostride, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const T ww = h[(size_t)b * hstride + nv];
  double acc = real_part(ww);
  for (int i = 0; i < nv; ++i) acc -= abs2(h[(size_t)b * hstride + i]);
  out[(size_t)b * ostride] = from_real<T>(acc > 0.0 ? acc : 0.0);
}

// Least-squares solve of the small GMRES Hessenberg systems, one thread per problem, in place.
// H is [B][kc][ld] column-major by Arnoldi step: H[b][j][i] = h_{i,j} for i <= j, and H[b][j][j+1]
// holds ||w_j||^2 (squared norm, as written by the dot kernel).  beta2[b] = ||r0||^2.
// Output y[b][0..kc).
template <typename T>
__global__ void gmres_lsq_kernel(T *H, int kc, int ld, const T *beta2, int bstride, T *y, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  T *Hb = H + (size_t)b * kc * ld;
  T *yb = y + (size_t)b * kc;
  // g is kept in the unused tail of y? no: use the last column slot of each H column (index ld-1)
  // g[i] lives at Hb[i*ld + ld-1] for i < kc, and g[kc] in a register.
  T b2 = beta2[(size_t)b * bstride];
  double beta = sqrt(fmax(0.0, real_part(b2)));
  T gnext = from_real<T>(beta);
  for (int j = 0; j < kc; ++j) {
    T *col = Hb + (size_t)j * ld;
    // sub-diagonal entry: sqrt of the stored squared norm
    T n2 = col[j + 1];
    double sub = sqrt(fmax(0.0, real_part(n2)));
    // apply previous rotations (stored in columns' slots ld-3 (c) and ld-2 (s))
    for (int i = 0; i < j; ++i) {
      const T c = Hb[(size_t)i * ld + ld - 3], sn = Hb[(size_t)i * ld + ld - 2];
      const T a0 = col[i], a1 = col[i + 1];
      col[i] = cj(c) * a0 + cj(sn) * a1;
      col[i + 1] = c * a1 - sn * a0;
    }
    const T a0 = col[j];
    const double d = sqrt(abs2(a0) + sub * sub);
    T c = from_real<T>(1.0), sn = zero_of<T>();
    if (d > 0.0) {
      c = (1.0 / d) * a0;
      sn = from_real<T>(sub / d);
    }
    col[ld - 3] = c;
    col[ld - 2] = sn;
    col[j] = from_real<T>(d);
    const T gj = gnext;
    col[ld - 1] = cj(c) * gj;   // g[j]
    gnext = -(sn * gj);          // g[j+1]
  }
  // back substitution R y = g
  for (int i = kc - 1; i >= 0; --i) {
    T acc = Hb[(size_t)i * ld + ld - 1];
    for (int j = i + 1; j < kc; ++j) acc -= Hb[(size_t)j * ld + i] * yb[j];
    const T rii = Hb[(size_t)i * ld + i];
    yb[i] = abs2(rii) > 1e-60 ? recip(rii) * acc : zero_of<T>();
  }
}

// ------------------------------------------------------------------------------------------------
// tensorial path (angled waveguides / off-diagonal eps): the 4N first-order operator of solver.py:604-666,
//   mat = msign * (-i) * M,   M [Ex;Ey;Hx;Hy] = [r1;r2;r3;r4]
// written with U = Ez and Tt = Hz of solver.py:708-711:
//   K = Dxb Hy - Dyb Hx,  G = Dxf Ey - Dyf Ex
//   U = K/ezz - (ezx/ezz) Ex - (ezy/ezz) Ey,   Tt = G/mzz - (mzx/mzz) Hx - (mzy/mzz) Hy
//   r1 = Dxf U + (myz/mzz) G + Sm_yx Hx + Sm_yy Hy      r3 = Dxb Tt + (eyz/ezz) K + Se_yx Ex + Se_yy Ey
//   r2 = Dyf U - (mxz/mzz) G - Sm_xx Hx - Sm_xy Hy      r4 = Dyb Tt - (exz/ezz) K - Se_xx Ex - Se_xy Ey
// with S_ab = t_ab - t_az t_zb / t_zz.  Coefficient fields ft[18]: for eps (0..8) and mu (9..17):
//   t_zx/t_zz, t_zy/t_zz, 1/t_zz, t_yz/t_zz, t_xz/t_zz, S_xx, S_xy, S_yx, S_yy.
// Vector layout [B][4][N].  A plain one-thread-per-cell kernel (neighbours through L1); this path is correctness
// first, the diagonal path is the tuned one.
// ------------------------------------------------------------------------------------------------
template <typename C>
struct TensorArgs {
  int nx, ny;
  const cplx *w;
  const cplx *rhs;   // optional: y = rhs - (mat - sigma) w
  cplx *y;
  const C *ft;       // [fb][18][N]
  size_t ft_bstride;
  const cplx *cx, *cy;  // [B][4][n] reference-operator difference coefficients
  const cplx *sigma;    // [B]
  double msign;
};

template <typename C>
struct TensorCell {
  const cplx *ex, *ey, *hx, *hy;
  const C *ft;
  const cplx *cx, *cy;
  int nx, ny;
  size_t N;
  __device__ __forceinline__ cplx ld(const cplx *p, int i, int j) const {
    return (i >= 0 && i < nx && j >= 0 && j < ny) ? ldg(p + (size_t)i * ny + j) : mk(0.0, 0.0);
  }
  __device__ __forceinline__ cplx CX(int w, int i) const { return (i >= 0 && i < nx) ? ldg(cx + (size_t)w * nx + i) : mk(0.0, 0.0); }
  __device__ __forceinline__ cplx CY(int w, int j) const { return (j >= 0 && j < ny) ? ldg(cy + (size_t)w * ny + j) : mk(0.0, 0.0); }
  __device__ __forceinline__ C F(int k, int i, int j) const { return ldg(ft + (size_t)k * N + (size_t)i * ny + j); }
  __device__ __forceinline__ cplx K(int i, int j) const {
    return CX(2, i) * ld(hy, i, j) + CX(3, i) * ld(hy, i - 1, j) - CY(2, j) * ld(hx, i, j) - CY(3, j) * ld(hx, i, j - 1);
  }
  __device__ __forceinline__ cplx G(int i, int j) const {
    return CX(0, i) * ld(ey, i, j) + CX(1, i) * ld(ey, i + 1, j) - CY(0, j) * ld(ex, i, j) - CY(1, j) * ld(ex, i, j + 1);
  }
  __device__ __forceinline__ cplx U(int i, int j) const {
    if (i < 0 || j < 0 || i >= nx || j >= ny) return mk(0.0, 0.0);
    return F(2, i, j) * K(i, j) - F(0, i, j) * ld(ex, i, j) - F(1, i, j) * ld(ey, i, j);
  }
  __device__ __forceinline__ cplx Tt(int i, int j) const {
    if (i < 0 || j < 0 || i >= nx || j >= ny) return mk(0.0, 0.0);
    return F(11, i, j) * G(i, j) - F(9, i, j) * ld(hx, i, j) - F(10, i, j) * ld(hy, i, j);
  }
};

template <typename C>
__global__ void __launch_bounds__(256) tensor_apply_kernel(TensorArgs<C> a) {
  const int nx = a.nx, ny = a.ny;
  const size_t N = (size_t)nx * ny;
  const int j = blockIdx.x * 64 + threadIdx.x, i = blockIdx.y * 4 + threadIdx.y, b = blockIdx.z;
  if (i >= nx || j >= ny) return;
  const cplx *wb = a.w + (size_t)b * 4 * N;
  TensorCell<C> t{wb, wb + N, wb + 2 * N, wb + 3 * N, a.ft + a.ft_bstride * b, a.cx + (size_t)b * 4 * nx, a.cy + (size_t)b * 4 * ny, nx, ny, N};
  const size_t g = (size_t)i * ny + j;
  const cplx ex = ldg(t.ex + g), ey = ldg(t.ey + g), hx = ldg(t.hx + g), hy = ldg(t.hy + g);
  const cplx u00 = t.U(i, j), u10 = t.U(i + 1, j), u01 = t.U(i, j + 1);
  const cplx t00 = t.Tt(i, j), tm0 = t.Tt(i - 1, j), t0m = t.Tt(i, j - 1);
  const cplx kk = t.K(i, j), gg = t.G(i, j);
  cplx r1 = t.CX(0, i) * u00 + t.CX(1, i) * u10 + t.F(12, i, j) * gg + t.F(16, i, j) * hx + t.F(17, i, j) * hy;
  cplx r2 = t.CY(0, j) * u00 + t.CY(1, j) * u01 - t.F(13, i, j) * gg - t.F(14, i, j) * hx - t.F(15, i, j) * hy;
  cplx r3 = t.CX(2, i) * t00 + t.CX(3, i) * tm0 + t.F(3, i, j) * kk + t.F(7, i, j) * ex + t.F(8, i, j) * ey;
  cplx r4 = t.CY(2, j) * t00 + t.CY(3, j) * t0m - t.F(4, i, j) * kk - t.F(5, i, j) * ex - t.F(6, i, j) * ey;
  const cplx mi = mk(0.0, -a.msign);  // msign * (-i)
  const cplx sg = ldg(a.sigma + b);
  cplx o1 = mi * r1 - sg * ex, o2 = mi * r2 - sg * ey, o3 = mi * r3 - sg * hx, o4 = mi * r4 - sg * hy;
  cplx *yb = a.y + (size_t)b * 4 * N;
  if (a.rhs) {
    const cplx *rb = a.rhs + (size_t)b * 4 * N;
    o1 = ldg(rb + g) - o1; o2 = ldg(rb + N + g) - o2; o3 = ldg(rb + 2 * N + g) - o3; o4 = ldg(rb + 3 * N + g) - o4;
  }
  yb[g] = o1; yb[N + g] = o2; yb[2 * N + g] = o3; yb[3 * N + g] = o4;
}

// Diagonal-part blocks of the first-order operator, M_d = [[0, P], [Q, 0]] (solver.py:479-489):
//   which = 0:  out = P h,  P h = [Dxf u + myy hy ; Dyf u - mxx hx],  u = (Dxb hy - Dyb hx) / ezz
//   which = 1:  out = Q e,  Q e = [Dxb t + eyy ey ; Dyb t - exx ex],  t = (Dxf ey - Dyf ex) / mzz
// in/out are two-component fields with arbitrary batch strides (they are halves of 4N Krylov vectors).
template <typename C>
__global__ void __launch_bounds__(256) pq_kernel(int which, int nx, int ny, const cplx *in, size_t in_bstride, cplx *out,
                                                 size_t out_bstride, const C *fields, size_t f_bstride, const cplx *cxs,
                                                 const cplx *cys) {
  const size_t N = (size_t)nx * ny;
  const int j = blockIdx.x * 64 + threadIdx.x, i = blockIdx.y * 4 + threadIdx.y, b = blockIdx.z;
  if (i >= nx || j >= ny) return;
  const cplx *a1 = in + in_bstride * b, *a2 = a1 + N;
  const C *fb = fields + f_bstride * b;
  const C *exx = fb, *eyy = fb + N, *iez = fb + 2 * N, *mxx = fb + 3 * N, *myy = fb + 4 * N, *imz = fb + 5 * N;
  const cplx *cx = cxs + (size_t)b * 4 * nx, *cy = cys + (size_t)b * 4 * ny;
  const cplx z = mk(0.0, 0.0);
  auto ld = [&](const cplx *p, int ii, int jj) { return (ii >= 0 && ii < nx && jj >= 0 && jj < ny) ? ldg(p + (size_t)ii * ny + jj) : z; };
  auto CX = [&](int w, int ii) { return (ii >= 0 && ii < nx) ? ldg(cx + (size_t)w * nx + ii) : z; };
  auto CY = [&](int w, int jj) { return (jj >= 0 && jj < ny) ? ldg(cy + (size_t)w * ny + jj) : z; };
  const size_t g = (size_t)i * ny + j;
  cplx o1, o2;
  if (which == 0) {  // a1 = hx, a2 = hy
    auto U = [&](int ii, int jj) {
      if (ii < 0 || jj < 0 || ii >= nx || jj >= ny) return z;
      cplx kd = CX(2, ii) * ld(a2, ii, jj) + CX(3, ii) * ld(a2, ii - 1, jj) - CY(2, jj) * ld(a1, ii, jj) - CY(3, jj) * ld(a1, ii, jj - 1);
      return ldg(iez + (size_t)ii * ny + jj) * kd;
    };
    const cplx u00 = U(i, j);
    o1 = CX(0, i) * u00 + CX(1, i) * U(i + 1, j) + ldg(myy + g) * ldg(a2 + g);
    o2 = CY(0, j) * u00 + CY(1, j) * U(i, j + 1) - ldg(mxx + g) * ldg(a1 + g);
  } else {  // a1 = ex, a2 = ey
    auto T = [&](int ii, int jj) {
      if (ii < 0 || jj < 0 || ii >= nx || jj >= ny) return z;
      cplx gd = CX(0, ii) * ld(a2, ii, jj) + CX(1, ii) * ld(a2, ii + 1, jj) - CY(0, jj) * ld(a1, ii, jj) - CY(1, jj) * ld(a1, ii, jj + 1);
      return ldg(imz + (size_t)ii * ny + jj) * gd;
    };
    const cplx t00 = T(i, j);
    o1 = CX(2, i) * t00 + CX(3, i) * T(i - 1, j) + ldg(eyy + g) * ldg(a2 + g);
    o2 = CY(2, j) * t00 + CY(3, j) * T(i, j - 1) - ldg(exx + g) * ldg(a1 + g);
  }
  cplx *ob = out + out_bstride * b;
  ob[g] = o1;
  ob[N + g] = o2;
}

// out[b][e] = ca[b] * x[b][e] + cb[b] * y[b][e]  (per-problem complex scalars, strided batches; y may be null)
__global__ void __launch_bounds__(256) lin2_kernel(size_t len, const cplx *ca, const cplx *x, size_t x_bstride, const cplx *cb,
                                                   const cplx *y, size_t y_bstride, cplx *out, size_t out_bstride) {
  const int b = blockIdx.y;
  const cplx a = ca[b], bb = cb ? cb[b] : mk(0.0, 0.0);
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < len; e += stride) {
    cplx v = a * ldg(x + x_bstride * b + e);
    if (y) v = v + bb * ldg(y + y_bstride * b + e);
    out[out_bstride * b + e] = v;
  }
}

// strided precision conversion: dst[b][e] = (D) src[b][e]
template <typename S, typename D>
__global__ void __launch_bounds__(256) convert_strided_kernel(size_t len, const S *src, size_t src_bstride, D *dst, size_t dst_bstride) {
  const int b = blockIdx.y;
  const size_t stride = (size_t)gridDim.x * 256;
  for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < len; e += stride) {
    D d;
    convert(src[src_bstride * b + e], d);
    dst[dst_bstride * b + e] = d;
  }
}

// six components of mode m at cell g into the reference layout [2][3][nx][ny][1][M], complex128 or complex64
__device__ __forceinline__ void store_fields(cplx *out, int single, size_t base, size_t N, size_t g, int M, int m, cplx Ex, cplx Ey,
                                             cplx Ez, cplx Hx, cplx Hy, cplx Hz) {
  const cplx v[6] = {Ex, Ey, Ez, Hx, Hy, Hz};
  if (single) {
    cplxf *o = reinterpret_cast<cplxf *>(out) + base;
#pragma unroll
    for (int c = 0; c < 6; ++c) o[((size_t)c * N + g) * M + m] = mkf((float)v[c].re, (float)v[c].im);
  } else {
    cplx *o = out + base;
#pragma unroll
    for (int c = 0; c < 6; ++c) o[((size_t)c * N + g) * M + m] = v[c];
  }
}

// tensorial epilogue (solver.py:701-719, 254-269): six components from w = [Ex;Ey;Hx;Hy], Ez = U, Hz = Tt
template <typename C>
struct TensorEpilogueArgs {
  int nx, ny, num_modes;
  const cplx *vec;   // mode m of problem b at vec + m*vstride + b*4N
  size_t vstride;
  const C *ft;
  size_t ft_bstride;
  const cplx *cx, *cy;
  const double *jz_e, *jz_h;  // bend scale of the z components or null
  int jz_axis, jz_len;
  double jac_a, jac_b;        // angled transform J[0][2], J[1][2]
  int conj_flip;              // tensorial_real with direction "-": E = conj(E), H = -conj(H) (solver.py:378-380)
  double h_scale;
  cplx *out;
  int single;                 // write complex64 (precision = "single", solver.py:265-267)
};
template <typename C>
__global__ void __launch_bounds__(256) tensor_epilogue_kernel(TensorEpilogueArgs<C> a) {
  const int nx = a.nx, ny = a.ny, M = a.num_modes;
  const size_t N = (size_t)nx * ny;
  const int j = blockIdx.x * 64 + threadIdx.x, i = blockIdx.y * 4 + threadIdx.y;
  const int m = blockIdx.z % M, b = blockIdx.z / M;
  if (i >= nx || j >= ny) return;
  const cplx *wb = a.vec + (size_t)m * a.vstride + (size_t)b * 4 * N;
  TensorCell<C> t{wb, wb + N, wb + 2 * N, wb + 3 * N, a.ft + a.ft_bstride * b, a.cx + (size_t)b * 4 * nx, a.cy + (size_t)b * 4 * ny, nx, ny, N};
  const size_t g = (size_t)i * ny + j;
  const cplx hs = mk(0.0, -a.h_scale);
  cplx Ex = ldg(t.ex + g), Ey = ldg(t.ey + g), Ez = t.U(i, j);
  cplx Hx = hs * ldg(t.hx + g), Hy = hs * ldg(t.hy + g), Hz = hs * t.Tt(i, j);
  if (a.conj_flip) {
    Ex = cj(Ex); Ey = cj(Ey); Ez = cj(Ez);
    Hx = -cj(Hx); Hy = -cj(Hy); Hz = -cj(Hz);
  }
  double de = 1.0, dh = 1.0;
  if (a.jz_axis >= 0) {
    const int q = a.jz_axis == 0 ? i : j;
    de = a.jz_e[(size_t)b * a.jz_len + q];
    dh = a.jz_h[(size_t)b * a.jz_len + q];
  }
  // E = J^T E' with J = [[1,0,a],[0,1,b],[0,0,d]]
  Ez = a.jac_a * Ex + a.jac_b * Ey + de * Ez;
  Hz = a.jac_a * Hx + a.jac_b * Hy + dh * Hz;
  store_fields(a.out, a.single, (size_t)b * 6 * N * M, N, g, M, m, Ex, Ey, Ez, Hx, Hy, Hz);
}

// ------------------------------------------------------------------------------------------------
// epilogue: eigenvector -> six field components in the reference layout (solver.py:556-589,254-269)
// ------------------------------------------------------------------------------------------------
template <typename T, typename C>
struct EpilogueArgs {
  int nx, ny, num_modes;
  const T *vec;      // [M][B][2][N] eigenvectors (mode-major like a Krylov basis): vec + m*vstride + b*2N
  size_t vstride;
  const C *fields;   // exx, eyy, iez, (mxx, myy, imz)
  size_t field_bstride;
  const T *cx, *cy;  // [B][4][n]
  const cplx *ncomplex;  // [B][M]  n_eff + i k_eff in solver (transformed) coordinates
  const double *jz_e, *jz_h;  // [B][n_jz] or null: bend back-transform of the z components
  int jz_axis, jz_len;
  int direction;
  double h_scale;    // 1 / ETA_0
  cplx *out;         // [B][2][3][nx][ny][M]
  int single;        // write complex64 (precision = "single", solver.py:265-267)
};

// E = (Ex, Ey, u / (i n)),  H = (-i/eta0) * (q1/(i n), q2/(i n), t)
// with q1 = Dxb t + eyy v2, q2 = Dyb t - exx v1 (Q v, solver.py:483-489,578-582); the Ez identity
// iez (Dxb Hy - Dyb Hx) = u/(i n) follows from Dxb Dyb = Dyb Dxb.
template <typename T, typename C, bool HAS_MU>
__global__ void __launch_bounds__(256) epilogue_kernel(EpilogueArgs<T, C> a) {
  const int nx = a.nx, ny = a.ny, M = a.num_modes;
  const size_t N = (size_t)nx * ny;
  const int j = blockIdx.x * 64 + threadIdx.x, i = blockIdx.y * 4 + threadIdx.y;
  const int m = blockIdx.z % M, b = blockIdx.z / M;
  if (i >= nx || j >= ny) return;
  const T *v1 = a.vec + (size_t)m * a.vstride + (size_t)b * 2 * N, *v2 = v1 + N;
  const C *fb = a.fields + a.field_bstride * b;
  const C *exx = fb, *eyy = fb + N, *iez = fb + 2 * N, *imz = fb + 5 * N;
  const T *cx = a.cx + (size_t)b * 4 * nx, *cy = a.cy + (size_t)b * 4 * ny;
  const T z = zero_of<T>();
  auto V1 = [&](int ii, int jj) { return (ii >= 0 && ii < nx && jj >= 0 && jj < ny) ? ldg(v1 + (size_t)ii * ny + jj) : z; };
  auto V2 = [&](int ii, int jj) { return (ii >= 0 && ii < nx && jj >= 0 && jj < ny) ? ldg(v2 + (size_t)ii * ny + jj) : z; };
  auto CX = [&](int w, int ii) { return (ii >= 0 && ii < nx) ? ldg(cx + (size_t)w * nx + ii) : z; };
  auto CY = [&](int w, int jj) { return (jj >= 0 && jj < ny) ? ldg(cy + (size_t)w * ny + jj) : z; };
  auto TT = [&](int ii, int jj) {
    if (ii < 0 || jj < 0 || ii >= nx || jj >= ny) return z;
    T acc = CX(0, ii) * V2(ii, jj) + CX(1, ii) * V2(ii + 1, jj) - CY(0, jj) * V1(ii, jj) - CY(1, jj) * V1(ii, jj + 1);
    if (HAS_MU) acc = ldg(imz + (size_t)ii * ny + jj) * acc;
    return acc;
  };
  const size_t g = (size_t)i * ny + j;
  const T e1 = V1(i, j), e2 = V2(i, j);
  const C ex = ldg(exx + g), ey = ldg(eyy + g);
  const T t00 = TT(i, j), tm0 = TT(i - 1, j), t0m = TT(i, j - 1);
  const T q1 = CX(2, i) * t00 + CX(3, i) * tm0 + ey * e2;
  const T q2 = CY(2, j) * t00 + CY(3, j) * t0m - ex * e1;
  T uacc = CX(2, i) * (ex * e1) + CY(2, j) * (ey * e2);
  if (i > 0) uacc += CX(3, i) * (ldg(exx + g - ny) * V1(i - 1, j));
  if (j > 0) uacc += CY(3, j) * (ldg(eyy + g - 1) * V2(i, j - 1));
  const T u = -(ldg(iez + g) * uacc);
  const cplx nc = a.ncomplex[(size_t)b * M + m];
  const cplx inv_in = recip(mk(-nc.im, nc.re));  // 1 / (i n)
  const cplx hs = mk(0.0, -a.h_scale);           // -i / eta0
  cplx Ex = to_cplx(e1), Ey = to_cplx(e2), Ez = to_cplx(u) * inv_in;
  cplx Hx = hs * (to_cplx(q1) * inv_in), Hy = hs * (to_cplx(q2) * inv_in), Hz = hs * to_cplx(t00);
  if (a.direction < 0) {  // solver.py:370-373
    Hx = -Hx; Hy = -Hy; Ez = -Ez;
  }
  if (a.jz_axis >= 0) {   // E = J^T E' with J = diag(1, 1, dwdz) (solver.py:254-259)
    const int t = a.jz_axis == 0 ? i : j;
    Ez = a.jz_e[(size_t)b * a.jz_len + t] * Ez;
    Hz = a.jz_h[(size_t)b * a.jz_len + t] * Hz;
  }
  store_fields(a.out, a.single, (size_t)b * 6 * N * M, N, g, M, m, Ex, Ey, Ez, Hx, Hy, Hz);
}

}  // namespace b200ms
