// Adjoint sensitivities of n_complex to the diagonal permittivity (DESIGN.md section 10).
//
// For the diagonal operator A = P Q of reciprocal media the left eigenvector follows from the right one v, so the derivative of
// an eigenvalue with respect to every eps entry is one pass over v (no second solve).  With h = Q v = (q1, q2), the Ez-site
// quantity u = iez (Dxb q2 - Dyb q1) (= E_z times i n, the `u` of epilogue_kernel) and the complex-stretched Yee areas
//   a_x = lf_x[i] lb_y[j]  (Ex site),   a_y = lb_x[i] lf_y[j]  (Ey site),   a_z = lb_x[i] lb_y[j]  (Ez site),
// where lb[0] is halved on an axis with a PMC wall (the 2 / lb[0] row of Db), the unconjugated discrete flux
//   S = sum_cells (a_x v1 q2 - a_y v2 q1)
// gives, with lambda = -n^2,
//   dn/deps_xx = -n a_x v1^2 / (2 S),   dn/deps_yy = -n a_y v2^2 / (2 S),   dn/deps_zz = -a_z u^2 / (2 n S).
// Scope: diagonal, non-bent, identity-mu problems without PEC-valued cells (the host rejects the rest before the solve).
//
// Two passes over the Ritz vectors, both deterministic: sens_scan_kernel writes per-chunk partial sums of S (no atomics),
// sens_write_kernel sums the partials in a fixed order and writes the three derivatives of every cell.  The per-cell arithmetic
// is in the HD functions below, shared with the host hook b200ms_debug_sensitivity (tests/test_sensitivity_cpu.py).
#pragma once
#include "kernels.cuh"

namespace b200ms {

constexpr int kSensChunks = 64;

// one mode of one problem: in-plane E (v1, v2), fp64 coefficient fields exx, eyy, iez (= 1 / eps_zz) and, if present, imz,
// and the level-0 1-D coefficients [4][n] (f0, f1, b0, bm) of both axes
template <typename T, typename C>
struct SensCell {
  int nx, ny;
  const T *v1, *v2;
  const C *exx, *eyy, *iez, *imz;  // imz: nullptr for mu = 1
  const T *cx, *cy;
};

// e1 = Ex, e2 = Ey, (q1, q2) = Q v and u = iez (Dxb q2 - Dyb q1) at cell (i, j), the radius-1 part of the operator
// (same arithmetic as epilogue_kernel, whose u uses Dxb Dyb = Dyb Dxb)
template <typename T, typename C>
HD void sens_cell(const SensCell<T, C> &a, int i, int j, cplx &e1, cplx &e2, cplx &q1, cplx &q2, cplx &u) {
  const int nx = a.nx, ny = a.ny;
  const T z = zero_of<T>();
  auto V1 = [&](int ii, int jj) { return (ii >= 0 && ii < nx && jj >= 0 && jj < ny) ? a.v1[(size_t)ii * ny + jj] : z; };
  auto V2 = [&](int ii, int jj) { return (ii >= 0 && ii < nx && jj >= 0 && jj < ny) ? a.v2[(size_t)ii * ny + jj] : z; };
  auto CX = [&](int w, int ii) { return (ii >= 0 && ii < nx) ? a.cx[(size_t)w * nx + ii] : z; };
  auto CY = [&](int w, int jj) { return (jj >= 0 && jj < ny) ? a.cy[(size_t)w * ny + jj] : z; };
  auto TT = [&](int ii, int jj) {
    if (ii < 0 || jj < 0 || ii >= nx || jj >= ny) return z;
    T acc = CX(0, ii) * V2(ii, jj) + CX(1, ii) * V2(ii + 1, jj) - CY(0, jj) * V1(ii, jj) - CY(1, jj) * V1(ii, jj + 1);
    if (a.imz) acc = a.imz[(size_t)ii * ny + jj] * acc;
    return acc;
  };
  const size_t g = (size_t)i * ny + j;
  const T v1 = V1(i, j), v2 = V2(i, j);
  const C ex = a.exx[g], ey = a.eyy[g];
  const T t00 = TT(i, j), tm0 = TT(i - 1, j), t0m = TT(i, j - 1);
  T uacc = CX(2, i) * (ex * v1) + CY(2, j) * (ey * v2);
  if (i > 0) uacc += CX(3, i) * (a.exx[g - ny] * V1(i - 1, j));
  if (j > 0) uacc += CY(3, j) * (a.eyy[g - 1] * V2(i, j - 1));
  e1 = to_cplx(v1);
  e2 = to_cplx(v2);
  q1 = to_cplx(CX(2, i) * t00 + CX(3, i) * tm0 + ey * v2);
  q2 = to_cplx(CY(2, j) * t00 + CY(3, j) * t0m - ex * v1);
  u = to_cplx(-(a.iez[g] * uacc));
}

// Yee areas of the three E sites of cell (i, j) from the per-axis lengths {lf[n], lb[n]} (lb[0] already halved at a PMC wall)
HD void sens_areas(const cplx *lx, const cplx *ly, int nx, int ny, int i, int j, cplx &ax, cplx &ay, cplx &az) {
  ax = lx[i] * ly[ny + j];
  ay = lx[nx + i] * ly[j];
  az = lx[nx + i] * ly[ny + j];
}

// the cell's term of S
HD cplx sens_flux_term(cplx ax, cplx ay, cplx e1, cplx e2, cplx q1, cplx q2) { return ax * (e1 * q2) - ay * (e2 * q1); }

// dn/deps_{xx,yy,zz} of the cell; inv2s = 1 / (2 S)
HD void sens_grad(cplx n, cplx inv2s, cplx ax, cplx ay, cplx az, cplx e1, cplx e2, cplx u, cplx g[3]) {
  g[0] = -((n * inv2s) * (ax * (e1 * e1)));
  g[1] = -((n * inv2s) * (ay * (e2 * e2)));
  g[2] = -((recip(n) * inv2s) * (az * (u * u)));
}

template <typename T, typename C>
struct SensArgs {
  int nx, ny, num_modes;
  const T *vec;          // [M][B][2][N] Ritz vectors in mode order (vec + m*vstride + b*2N)
  size_t vstride;
  const C *fields;       // exx, eyy, iez, (mxx, myy, imz) of problem b at fields + b * field_bstride
  size_t field_bstride;
  int has_mu;
  const T *cx, *cy;      // [B][4][n]
  const cplx *len_x, *len_y;  // [B][2][n]: lf, lb (lb[0] halved at a PMC wall)
  const cplx *ncomplex;  // [B][M]
  cplx *const *out;      // [B]: [M][3][nx][ny] complex128, or nullptr (no gradient asked for this problem)
};

template <typename T, typename C>
__device__ __forceinline__ SensCell<T, C> sens_view(const SensArgs<T, C> &a, int b, int m) {
  const size_t N = (size_t)a.nx * a.ny;
  const C *fb = a.fields + a.field_bstride * b;
  SensCell<T, C> c;
  c.nx = a.nx; c.ny = a.ny;
  c.v1 = a.vec + (size_t)m * a.vstride + (size_t)b * 2 * N;
  c.v2 = c.v1 + N;
  c.exx = fb; c.eyy = fb + N; c.iez = fb + 2 * N; c.imz = a.has_mu ? fb + 5 * N : nullptr;
  c.cx = a.cx + (size_t)b * 4 * a.nx; c.cy = a.cy + (size_t)b * 4 * a.ny;
  return c;
}

// partial[(b * M + m) * kSensChunks + chunk] = this chunk's part of S; grid (kSensChunks, B * M)
template <typename T, typename C>
__global__ void __launch_bounds__(256) sens_scan_kernel(SensArgs<T, C> a, cplx *partial) {
  const int M = a.num_modes, b = blockIdx.y / M, m = blockIdx.y % M;
  if (!a.out[b]) return;
  const SensCell<T, C> c = sens_view(a, b, m);
  const cplx *lx = a.len_x + (size_t)b * 2 * a.nx, *ly = a.len_y + (size_t)b * 2 * a.ny;
  const size_t N = (size_t)a.nx * a.ny;
  cplx acc = mk(0.0, 0.0);
  for (size_t t = (size_t)blockIdx.x * 256 + threadIdx.x; t < N; t += (size_t)gridDim.x * 256) {
    const int i = (int)(t / a.ny), j = (int)(t % a.ny);
    cplx e1, e2, q1, q2, u, ax, ay, az;
    sens_cell(c, i, j, e1, e2, q1, q2, u);
    sens_areas(lx, ly, a.nx, a.ny, i, j, ax, ay, az);
    acc += sens_flux_term(ax, ay, e1, e2, q1, q2);
  }
  acc = warp_sum(acc);
  __shared__ cplx red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    cplx s = red[0];
    for (int w = 1; w < 8; ++w) s += red[w];
    partial[(size_t)blockIdx.y * kSensChunks + blockIdx.x] = s;
  }
}

// out[b][m][3][nx][ny]; grid (cell blocks, B * M)
template <typename T, typename C>
__global__ void __launch_bounds__(256) sens_write_kernel(SensArgs<T, C> a, const cplx *partial) {
  const int M = a.num_modes, b = blockIdx.y / M, m = blockIdx.y % M;
  cplx *out = a.out[b];
  if (!out) return;
  __shared__ cplx sh[2];
  if (threadIdx.x == 0) {
    cplx s = mk(0.0, 0.0);
    for (int q = 0; q < kSensChunks; ++q) s += partial[(size_t)blockIdx.y * kSensChunks + q];
    sh[0] = recip(2.0 * s);
    sh[1] = a.ncomplex[(size_t)b * M + m];
  }
  __syncthreads();
  const cplx inv2s = sh[0], n = sh[1];
  const SensCell<T, C> c = sens_view(a, b, m);
  const cplx *lx = a.len_x + (size_t)b * 2 * a.nx, *ly = a.len_y + (size_t)b * 2 * a.ny;
  const size_t N = (size_t)a.nx * a.ny;
  out += (size_t)m * 3 * N;
  for (size_t t = (size_t)blockIdx.x * 256 + threadIdx.x; t < N; t += (size_t)gridDim.x * 256) {
    const int i = (int)(t / a.ny), j = (int)(t % a.ny);
    cplx e1, e2, q1, q2, u, ax, ay, az, g[3];
    sens_cell(c, i, j, e1, e2, q1, q2, u);
    sens_areas(lx, ly, a.nx, a.ny, i, j, ax, ay, az);
    sens_grad(n, inv2s, ax, ay, az, e1, e2, u, g);
    out[t] = g[0];
    out[N + t] = g[1];
    out[2 * N + t] = g[2];
  }
}

}  // namespace b200ms
