// Batched device eigen-solver: multigrid-preconditioned FGMRES shift-invert inside a Krylov-Schur
// (thick-restart Arnoldi) iteration.  Replaces scipy.sparse.linalg.eigs(mat, k, sigma, tol, v0)
// (ARPACK + SuperLU) at tidy3d/plugins/mode/solver.py:744-746 for a batch of same-shaped problems.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "dense.hpp"
#include "host_setup.hpp"
#include "kernels.cuh"
#include "krylov_kernels.cuh"
#include "coarse_kernel.cuh"
#include "march2.cuh"
#include "march2_tma.cuh"
#include "sensitivity.cuh"

namespace b200ms {

#define CUDA_CHECK(expr)                                                                              \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess)                                                                            \
      throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " + __FILE__ + ":" + \
                               std::to_string(__LINE__));                                             \
  } while (0)

// the solver arena of a device batch does not fit: the caller retries with fewer problems per batch (api.cu)
struct DeviceOutOfMemory : std::runtime_error {
  size_t bytes;
  explicit DeviceOutOfMemory(size_t n) : std::runtime_error("CUDA error: out of memory reserving " + std::to_string(n) + " bytes for the solver arena"), bytes(n) {}
};

// ---- simple device arena ---------------------------------------------------------------------------
struct Arena {
  unsigned char *base = nullptr;
  size_t cap = 0, used = 0;
  void reserve(size_t bytes) {
    if (bytes <= cap) {
      used = 0;
      return;
    }
    if (base) cudaFree(base);
    base = nullptr;
    cap = 0;
    const cudaError_t e = cudaMalloc(&base, bytes);
    if (e == cudaErrorMemoryAllocation) {
      cudaGetLastError();  // clear the sticky-free allocation error: the context is intact
      base = nullptr;
      throw DeviceOutOfMemory(bytes);
    }
    CUDA_CHECK(e);
    cap = bytes;
    used = 0;
  }
  template <typename U>
  U *get(size_t count) {
    size_t bytes = (count * sizeof(U) + 255) & ~size_t(255);
    if (used + bytes > cap) throw std::runtime_error("device arena exhausted");
    U *p = reinterpret_cast<U *>(base + used);
    used += bytes;
    return p;
  }
  void release() {
    if (base) cudaFree(base);
    base = nullptr;
    cap = used = 0;
  }
};
struct ArenaSizer {
  size_t total = 0;
  template <typename U>
  void add(size_t count) { total += (count * sizeof(U) + 255) & ~size_t(255); }
};

struct SolveStats {
  int op_applies = 0, inner_iters = 0, restarts = 0;
  long stencil_applies = 0, launches = 0;
  int inner_failures = 0;  // shift-invert solves that stopped above 1e4 x inner_tol
  long host_syncs = 0;     // stream synchronisations inside the inner solves
  int inner_cycles = 0;    // FGMRES cycles (iterative-refinement steps)
  int outer_second_pass = 0;  // Krylov-Schur orthogonalisations that needed the second Gram-Schmidt pass (DGKS test)
};

template <typename T> inline cd to_cd(T v);
template <> inline cd to_cd<double>(double v) { return cd(v, 0.0); }
template <> inline cd to_cd<cplx>(cplx v) { return cd(v.re, v.im); }
template <typename T> inline T from_cd(cd v);
template <> inline double from_cd<double>(cd v) { return v.real(); }
template <> inline cplx from_cd<cplx>(cd v) { return mk(v.real(), v.imag()); }
template <> inline float from_cd<float>(cd v) { return (float)v.real(); }
template <> inline cplxf from_cd<cplxf>(cd v) { return mkf((float)v.real(), (float)v.imag()); }
template <> inline cd to_cd<float>(float v) { return cd(v, 0.0); }
template <> inline cd to_cd<cplxf>(cplxf v) { return cd(v.re, v.im); }

// ------------------------------------------------------------------------------------------------------
// T / C: Krylov vector and coefficient-field types (fp64).  P / PC: their fp32 twins, the types of the multigrid
// preconditioner (mixed precision: the V-cycle moves half the bytes).
template <typename T, typename C, typename P, typename PC>
class BatchSolver {
 public:
  struct Level {
    int nx = 0, ny = 0;
    size_t N = 0;
    PC *fields = nullptr;
    C *fields_true = nullptr;  // level 0 only: fp64 fields of the reference operator
    size_t fbstride = 0;
    P *cx = nullptr, *cy = nullptr;          // multigrid (phase-limited PML) coefficients
    T *cx_true = nullptr, *cy_true = nullptr;  // level 0 only: the reference operator
    P *x = nullptr, *b = nullptr, *r = nullptr, *tmp = nullptr;
    P *dinv = nullptr;  // omega / diag(A_l - sigma), [B][2][N]
    TransferArgs tr;  // to the next coarser level
  };

  BatchSolver(Arena &arena, cudaStream_t stream, const b200ms_options &opt) : arena_(arena), st_(stream), opt_(opt) {}

  int B = 0, nx = 0, ny = 0, k = 0, m = 0, restart = 0, nf = 3;
  size_t N = 0, len = 0, vstride = 0, lenE = 0, vsE = 0;
  bool tensor_ = false;
  bool masked_ = false;      // incidence-matrix formulation: unknowns marked by exx == 0 / eyy == 0 are held at zero
  bool single_out_ = false;  // fields are delivered as complex64 (mode_spec.precision == "single")
  double msign_ = 1.0;
  bool has_mu = false, shared_fields = false;
  std::vector<Level> lv;
  SolveStats stats;
  std::vector<int> level_shapes;

  // -- build ---------------------------------------------------------------------------------------
  // d_refs: device array of the raw media of the problems (B entries, or one when share_fields): the coefficient fields
  // are generated on the device from the raw eps/mu uploaded by the caller (csrc/medium.cuh)
  void build(const std::vector<const ProblemSetup *> &ps, bool share_fields, const MediumRef *d_refs) {
    B = (int)ps.size();
    const ProblemSetup &p0 = *ps[0];
    nx = p0.nx;
    ny = p0.ny;
    N = (size_t)nx * ny;
    tensor_ = p0.tensorial;
    lenE = 2 * N;
    vsE = (size_t)B * lenE;
    len = (tensor_ ? 4 : 2) * N;  // Krylov vectors: [Ex;Ey] or, tensorial, [Ex;Ey;Hx;Hy]
    vstride = (size_t)B * len;
    msign_ = (tensor_ && p0.eps_complex && p0.direction < 0) ? -1.0 : 1.0;  // solver.py:669-670
    k = p0.num_modes;
    has_mu = p0.has_mu;
    masked_ = p0.masked;
    nf = has_mu ? 6 : 3;
    shared_fields = share_fields;
    const int ncv = opt_.ncv > 0 ? opt_.ncv : std::max(2 * k + 1, 20);
    m = std::min(ncv, (int)std::min<size_t>(len - 1, 1 << 20));
    if (m < k + 2) m = std::min<int>(k + 2, (int)len);
    restart = std::max(2, opt_.gmres_restart);
    restart = std::min(restart, kGsMaxCoef - 4);
    mask_x_ = (!p0.ax[0].pmc && nx > 1) ? 1 : 0;
    mask_y_ = (!p0.ax[1].pmc && ny > 1) ? 1 : 0;

    // hierarchy geometry from problem 0; indefinite shifts limit the coarsest spacing
    double kh_limit = 0.0, kmax = 0.0;
    double max_k2 = 0.0;
    for (auto *p : ps) max_k2 = std::max(max_k2, p->max_k2);
    if (max_k2 > 1e-6 && opt_.mg_ppw > 0) {
      kmax = std::sqrt(max_k2);
      kh_limit = 2.0 * M_PI / opt_.mg_ppw;
    }
    std::vector<std::vector<Axis>> axes0;
    plan_hierarchy(p0.ax, opt_.mg_min_size, 12, kh_limit, kmax, plan_, &axes0);
    const int L = (int)plan_.nx.size();
    level_shapes.clear();
    for (int l = 0; l < L; ++l) {
      level_shapes.push_back(plan_.nx[l]);
      level_shapes.push_back(plan_.ny[l]);
    }

    // ---- size the arena ----
    ArenaSizer sz;
    const size_t fB = shared_fields ? 1 : B;
    for (int l = 0; l < L; ++l) {
      size_t Nl = (size_t)plan_.nx[l] * plan_.ny[l];
      sz.add<C>(fB * nf * Nl * (l == 0 ? 2 : 1));
      sz.add<T>((size_t)B * 4 * plan_.nx[l] * (l == 0 ? 2 : 1));
      sz.add<T>((size_t)B * 4 * plan_.ny[l] * (l == 0 ? 2 : 1));
      for (int q = 0; q < 5; ++q) sz.add<T>((size_t)B * 2 * Nl);
      if (l + 1 < L) {
        size_t ints = 0, dbls = 0;
        transfer_sizes(plan_.trx[l], ints, dbls);
        transfer_sizes(plan_.try_[l], ints, dbls);
        sz.add<int>(ints + 64);
        sz.add<double>(dbls + 64);
      }
    }
    sz.add<T>((size_t)(m + 1) * vstride);        // outer basis
    sz.add<T>((size_t)(restart + 1) * vstride);  // FGMRES V
    sz.add<T>((size_t)restart * vstride);        // FGMRES Z
    sz.add<T>(vstride * 4);                      // xsol, rhs scratch, preconditioner scratch
    sz.add<T>((size_t)k * vstride);              // Ritz vectors
    sz.add<T>((size_t)B * kDotChunks * pstride());
    sz.add<T>((size_t)B * hstride());
    sz.add<T>((size_t)B * (m + 1) * (m + 1));
    sz.add<T>((size_t)B * 8);
    sz.add<P>((size_t)B * 4 * nx);
    sz.add<P>((size_t)B * 4 * ny);
    sz.add<T>((size_t)B * restart * (restart + 4));
    sz.add<T>((size_t)B * restart);
    sz.add<T>((size_t)3 * B * kDotChunks * pstride());
    sz.add<cplx>((size_t)B * ((size_t)(restart + 1) * restart + 3 * restart + 2));
    sz.add<double>((size_t)4 * B + 64);
    sz.add<int>((size_t)B + 64);
    sz.add<unsigned char>((size_t)B + 64);
    sz.add<cplx>((size_t)B * k);
    sz.add<double>((size_t)B * 2 * std::max(nx, ny) + 64);
    if (tensor_) {
      sz.add<C>(fB * 18 * N);
      sz.add<T>(vsE * 6);
      sz.add<cplx>((size_t)B * 8);
    }
    coarse_krylov_ = kh_limit > 0.0;
    kc_ = std::max(2, std::min(opt_.mg_coarse_iters, std::max(m, restart) - 1));
    {
      const size_t NL = (size_t)plan_.nx[L - 1] * plan_.ny[L - 1];
      if (coarse_krylov_) {
        sz.add<T>((size_t)(kc_ + 1) * B * 2 * NL);
        sz.add<T>((size_t)kc_ * B * 2 * NL);
        sz.add<T>((size_t)B * kc_ * (kc_ + 4));
        sz.add<T>((size_t)B * (kc_ + 1));
        sz.add<T>((size_t)B * kc_);
        sz.add<T>((size_t)B + 8);
        sz.add<T>(8);
      }
    }
    // permittivity gradient (sensitivity()): S partials, per-axis lengths, output pointers
    sz.add<cplx>((size_t)B * k * kSensChunks);
    sz.add<cplx>((size_t)B * 2 * (nx + ny));
    sz.add<cplx *>((size_t)B);
    arena_.reserve(sz.total + (1 << 20));

    // ---- allocate + upload ----
    lv.assign(L, Level());
    std::vector<std::vector<Axis>> axes_b(B);  // per problem, per level axes (2 per level flattened)
    for (int l = 0; l < L; ++l) {
      Level &v = lv[l];
      v.nx = plan_.nx[l];
      v.ny = plan_.ny[l];
      v.N = (size_t)v.nx * v.ny;
      v.fbstride = shared_fields ? 0 : nf * v.N;
      v.fields = arena_.get<PC>(fB * nf * v.N);
      if (l == 0) v.fields_true = arena_.get<C>(fB * nf * v.N);
      v.cx = arena_.get<P>((size_t)B * 4 * v.nx);
      v.cy = arena_.get<P>((size_t)B * 4 * v.ny);
      if (l == 0) {
        v.cx_true = arena_.get<T>((size_t)B * 4 * v.nx);
        v.cy_true = arena_.get<T>((size_t)B * 4 * v.ny);
      }
      v.x = arena_.get<P>((size_t)B * 2 * v.N);
      v.b = arena_.get<P>((size_t)B * 2 * v.N);
      v.r = arena_.get<P>((size_t)B * 2 * v.N);
      v.tmp = arena_.get<P>((size_t)B * 2 * v.N);
      v.dinv = arena_.get<P>((size_t)B * 2 * v.N);
    }
    // 1-D coefficients for every problem and level
    for (int l = 0; l < L; ++l) {
      std::vector<P> hx((size_t)B * 4 * lv[l].nx), hy((size_t)B * 4 * lv[l].ny);
      std::vector<T> hxt, hyt;
      if (l == 0) {
        hxt.resize(hx.size());
        hyt.resize(hy.size());
      }
      for (int b = 0; b < B; ++b) {
        if (l == 0) {
          axes_b[b] = {ps[b]->ax[0], ps[b]->ax[1]};
          // reference operator coefficients
          std::vector<cd> ct;
          ps[b]->ax[0].coefficients(ct);
          for (size_t i = 0; i < ct.size(); ++i) hxt[(size_t)b * 4 * lv[0].nx + i] = from_cd<T>(ct[i]);
          ps[b]->ax[1].coefficients(ct);
          for (size_t i = 0; i < ct.size(); ++i) hyt[(size_t)b * 4 * lv[0].ny + i] = from_cd<T>(ct[i]);
          // multigrid operator: same |stretch|, phase clamped so that Re(1/s^2) >= 0 (point smoothers are unstable on
          // the strongly rotated PML operator; the outer FGMRES on the true operator absorbs the difference)
          if (opt_.mg_pml_phase > 0)
            for (int a = 0; a < 2; ++a)
              for (std::vector<cd> *vec : {&axes_b[b][a].lf, &axes_b[b][a].lb})
                for (cd &z : *vec) {
                  double ph = std::arg(z);
                  if (std::abs(ph) > opt_.mg_pml_phase) z = std::polar(std::abs(z), ph > 0 ? opt_.mg_pml_phase : -opt_.mg_pml_phase);
                }
        } else {
          Axis cxa, cya;
          coarsen_axis(axes_b[b][0], plan_.trx[l - 1].start, cxa);
          coarsen_axis(axes_b[b][1], plan_.try_[l - 1].start, cya);
          axes_b[b] = {cxa, cya};
        }
        std::vector<cd> c;
        axes_b[b][0].coefficients(c);
        for (size_t i = 0; i < c.size(); ++i) hx[(size_t)b * 4 * lv[l].nx + i] = from_cd<P>(c[i]);
        axes_b[b][1].coefficients(c);
        for (size_t i = 0; i < c.size(); ++i) hy[(size_t)b * 4 * lv[l].ny + i] = from_cd<P>(c[i]);
      }
      CUDA_CHECK(cudaMemcpyAsync(lv[l].cx, hx.data(), hx.size() * sizeof(P), cudaMemcpyHostToDevice, st_));
      CUDA_CHECK(cudaMemcpyAsync(lv[l].cy, hy.data(), hy.size() * sizeof(P), cudaMemcpyHostToDevice, st_));
      if (l == 0) {
        CUDA_CHECK(cudaMemcpyAsync(lv[0].cx_true, hxt.data(), hxt.size() * sizeof(T), cudaMemcpyHostToDevice, st_));
        CUDA_CHECK(cudaMemcpyAsync(lv[0].cy_true, hyt.data(), hyt.size() * sizeof(T), cudaMemcpyHostToDevice, st_));
      }
      CUDA_CHECK(cudaStreamSynchronize(st_));
    }
    // fine-level coefficient fields: exx, eyy, 1/ezz, (mxx, myy, 1/mzz) from the raw media, in both precisions at once
    {
      dim3 grd((unsigned)std::min<size_t>((N + 255) / 256, 2048), (unsigned)fB);
      fields_kernel<C, PC><<<grd, 256, 0, st_>>>(d_refs, nf, lv[0].fields_true, lv[0].fields, (size_t)nf * N);
      stats.launches++;
      CUDA_CHECK(cudaGetLastError());
    }
    // transfer lists + coarse fields
    for (int l = 0; l + 1 < L; ++l) {
      TransferArgs &t = lv[l].tr;
      t.nxf = lv[l].nx;
      t.nyf = lv[l].ny;
      t.nxc = lv[l + 1].nx;
      t.nyc = lv[l + 1].ny;
      t.mask_x = mask_x_;
      t.mask_y = mask_y_;
      upload_transfer(plan_.trx[l].node, t.xn);
      upload_transfer(plan_.trx[l].edge, t.xe);
      upload_transfer(plan_.try_[l].node, t.yn);
      upload_transfer(plan_.try_[l].edge, t.ye);
      // site types: exx (e,n)  eyy (n,e)  ezz (n,n)  mxx (n,e)  myy (e,n)  mzz (e,e)
      const Transfer1DDev *fx[6] = {&t.xe, &t.xn, &t.xn, &t.xn, &t.xe, &t.xe};
      const Transfer1DDev *fy[6] = {&t.yn, &t.ye, &t.yn, &t.ye, &t.yn, &t.ye};
      dim3 blk(64, 4), grd((t.nyc + 63) / 64, (t.nxc + 3) / 4, (unsigned)fB);
      for (int q = 0; q < nf; ++q) {
        const bool inv = (q == 2 || q == 5);
        restrict_field_kernel<PC><<<grd, blk, 0, st_>>>(t.nxf, t.nyf, t.nxc, t.nyc, *fx[q], *fy[q],
                                                       lv[l].fields + (size_t)q * lv[l].N, shared_fields ? 0 : nf * lv[l].N,
                                                       lv[l + 1].fields + (size_t)q * lv[l + 1].N,
                                                       shared_fields ? 0 : nf * lv[l + 1].N, inv ? 1 : 0);
      }
      CUDA_CHECK(cudaGetLastError());
    }
    // Krylov storage
    Vout_ = arena_.get<T>((size_t)(m + 1) * vstride);
    Vg_ = arena_.get<T>((size_t)(restart + 1) * vstride);
    Zg_ = arena_.get<T>((size_t)restart * vstride);
    xsol_ = arena_.get<T>(vstride);
    rhs_ = arena_.get<T>(vstride);
    pre_a_ = arena_.get<P>(vstride);
    pre_b_ = arena_.get<P>(vstride);
    ritz_ = arena_.get<T>((size_t)k * vstride);
    partial_ = arena_.get<T>((size_t)B * kDotChunks * pstride());
    hbuf_ = arena_.get<T>((size_t)B * hstride());
    qbuf_ = arena_.get<T>((size_t)B * (m + 1) * (m + 1));
    sigma_ = arena_.get<T>((size_t)B * 4);
    sigma_p_ = arena_.get<P>((size_t)B * 4);
    cx_true_p_ = arena_.get<P>((size_t)B * 4 * nx);
    cy_true_p_ = arena_.get<P>((size_t)B * 4 * ny);
    {
      const size_t tx = (size_t)B * 4 * nx, ty = (size_t)B * 4 * ny;
      convert_kernel<T, P><<<(unsigned)std::min<size_t>((tx + 255) / 256, 1024), 256, 0, st_>>>(tx, lv[0].cx_true, cx_true_p_);
      convert_kernel<T, P><<<(unsigned)std::min<size_t>((ty + 255) / 256, 1024), 256, 0, st_>>>(ty, lv[0].cy_true, cy_true_p_);
    }
    Hd_ = arena_.get<T>((size_t)B * restart * (restart + 4));
    ydev_ = arena_.get<T>((size_t)B * restart);
    gpart_ = arena_.get<T>((size_t)3 * B * kDotChunks * pstride());
    lsq_work_ = arena_.get<cplx>((size_t)B * ((size_t)(restart + 1) * restart + 3 * restart + 2));
    tol_dev_ = arena_.get<double>((size_t)4 * B + 64);
    res_dev_ = tol_dev_ + B;
    n2_dev_ = tol_dev_ + 2 * B;
    bn2_dev_ = tol_dev_ + 3 * B;
    jused_dev_ = arena_.get<int>((size_t)B + 64);
    skip_dev_ = arena_.get<unsigned char>((size_t)B + 64);
    ncomplex_ = arena_.get<cplx>((size_t)B * k);
    jz_ = arena_.get<double>((size_t)B * 2 * std::max(nx, ny) + 64);
    if (tensor_) {
      ft_ = arena_.get<C>(fB * 18 * N);
      for (int q = 0; q < 6; ++q) tb_[q] = arena_.get<T>(vsE);
      tcoef_ = arena_.get<cplx>((size_t)B * 8);
      {
        dim3 grd((unsigned)std::min<size_t>((N + 255) / 256, 2048), (unsigned)fB);
        tensor_fields_kernel<C><<<grd, 256, 0, st_>>>(d_refs, ft_, (size_t)18 * N);
        stats.launches++;
        CUDA_CHECK(cudaGetLastError());
      }
      // per-problem scalars of the preconditioner: [0] -sigma_t, [1] i*msign, [2] 1/s, [3] -1/s, [4] 1  (s = -sigma_t^2)
      std::vector<cplx> hc((size_t)B * 8);
      for (int b = 0; b < B; ++b) {
        const cd st = ps[b]->sigma_t, sd = -st * st;
        const cd v[5] = {-st, cd(0, msign_), 1.0 / sd, -1.0 / sd, cd(1, 0)};
        for (int q = 0; q < 5; ++q) hc[(size_t)q * B + b] = mk(v[q].real(), v[q].imag());
      }
      CUDA_CHECK(cudaMemcpyAsync(tcoef_, hc.data(), hc.size() * sizeof(cplx), cudaMemcpyHostToDevice, st_));
      CUDA_CHECK(cudaStreamSynchronize(st_));
    }
    if (coarse_krylov_) {
      const size_t NL = lv[L - 1].N;
      cV_ = arena_.get<P>((size_t)(kc_ + 1) * B * 2 * NL);
      cZ_ = arena_.get<P>((size_t)kc_ * B * 2 * NL);
      cH_ = arena_.get<P>((size_t)B * kc_ * (kc_ + 4));
      cH2_ = arena_.get<P>((size_t)B * (kc_ + 1));
      cy_ = arena_.get<P>((size_t)B * kc_);
      cbeta_ = arena_.get<P>((size_t)B + 8);
      cone_ = arena_.get<P>(8);
      P one = from_real<P>(1.0);
      CUDA_CHECK(cudaMemcpyAsync(cone_, &one, sizeof(P), cudaMemcpyHostToDevice, st_));
      CUDA_CHECK(cudaStreamSynchronize(st_));
    }
    hhost_.resize((size_t)B * hstride());
    sig_host_.resize(B);
    sig_mg_host_.resize(B);
    for (int b = 0; b < B; ++b) {
      sig_mg_host_[b] = ps[b]->sigma;                                   // multigrid / diagonal operator: -(target^2)
      sig_host_[b] = tensor_ ? ps[b]->sigma_t : ps[b]->sigma;           // Krylov-side operator
    }
    set_sigma(sig_host_);
    set_sigma_mg(sig_mg_host_);
    // omega / diag(A_l - sigma) on every level: one recomputed-diagonal sweep applied to a vector of ones
    dinv_ready_ = false;
    for (int l = 0; l < L; ++l) {
      const size_t tot = (size_t)B * 2 * lv[l].N;
      fill_kernel<P><<<(unsigned)std::min<size_t>((tot + 255) / 256, 8192), 256, 0, st_>>>(tot, from_real<P>(1.0), lv[l].tmp);
      jacobi0(l, lv[l].tmp, lv[l].dinv);
    }
    dinv_ready_ = true;
    CUDA_CHECK(cudaStreamSynchronize(st_));
    CUDA_CHECK(cudaGetLastError());
    prime_march2();
    plan_fused_tail();
    capture_precondition_graph();
  }

  // shift of the Krylov-side (reference) operator
  void set_sigma(const std::vector<cd> &s) {
    std::vector<T> h(B);
    for (int b = 0; b < B; ++b) h[b] = from_cd<T>(s[b]);
    CUDA_CHECK(cudaMemcpyAsync(sigma_, h.data(), B * sizeof(T), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaStreamSynchronize(st_));
  }
  // shift of the multigrid operator (always the second-order diagonal-path operator A - sigma)
  void set_sigma_mg(const std::vector<cd> &s) {
    std::vector<P> hp(B);
    std::vector<T> ht(B);
    for (int b = 0; b < B; ++b) {
      hp[b] = from_cd<P>(s[b]);
      ht[b] = from_cd<T>(s[b]);
    }
    CUDA_CHECK(cudaMemcpyAsync(sigma_p_, hp.data(), B * sizeof(P), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaMemcpyAsync(sigma_ + B, ht.data(), B * sizeof(T), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaStreamSynchronize(st_));
  }

  // -- operator ------------------------------------------------------------------------------------
  template <typename TT, typename CC>
  void launch_stencil(const Level &v, int mode, const TT *x, const TT *rhs, TT *y, const CC *fields, const TT *cx, const TT *cy,
                      const TT *sigma, const TT *dinv = nullptr) {
    StencilArgs<TT, CC> a;
    a.nx = v.nx; a.ny = v.ny; a.x = x; a.rhs = rhs; a.y = y;
    a.fields = fields; a.field_bstride = v.fbstride; a.sigma = sigma; a.cx = cx; a.cy = cy;
    a.omega = opt_.mg_omega;
    a.dinv = dinv;
    stats.launches++;
    if (launch_march2<TT, CC>(v, mode, a, dinv != nullptr)) return;
    if (v.nx >= 32 && v.ny >= 2) {
      // rows marched per CTA: the march is a serial chain of (TXR + 3) row steps, each waiting on one global-load
      // round trip, so small levels (few CTAs per SM, nothing to hide that latency behind) get short chains
      bool rows32 = v.nx >= 384;
      if (rows32) {
        // wave quantisation: 7 CTAs of 128 threads per SM are resident; when 32-row CTAs leave the last wave mostly empty
        // (e.g. 32 problems of 512^2: 2.47 waves) 16-row CTAs fill it at the price of 9 % more halo rows
        const double per_wave = 148.0 * 7.0;
        const double c32 = (double)((v.ny + kMarchOut - 1) / kMarchOut) * ((v.nx + 31) / 32) * B / per_wave;
        const double c16 = (double)((v.ny + kMarchOut - 1) / kMarchOut) * ((v.nx + 15) / 16) * B / per_wave;
        const double t32 = std::ceil(c32) * 35.0, t16 = std::ceil(c16) * 19.0;  // waves x row steps per CTA
        if (t16 < 0.97 * t32) rows32 = false;
      }
      if (rows32) launch_march<TT, CC, 32>(v, mode, a, dinv != nullptr);
      else if (v.nx >= 192) launch_march<TT, CC, 16>(v, mode, a, dinv != nullptr);
      else launch_march<TT, CC, 8>(v, mode, a, dinv != nullptr);
      return;
    }
    constexpr int TX = Tile<TT>::TX, TY = Tile<TT>::TY;
    dim3 blk(TY, 256 / TY), grd((v.ny + TY - 1) / TY, (v.nx + TX - 1) / TX, B);
    if (has_mu) {
      if (mode == MODE_APPLY) stencil_kernel<TT, CC, MODE_APPLY, true><<<grd, blk, 0, st_>>>(a);
      else if (mode == MODE_RESID) stencil_kernel<TT, CC, MODE_RESID, true><<<grd, blk, 0, st_>>>(a);
      else stencil_kernel<TT, CC, MODE_JACOBI, true><<<grd, blk, 0, st_>>>(a);
    } else {
      if (mode == MODE_APPLY) stencil_kernel<TT, CC, MODE_APPLY, false><<<grd, blk, 0, st_>>>(a);
      else if (mode == MODE_RESID) stencil_kernel<TT, CC, MODE_RESID, false><<<grd, blk, 0, st_>>>(a);
      else stencil_kernel<TT, CC, MODE_JACOBI, false><<<grd, blk, 0, st_>>>(a);
    }
  }
  // pair-marching kernels (csrc/march2.cuh, csrc/march2_tma.cuh), stencil_pair = 1: real fp32 multigrid operators without mu
  // fields on even-width levels.  TMA row staging (ring of three stages) where it applies (ny % 4 == 0, not the fused first
  // sweeps), the register version with two rows of prefetch registers elsewhere.
  using March2Fn = void (*)(StencilArgs<float, float>, int);
  struct March2Pick {
    March2Fn fn = nullptr;
    int stages = 0, narr = 0;  // stages > 0: TMA version with that ring depth
  };
  March2Pick march2_pick(int md, int ny) const {
    March2Pick p;
    if ((ny % 4) == 0 && md != MODE_JACOBI_D0) {
      p.stages = 3;
      p.narr = md == MODE_APPLY ? 5 : (md == MODE_RESID ? 7 : 9);
      if (md == MODE_APPLY) p.fn = stencil_march2_tma_kernel<MODE_APPLY, 3>;
      else if (md == MODE_RESID) p.fn = stencil_march2_tma_kernel<MODE_RESID, 3>;
      else if (md == MODE_JACOBI_D) p.fn = stencil_march2_tma_kernel<MODE_JACOBI_D, 3>;
      return p;
    }
    if (md == MODE_APPLY) p.fn = stencil_march2_kernel<float, MODE_APPLY, 2>;
    else if (md == MODE_RESID) p.fn = stencil_march2_kernel<float, MODE_RESID, 2>;
    else if (md == MODE_JACOBI_D) p.fn = stencil_march2_kernel<float, MODE_JACOBI_D, 2>;
    else if (md == MODE_JACOBI_D0) p.fn = stencil_march2_kernel<float, MODE_JACOBI_D0, 2>;
    return p;
  }
  bool march2_eligible(const Level &v) const {
    return opt_.stencil_pair > 0 && !has_mu && !(v.ny & 1) && v.ny >= 8 && v.nx >= 32;
  }
  static size_t march2_smem(const March2Pick &p, int W) { return (size_t)p.stages * p.narr * W * sizeof(float2); }
  // resident CTAs on the device for this kernel at this CTA width; also raises the kernel's dynamic shared-memory limit once
  int march2_resident(const March2Pick &p, int md, int W) {
    const long key = ((long)md * 32 + p.stages) * 1024 + W;
    auto it = m2_resident_.find(key);
    if (it == m2_resident_.end()) {
      int per_sm = 0, dev = 0, sms = 148;
      if (p.stages > 0)
        CUDA_CHECK(cudaFuncSetAttribute(p.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)march2_smem(p, kM2MaxW)));
      CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, p.fn, W, march2_smem(p, W)));
      CUDA_CHECK(cudaGetDevice(&dev));
      CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
      it = m2_resident_.emplace(key, std::max(1, per_sm) * sms).first;
    }
    return it->second;
  }
  // occupancy queries and attribute changes happen here, before the V-cycle is captured into a CUDA graph
  void prime_march2() {
    if constexpr (std::is_same<P, float>::value && std::is_same<PC, float>::value) {
      for (const Level &v : lv) {
        if (!march2_eligible(v)) continue;
        int W = 0, nstrips = 0;
        march2_strips(v.ny, W, nstrips);
        for (int md : {MODE_APPLY, MODE_RESID, MODE_JACOBI_D, MODE_JACOBI_D0}) {
          const March2Pick p = march2_pick(md, v.ny);
          if (p.fn) march2_resident(p, md, W);
        }
      }
    }
  }
  template <typename TT, typename CC>
  bool launch_march2(const Level &v, int mode, const StencilArgs<TT, CC> &a, bool have_dinv) {
    if constexpr (std::is_same<TT, float>::value && std::is_same<CC, float>::value) {
      if (!march2_eligible(v)) return false;
      int md = mode;
      if (mode == MODE_JACOBI) {
        if (!have_dinv) return false;
        md = MODE_JACOBI_D;
      }
      if (md == MODE_JACOBI_D0 && !have_dinv) return false;
      const March2Pick p = march2_pick(md, v.ny);
      if (!p.fn) return false;
      int W = 0, nstrips = 0;
      march2_strips(v.ny, W, nstrips);
      const int resident = march2_resident(p, md, W);
      const int rows = opt_.stencil_pair_rows > 0 ? std::min(kM2MaxSteps - 3, 6 * ((opt_.stencil_pair_rows + 3 + 5) / 6) - 3)
                                                  : march2_rows(v.nx, nstrips, B, resident);
      dim3 grd(nstrips, (v.nx + rows - 1) / rows, B);
      p.fn<<<grd, W, march2_smem(p, W), st_>>>(a, rows);
      return true;
    }
    return false;
  }
  template <typename TT, typename CC, int TXR>
  void launch_march(const Level &v, int mode, const StencilArgs<TT, CC> &a, bool have_dinv) {
    dim3 blk(kMarchCols), grd((v.ny + kMarchOut - 1) / kMarchOut, (v.nx + TXR - 1) / TXR, B);
    if (mode == MODE_JACOBI_D0) {  // two sweeps from zero in one pass (needs the stored diagonal)
      if (has_mu) stencil_march_kernel<TT, CC, MODE_JACOBI_D0, true, TXR><<<grd, blk, 0, st_>>>(a);
      else stencil_march_kernel<TT, CC, MODE_JACOBI_D0, false, TXR><<<grd, blk, 0, st_>>>(a);
      return;
    }
    if (mode == MODE_JACOBI && have_dinv) {  // stored-diagonal sweep: fewer registers and instructions than recomputing it
      if (has_mu) stencil_march_kernel<TT, CC, MODE_JACOBI_D, true, TXR><<<grd, blk, 0, st_>>>(a);
      else stencil_march_kernel<TT, CC, MODE_JACOBI_D, false, TXR><<<grd, blk, 0, st_>>>(a);
      return;
    }
    if (has_mu) {
      if (mode == MODE_APPLY) stencil_march_kernel<TT, CC, MODE_APPLY, true, TXR><<<grd, blk, 0, st_>>>(a);
      else if (mode == MODE_RESID) stencil_march_kernel<TT, CC, MODE_RESID, true, TXR><<<grd, blk, 0, st_>>>(a);
      else stencil_march_kernel<TT, CC, MODE_JACOBI, true, TXR><<<grd, blk, 0, st_>>>(a);
    } else {
      if (mode == MODE_APPLY) stencil_march_kernel<TT, CC, MODE_APPLY, false, TXR><<<grd, blk, 0, st_>>>(a);
      else if (mode == MODE_RESID) stencil_march_kernel<TT, CC, MODE_RESID, false, TXR><<<grd, blk, 0, st_>>>(a);
      else stencil_march_kernel<TT, CC, MODE_JACOBI, false, TXR><<<grd, blk, 0, st_>>>(a);
    }
  }
  // incidence-matrix formulation (solver.py:441-449, 506-508): zero the components of removed (PEC) unknowns
  void mask_E(T *y, size_t y_bs) {
    if (!masked_) return;
    dim3 grd((unsigned)std::min<size_t>((N + 255) / 256, 1024), B);
    mask_kernel<T, C><<<grd, 256, 0, st_>>>(y, y_bs, lv[0].fields_true, lv[0].fbstride, N);
    stats.launches++;
  }
  // the reference operator (fp64, true PML) on the fine level
  void apply_true(int mode, const T *x, const T *rhs, T *y) {
    apply_true_raw(mode, x, rhs, y);
    if (!tensor_) mask_E(y, len);
  }
  void apply_true_raw(int mode, const T *x, const T *rhs, T *y) {
    stats.stencil_applies++;
    if constexpr (std::is_same<T, cplx>::value) {
      if (tensor_) {  // y = (mat - sigma) x  or  rhs - (mat - sigma) x,  mat = msign (-i) M  (solver.py:655-670)
        TensorArgs<C> a;
        a.nx = nx; a.ny = ny; a.w = x; a.rhs = (mode == MODE_RESID) ? rhs : nullptr; a.y = y;
        a.ft = ft_; a.ft_bstride = shared_fields ? 0 : 18 * N; a.cx = lv[0].cx_true; a.cy = lv[0].cy_true;
        a.sigma = sigma_; a.msign = msign_;
        dim3 blk(64, 4), grd((ny + 63) / 64, (nx + 3) / 4, B);
        tensor_apply_kernel<C><<<grd, blk, 0, st_>>>(a);
        stats.launches++;
        return;
      }
    }
    launch_stencil<T, C>(lv[0], mode, x, rhs, y, lv[0].fields_true, lv[0].cx_true, lv[0].cy_true, sigma_);
  }
  // P h / Q e with the diagonal parts of eps, mu (blocks of the first-order operator), strided two-component fields
  void apply_pq(int which, const T *in, size_t in_bs, T *out, size_t out_bs) {
    if constexpr (std::is_same<T, cplx>::value) {
      dim3 blk(64, 4), grd((ny + 63) / 64, (nx + 3) / 4, B);
      pq_kernel<C><<<grd, blk, 0, st_>>>(which, nx, ny, in, in_bs, out, out_bs, lv[0].fields_true, lv[0].fbstride, lv[0].cx_true,
                                         lv[0].cy_true);
      stats.launches++;
    }
  }
  void lin2(const cplx *ca, const T *x, size_t xbs, const cplx *cb, const T *y, size_t ybs, T *out, size_t obs) {
    if constexpr (std::is_same<T, cplx>::value) {
      dim3 grd((unsigned)std::min<size_t>((lenE + 255) / 256, 1024), B);
      lin2_kernel<<<grd, 256, 0, st_>>>(lenE, ca, x, xbs, cb, y, ybs, out, obs);
      stats.launches++;
    }
  }
  // Tensorial preconditioner: z ~ (mat_d - sigma)^-1 v with mat_d = msign (-i) [[0,P],[Q,0]] the diagonal-tensor part:
  //   (mat_d - sigma)^-1 = -(mat_d + sigma) blockdiag((PQ - s)^-1, (QP - s)^-1),  s = -sigma^2,
  //   (PQ - s)^-1 ~ B_E = the multigrid V-cycle of the diagonal path,  (QP - s)^-1 = -(1/s) (I - Q B_E P).
  // The off-diagonal tensor terms are left to the outer FGMRES.
  void precondition_tensor(const T *v, T *z) {
    const cplx *c_negsig = tcoef_, *c_ims = tcoef_ + B, *c_is = tcoef_ + 2 * B, *c_mis = tcoef_ + 3 * B, *c_one = tcoef_ + 4 * B;
    const T *ve = v, *vh = v + lenE;
    T *ye = tb_[0], *t1 = tb_[1], *g = tb_[2], *t2 = tb_[3], *yh = tb_[4], *t3 = tb_[5];
    precondition_E(ve, len, ye, lenE);          // y_e = B_E v_e
    apply_pq(0, vh, len, t1, lenE);             // t1 = P v_h
    precondition_E(t1, lenE, g, lenE);          // g = B_E t1
    apply_pq(1, g, lenE, t2, lenE);             // t2 = Q g
    lin2(c_mis, vh, len, c_is, t2, lenE, yh, lenE);  // y_h = -(1/s) v_h + (1/s) t2
    apply_pq(0, yh, lenE, t3, lenE);            // P y_h
    lin2(c_negsig, ye, lenE, c_ims, t3, lenE, z, len);          // z_e = -sigma y_e + i msign P y_h
    apply_pq(1, ye, lenE, t3, lenE);            // Q y_e
    lin2(c_negsig, yh, lenE, c_ims, t3, lenE, z + lenE, len);   // z_h = -sigma y_h + i msign Q y_e
    (void)c_one;
  }
  // the multigrid operator on level l (preconditioner precision, phase-limited PML)
  void apply(int l, int mode, const P *x, const P *rhs, P *y) {
    if (l == 0) stats.stencil_applies++;
    launch_stencil<P, PC>(lv[l], mode, x, rhs, y, lv[l].fields, lv[l].cx, lv[l].cy, sigma_p_, dinv_ready_ ? lv[l].dinv : nullptr);
  }
  void jacobi0(int l, const P *rhs, P *y) {
    Level &v = lv[l];
    if (dinv_ready_) {
      const size_t tot = (size_t)B * 2 * v.N;
      mul_kernel<P><<<(unsigned)std::min<size_t>((tot + 255) / 256, 8192), 256, 0, st_>>>(tot, v.dinv, rhs, y);
      stats.launches++;
      return;
    }
    StencilArgs<P, PC> a;
    a.nx = v.nx; a.ny = v.ny; a.x = nullptr; a.rhs = rhs; a.y = y;
    a.fields = v.fields; a.field_bstride = v.fbstride; a.cx = v.cx; a.cy = v.cy; a.sigma = sigma_p_;
    a.omega = opt_.mg_omega;
    stats.launches++;
    dim3 blk(64, 4), grd((v.ny + 63) / 64, (v.nx + 3) / 4, B);
    if (has_mu) jacobi0_kernel<P, PC, true><<<grd, blk, 0, st_>>>(a);
    else jacobi0_kernel<P, PC, false><<<grd, blk, 0, st_>>>(a);
  }
  // z = M^-1 v for Krylov-precision vectors: `mg_cycles` multigrid V-cycles (iterated on the multigrid operator's own
  // residual), converting on the way in and out when the multigrid runs in fp32.  Two cycles per application roughly
  // halve the FGMRES iteration count, which pays because the Gram-Schmidt cost grows quadratically with it.
  void precondition(const T *v, T *z) {
    if (tensor_) {
      precondition_tensor(v, z);
    } else {
      precondition_E(v, len, z, len);
      mask_E(z, len);
    }
  }
  // z = B_E v on two-component fields with batch strides v_bs / z_bs (== lenE for plain batched vectors)
  void precondition_E(const T *v, size_t v_bs, T *z, size_t z_bs) {
    const int ncyc = mg_cycles_();
    dim3 cg((unsigned)std::min<size_t>((lenE + 255) / 256, 1024), B);
    convert_strided_kernel<T, P><<<cg, 256, 0, st_>>>(lenE, v, v_bs, lv[0].b, lenE);
    if (graph_exec_) {
      CUDA_CHECK(cudaGraphLaunch(graph_exec_, st_));
      stats.launches += graph_nodes_;
      stats.stencil_applies += graph_fine_applies_;
    } else {
      precondition_body(lv[0].b, nullptr, ncyc);
      graph_result_ = ncyc == 1 ? lv[0].x : pre_b_;
    }
    convert_strided_kernel<P, T><<<cg, 256, 0, st_>>>(lenE, graph_result_, lenE, z, z_bs);
    stats.launches += 2;
  }
  // V-cycles per application of the E-block inverse.  The tensorial block preconditioner needs an accurate one: its H block is
  // -(1/s)(I - Q B_E P), the difference of two O(K^2) terms (K = 1/(k0 h)) whose exact value is O(K^-2), so a B_E with the ~0.15
  // relative error of one V-cycle leaves an O(0.15 K^2) error there and the outer FGMRES count grows with the resolution
  // (tools/proto_tensor.py: 25 / 52 / 90 / > 200 iterations at 64^2 / 96^2 / 128^2 / 192^2, against 17 at 128^2 and 49 at 256^2
  // with three defect-correction cycles in both blocks).
  int mg_cycles_() const { return (tensor_ && opt_.tensor_mg_cycles > 0) ? opt_.tensor_mg_cycles : std::max(1, opt_.mg_cycles); }
  // rin -> M^-1 rin in multigrid precision.  out == nullptr: result in lv[0].x (one cycle) or pre_b_ (several)
  void precondition_body(const P *rin, P *out, int ncyc) {
    const unsigned nb = (unsigned)std::min<size_t>((vsE + 255) / 256, 8192);
    if (ncyc == 1) {
      vcycle(0, rin, out);
      return;
    }
    P *acc = out ? out : pre_b_;
    vcycle(0, rin, acc);
    for (int c = 1; c < ncyc; ++c) {
      apply(0, MODE_RESID, acc, rin, pre_a_);
      vcycle(0, pre_a_, nullptr);
      axpby_kernel<P><<<nb, 256, 0, st_>>>(vsE, 1.0, lv[0].x, 1.0, acc);
      stats.launches++;
    }
  }
  // Capture the V-cycle(s) into a CUDA graph (its input and output buffers are fixed).  The cycle is ~60-250 small
  // launches; replaying it as one graph removes most of the launch latency of the coarse levels.
  void capture_precondition_graph() {
    if (!opt_.use_graph) return;
    const int ncyc = mg_cycles_();
    const long l0 = stats.launches, a0 = stats.stencil_applies;
    cudaGraph_t graph = nullptr;
    CUDA_CHECK(cudaStreamSynchronize(st_));
    CUDA_CHECK(cudaStreamBeginCapture(st_, cudaStreamCaptureModeRelaxed));
    precondition_body(lv[0].b, nullptr, ncyc);
    cudaError_t e = cudaStreamEndCapture(st_, &graph);
    graph_nodes_ = stats.launches - l0;
    graph_fine_applies_ = stats.stencil_applies - a0;
    stats.launches = l0;
    stats.stencil_applies = a0;
    graph_result_ = ncyc == 1 ? lv[0].x : pre_b_;
    if (e != cudaSuccess || !graph) {
      cudaGetLastError();
      graph_exec_ = nullptr;
      return;
    }
    if (cudaGraphInstantiate(&graph_exec_, graph, 0) != cudaSuccess) {
      cudaGetLastError();
      graph_exec_ = nullptr;
    }
    cudaGraphDestroy(graph);
  }
  ~BatchSolver() {
    if (graph_exec_) cudaGraphExecDestroy(graph_exec_);
  }

  // Levels [fused_l0_, L) run as one kernel (csrc/coarse_kernel.cuh) when they fit in shared memory together: the
  // largest tail whose level vectors (8 N elements per level) stay under ~200 KB, starting at <= 64^2 cells.
  void plan_fused_tail() {
    fused_l0_ = -1;
    const int L = (int)lv.size();
    if (!opt_.mg_fused_tail || coarse_krylov_ || opt_.mg_nu_growth != 0) return;
    int l0 = L;
    size_t elems = 0;
    while (l0 > 0 && L - (l0 - 1) <= kFusedMaxLevels) {
      const size_t add = (size_t)8 * lv[l0 - 1].N;
      if (lv[l0 - 1].N > 4096 || (elems + add) * sizeof(P) > (size_t)200 * 1024) break;
      elems += add;
      --l0;
    }
    if (l0 >= L || L - l0 < 2) return;  // nothing worth fusing
    fused_l0_ = l0;
    fused_smem_ = elems * sizeof(P);
    if (has_mu) CUDA_CHECK(cudaFuncSetAttribute(fused_vcycle_kernel<P, PC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fused_smem_));
    else CUDA_CHECK(cudaFuncSetAttribute(fused_vcycle_kernel<P, PC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fused_smem_));
  }
  void launch_fused_tail(const P *rin, P *xout) {
    const int L = (int)lv.size();
    FusedArgs<P, PC> a;
    a.nl = L - fused_l0_;
    a.nu = std::max(1, opt_.mg_nu);
    a.ncoarse = std::max(2, opt_.mg_coarse_iters);
    for (int q = 0; q < a.nl; ++q) {
      const Level &v = lv[fused_l0_ + q];
      a.lv[q].nx = v.nx; a.lv[q].ny = v.ny; a.lv[q].fields = v.fields; a.lv[q].fbstride = v.fbstride;
      a.lv[q].cx = v.cx; a.lv[q].cy = v.cy; a.lv[q].dinv = v.dinv; a.lv[q].tr = v.tr;
    }
    a.rin = rin; a.xout = xout; a.sigma = sigma_p_;
    stats.launches++;
    if (has_mu) fused_vcycle_kernel<P, PC, true><<<B, 512, fused_smem_, st_>>>(a);
    else fused_vcycle_kernel<P, PC, false><<<B, 512, fused_smem_, st_>>>(a);
  }

  // -- multigrid V-cycle: z = M^-1 rin on level l.  Result lands in `out` (or lv[l].x if null). ----
  void vcycle(int l, const P *rin, P *out) {
    Level &v = lv[l];
    if (l == fused_l0_) {
      launch_fused_tail(rin, out ? out : v.x);
      return;
    }
    const int L = (int)lv.size();
    const int nu = std::max(1, opt_.mg_nu + l * opt_.mg_nu_growth);  // optional variable V-cycle: more sweeps on coarser levels
    P *cur = v.x, *oth = v.tmp;
    auto sweep = [&](P *dst) {  // dst = jacobi(cur)
      apply(l, MODE_JACOBI, cur, rin, dst);
    };
    if (l == L - 1 && coarse_krylov_) {
      coarse_gmres(l, rin, out ? out : cur);
      return;
    }
    if (l == L - 1) {
      const int n_sw = std::max(2, opt_.mg_coarse_iters);
      jacobi0(l, rin, cur);
      for (int s = 1; s < n_sw; ++s) {
        P *dst = (s == n_sw - 1 && out) ? out : oth;
        sweep(dst);
        if (dst != out) std::swap(cur, oth);
      }
      if (!out) { v.x = cur; v.tmp = oth; }
      return;
    }
    // (real fp32 only: the complex variant needs more registers and measured 3 % slower on c3_512)
    if (nu >= 2 && dinv_ready_ && opt_.mg_fuse_first && sizeof(P) <= 4 && v.nx >= 32 && v.ny >= 2) {
      apply(l, MODE_JACOBI_D0, cur, rin, cur);  // sweeps 1 and 2 from the zero guess in one pass (x argument unused)
      for (int s = 2; s < nu; ++s) {
        sweep(oth);
        std::swap(cur, oth);
      }
    } else {
      jacobi0(l, rin, cur);
      for (int s = 1; s < nu; ++s) {
        sweep(oth);
        std::swap(cur, oth);
      }
    }
    apply(l, MODE_RESID, cur, rin, v.r);
    {
      const TransferArgs &t = v.tr;
      dim3 blk(64, 4), grd((t.nyc + 63) / 64, (t.nxc + 3) / 4, 2 * B);
      const bool packed = (opt_.transfer_vec & 2) && t.xn.r4 && t.xe.r4 && t.yn.r4 && t.ye.r4;
      if (packed) restrict4_kernel<P><<<grd, blk, 0, st_>>>(t, v.r, lv[l + 1].b);
      else restrict_kernel<P><<<grd, blk, 0, st_>>>(t, v.r, lv[l + 1].b);
      stats.launches += 2;
    }
    vcycle(l + 1, lv[l + 1].b, nullptr);
    {
      const TransferArgs &t = v.tr;
      if (t.nyf >= 256) {  // four fine columns per thread
        dim3 blk(64, 4), grd((t.nyf + 255) / 256, (t.nxf + 3) / 4, 2 * B);
        if ((opt_.transfer_vec & 1) && std::is_same<P, float>::value && (t.nyf % 4) == 0) prolong_add4_kernel<P, true><<<grd, blk, 0, st_>>>(t, lv[l + 1].x, cur);
        else prolong_add4_kernel<P, false><<<grd, blk, 0, st_>>>(t, lv[l + 1].x, cur);
      } else {
        dim3 blk(64, 4), grd((t.nyf + 63) / 64, (t.nxf + 3) / 4, 2 * B);
        prolong_add_kernel<P><<<grd, blk, 0, st_>>>(t, lv[l + 1].x, cur);
      }
    }
    for (int s = 0; s < nu; ++s) {
      P *dst = (s == nu - 1 && out) ? out : oth;
      sweep(dst);
      if (dst != out) std::swap(cur, oth);
    }
    if (!out) { v.x = cur; v.tmp = oth; }
  }

  // -- coarsest-level Krylov solve (indefinite shifts): GMRES(kc), Jacobi right-preconditioned, CGS2, run entirely
  //    on the device (no host synchronisation; the small least-squares problem is solved by one thread per problem)
  void coarse_gmres(int l, const P *rin, P *xout) {
    Level &v = lv[l];
    const int kc = kc_;
    const size_t ln = 2 * v.N, vs = (size_t)B * ln;
    const int ld = kc + 4;
    CUDA_CHECK(cudaMemsetAsync(cH_, 0, (size_t)B * kc * ld * sizeof(P), st_));
    dots(rin, 1, rin, cbeta_, 1, 0, false, ln, vs);
    scale_inv_norm(rin, cV_, cbeta_, 1, ln);
    for (int j = 0; j < kc; ++j) {
      P *vj = cV_ + (size_t)j * vs, *zj = cZ_ + (size_t)j * vs, *w = cV_ + (size_t)(j + 1) * vs;
      jacobi0(l, vj, zj);
      apply(l, MODE_APPLY, zj, nullptr, w);
      P *col = cH_ + (size_t)j * ld;  // problem stride kc*ld
      dots(cV_, j + 1, w, col, kc * ld, 0, false, ln, vs);
      axpys(cV_, j + 1, col, kc * ld, -1.0, w, ln, vs);
      dots(cV_, j + 1, w, cH2_, kc + 1, 0, false, ln, vs);
      axpys(cV_, j + 1, cH2_, kc + 1, -1.0, w, ln, vs);
      add_small_kernel<P><<<B, 64, 0, st_>>>(col, kc * ld, cH2_, kc + 1, j + 1);  // H[:, j] += second-pass coefficients
      dots(w, 1, w, col, kc * ld, j + 1, false, ln, vs);
      scale_inv_norm(w, w, col + j + 1, kc * ld, ln);
    }
    gmres_lsq_kernel<P><<<(B + 31) / 32, 32, 0, st_>>>(cH_, kc, ld, cbeta_, 1, cy_, B);
    CUDA_CHECK(cudaMemsetAsync(xout, 0, vs * sizeof(P), st_));
    axpys(cZ_, kc, cy_, kc, +1.0, xout, ln, vs);
  }

  // -- batched BLAS-1 helpers -----------------------------------------------------------------------
  int pstride() const { return std::max(m, restart) + 2; }
  int hstride() const { return 2 * (std::max(m, restart) + 2) + 2; }
  int vec_blocks() const { return (int)std::min<size_t>((len + 255) / 256, 1024); }

  // dst[b][off + i] (+)= <V_i, w>, i < nv   (vectors of length ln, basis stride vs)
  template <typename U>
  void dots(const U *V, int nv, const U *w, U *dst, int dstride, int off, bool accumulate, size_t ln = 0, size_t vs = 0) {
    if (!ln) { ln = len; vs = vstride; }
    const int chunks = (int)std::max<size_t>(1, std::min<size_t>(kDotChunks, (ln + 2047) / 2048));
    stats.launches += 2;
    dim3 grd(chunks, B);
    U *part = reinterpret_cast<U *>(partial_);
    multidot_partial_kernel<U><<<grd, 256, 0, st_>>>(V, vs, ln, w, nv, part, pstride());
    multidot_final_kernel<U><<<B, std::max(32, ((nv + 31) / 32) * 32), 0, st_>>>(part, chunks, pstride(), nv, dst + off,
                                                                                dstride, accumulate ? 1 : 0);
  }
  template <typename U>
  void axpys(const U *V, int nv, const U *coef, int cstride, double sign, U *w, size_t ln = 0, size_t vs = 0) {
    if (!ln) { ln = len; vs = vstride; }
    stats.launches++;
    dim3 grd((unsigned)std::min<size_t>((ln + 255) / 256, 1024), B);
    multiaxpy_kernel<U><<<grd, 256, nv * sizeof(U), st_>>>(V, vs, ln, coef, cstride, nv, sign, w);
  }
  template <typename U>
  void scale_inv_norm(const U *x, U *y, const U *nrm2, int stride, size_t ln = 0) {
    if (!ln) ln = len;
    stats.launches++;
    dim3 grd((unsigned)std::min<size_t>((ln + 255) / 256, 1024), B);
    scale_kernel<U><<<grd, 256, 0, st_>>>(x, y, ln, nrm2, stride, 1);
  }
  void copy(const T *src, T *dst) { CUDA_CHECK(cudaMemcpyAsync(dst, src, vstride * sizeof(T), cudaMemcpyDeviceToDevice, st_)); }
  void fetch_h(size_t count) {
    CUDA_CHECK(cudaMemcpyAsync(hhost_.data(), hbuf_, count * sizeof(T), cudaMemcpyDeviceToHost, st_));
    CUDA_CHECK(cudaStreamSynchronize(st_));
  }

  // Gram-Schmidt of w = V_nv (the slot right after the basis) against V_0..V_{nv-1}, then normalise into dst.
  // selective = false: two classical passes (CGS2).  selective = true: one pass, a second one only when the
  // cancellation test ||w'|| < 1e-2 ||w|| fires for some problem (w.w comes for free as an extra column of the first
  // multi-dot).  Leaves h (nv values per problem) and ||w'|| in the output vectors.
  void orthonormalise(const T *V, int nv, T *w, T *dst, std::vector<cd> &h, std::vector<double> &nrm, bool selective = false,
                      const std::vector<char> *skip = nullptr) {
    const int hs = hstride(), half = std::max(m, restart) + 2;
    h.assign((size_t)B * nv, cd(0, 0));
    nrm.assign(B, 0.0);
    bool second = !selective;
    if (selective) {
      dots(V, nv + 1, w, hbuf_, hs, 0, false);  // column nv is w.w (w sits in slot nv)
      axpys(V, nv, hbuf_, hs, -1.0, w);
      pythagoras_kernel<T><<<(B + 31) / 32, 32, 0, st_>>>(hbuf_, hs, nv, hbuf_ + 2 * half, hs, B);
      stats.launches++;
      fetch_h((size_t)B * hs);
      for (int b = 0; b < B; ++b) {
        if (skip && (*skip)[b]) continue;
        const double ww = to_cd(hhost_[(size_t)b * hs + nv]).real();
        const double after = to_cd(hhost_[(size_t)b * hs + 2 * half]).real();
        if (!(after >= 1e-4 * ww)) second = true;  // ||w'|| < 1e-2 ||w||: cancellation would cost > 2 digits of orthogonality
      }
      for (int b = 0; b < B; ++b)
        for (int i = 0; i < nv; ++i) h[(size_t)b * nv + i] = to_cd(hhost_[(size_t)b * hs + i]);
      if (!second) {
        scale_inv_norm(w, dst, hbuf_ + 2 * half, hs);
        for (int b = 0; b < B; ++b) nrm[b] = std::sqrt(std::max(0.0, to_cd(hhost_[(size_t)b * hs + 2 * half]).real()));
        return;
      }
    } else {
      dots(V, nv, w, hbuf_, hs, 0, false);
      axpys(V, nv, hbuf_, hs, -1.0, w);
    }
    dots(V, nv, w, hbuf_, hs, half, false);
    axpys(V, nv, hbuf_ + half, hs, -1.0, w);
    dots(w, 1, w, hbuf_, hs, 2 * half, false);
    scale_inv_norm(w, dst, hbuf_ + 2 * half, hs);
    fetch_h((size_t)B * hs);
    for (int b = 0; b < B; ++b) {
      for (int i = 0; i < nv; ++i) {
        cd first = selective ? h[(size_t)b * nv + i] : to_cd(hhost_[(size_t)b * hs + i]);
        h[(size_t)b * nv + i] = first + to_cd(hhost_[(size_t)b * hs + half + i]);
      }
      nrm[b] = std::sqrt(std::max(0.0, to_cd(hhost_[(size_t)b * hs + 2 * half]).real()));
    }
  }

  // -- FGMRES: xsol_ = (A - sigma)^-1 rhs ------------------------------------------------------------
  // returns max relative residual estimate; iters_out = iterations of the slowest problem
  double fgmres(const T *rhs, T *xsol, int &iters_out, const std::vector<char> *skip = nullptr,
                const std::vector<double> *tolv = nullptr) {
    auto tol_of = [&](int b) { return tolv ? (*tolv)[b] : opt_.inner_tol; };
    std::vector<char> done(B, 0);
    if (skip) done = *skip;
    std::vector<double> bnorm(B, 0.0), res(B, 0.0);
    std::vector<cd> h;
    std::vector<double> nrm;
    CUDA_CHECK(cudaMemsetAsync(xsol, 0, vstride * sizeof(T), st_));
    int total_it = 0;
    bool first = true;
    while (true) {
      // r -> Vg_[0] normalised
      T *r0 = Vg_;
      if (first) copy(rhs, rhs_); else apply_true(MODE_RESID, xsol, rhs, rhs_);
      dots(rhs_, 1, rhs_, hbuf_, hstride(), 0, false);
      scale_inv_norm(rhs_, r0, hbuf_, hstride());
      fetch_h((size_t)B * hstride());
      std::vector<double> beta(B);
      bool all_done = true;
      for (int b = 0; b < B; ++b) {
        beta[b] = std::sqrt(std::max(0.0, to_cd(hhost_[(size_t)b * hstride()]).real()));
        if (first) bnorm[b] = beta[b];
        res[b] = bnorm[b] > 0 ? beta[b] / bnorm[b] : 0.0;
        if (!(beta[b] > 0) || res[b] <= tol_of(b)) done[b] = 1;
        if (!done[b]) all_done = false;
      }
      first = false;
      if (all_done || total_it >= opt_.gmres_maxit) break;
      // per-problem least-squares state
      std::vector<CMat> R(B, CMat(restart + 1, restart));
      std::vector<std::vector<cd>> g(B, std::vector<cd>(restart + 1, cd(0, 0))), cs(B), sn(B);
      std::vector<int> kused(B, 0);
      std::vector<char> cyc_done = done;
      for (int b = 0; b < B; ++b) g[b][0] = beta[b];
      int kk = 0;
      for (; kk < restart && total_it < opt_.gmres_maxit; ++kk) {
        T *vk = Vg_ + (size_t)kk * vstride, *zk = Zg_ + (size_t)kk * vstride, *w = Vg_ + (size_t)(kk + 1) * vstride;
        precondition(vk, zk);
        apply_true(MODE_APPLY, zk, nullptr, w);
        // classical Gram-Schmidt loses orthogonality like eps * kappa^2 with kappa ~ 1 / (relative residual): one pass
        // is enough while every active problem is still above ~1e-6, two passes (CGS2) below that
        double minres = 1.0;
        for (int b = 0; b < B; ++b)
          if (!cyc_done[b]) minres = std::min(minres, res[b]);
        const bool one_pass = opt_.gmres_cgs2 == 0 || (opt_.gmres_cgs2 == 2 && minres > 3e-6);
        orthonormalise(Vg_, kk + 1, w, w, h, nrm, one_pass, &cyc_done);
        ++total_it;
        bool all = true;
        for (int b = 0; b < B; ++b) {
          if (cyc_done[b]) continue;
          CMat &Rb = R[b];
          for (int i = 0; i <= kk; ++i) Rb(i, kk) = h[(size_t)b * (kk + 1) + i];
          Rb(kk + 1, kk) = nrm[b];
          for (int i = 0; i < kk; ++i) {  // previous rotations
            cd a0 = Rb(i, kk), a1 = Rb(i + 1, kk);
            Rb(i, kk) = std::conj(cs[b][i]) * a0 + std::conj(sn[b][i]) * a1;
            Rb(i + 1, kk) = -sn[b][i] * a0 + cs[b][i] * a1;
          }
          cd a0 = Rb(kk, kk), a1 = Rb(kk + 1, kk);
          double d = std::sqrt(std::norm(a0) + std::norm(a1));
          cd c = d > 0 ? a0 / d : cd(1, 0), s = d > 0 ? a1 / d : cd(0, 0);
          cs[b].push_back(c);
          sn[b].push_back(s);
          Rb(kk, kk) = d;
          Rb(kk + 1, kk) = 0.0;
          g[b][kk + 1] = -s * g[b][kk];
          g[b][kk] = std::conj(c) * g[b][kk];
          kused[b] = kk + 1;
          res[b] = std::abs(g[b][kk + 1]) / bnorm[b];
          if (res[b] <= tol_of(b) || !(nrm[b] > 0)) cyc_done[b] = 1;
          if (!cyc_done[b]) all = false;
        }
        if (all) {
          ++kk;
          break;
        }
      }
      // y = R^-1 g, x += Z y
      const int kmax = kk;
      std::vector<T> yh((size_t)B * restart, zero_of<T>());
      for (int b = 0; b < B; ++b) {
        if (done[b]) continue;
        const int ku = kused[b];
        std::vector<cd> y(ku);
        for (int i = ku - 1; i >= 0; --i) {
          cd acc = g[b][i];
          for (int j = i + 1; j < ku; ++j) acc -= R[b](i, j) * y[j];
          y[i] = (std::abs(R[b](i, i)) > 0) ? acc / R[b](i, i) : cd(0, 0);
        }
        for (int i = 0; i < ku; ++i) yh[(size_t)b * restart + i] = from_cd<T>(y[i]);
      }
      CUDA_CHECK(cudaMemcpyAsync(qbuf_, yh.data(), yh.size() * sizeof(T), cudaMemcpyHostToDevice, st_));
      if (kmax > 0) axpys(Zg_, kmax, qbuf_, restart, +1.0, xsol);
      CUDA_CHECK(cudaStreamSynchronize(st_));
      bool all_conv = true;
      for (int b = 0; b < B; ++b) {
        if (cyc_done[b] && res[b] <= tol_of(b)) done[b] = 1;
        if (!done[b]) all_conv = false;
      }
      if (all_conv) break;  // the FGMRES residual estimate is the true residual up to rounding
    }
    iters_out = total_it;
    stats.inner_iters += total_it;
    double worst = 0.0;
    for (int b = 0; b < B; ++b)
      if (!skip || !(*skip)[b]) worst = std::max(worst, res[b]);
    return worst;
  }


  // =====================================================================================================
  // Round-2 inner solver: device-resident FGMRES cycles (Gram-Schmidt coefficients never visit the host, the
  // least-squares problem is solved by one thread per problem, the host reads back only (estimate, columns used)
  // once or twice per cycle), run in the multigrid precision (fp32) inside an fp64 iterative refinement:
  //   r = b - (A - sigma) x  (fp64)  ->  d = FGMRES_fp32(r / ||r||)  ->  x += ||r|| d  (fp64)
  // Each fp32 cycle needs only ~1e-4 of reduction, so its Krylov basis is short, its Gram-Schmidt bytes are halved and
  // no fp64<->fp32 conversion surrounds the V-cycle.  Falls back to fp64 cycles when refinement stagnates.
  // =====================================================================================================
  template <typename U>
  static bool vec_ok(size_t ln) { return ln % PackTraits<U>::EPV == 0; }
  int gs_chunks(size_t ln) const {
    const size_t packs = std::max<size_t>(1, ln / 2);
    return (int)std::max<size_t>(1, std::min<size_t>({(size_t)kDotChunks, packs / 1024 + 1, (size_t)(1184 + B - 1) / B}));
  }
  // CTAs per problem for the streaming kernels with a reduction prologue (scale, ir_begin, ir_update): ~8 per SM in total
  int stream_blocks(size_t ln) const {
    return (int)std::max<size_t>(1, std::min<size_t>({(size_t)256, ln / 2048 + 1, (size_t)(148 * 8 + B - 1) / B}));
  }
  template <typename U>
  U *gpart(int region) { return reinterpret_cast<U *>(gpart_) + (size_t)region * B * kDotChunks * pstride(); }

  // partial[b][chunk][poff + i] = <V_i, w>, i < nv (groups of kGsGroup)
  template <typename U>
  void k_dots(const U *V, size_t vs, size_t ln, const U *w, int nv, U *part, int poff, int nch) {
    dim3 grd(nch, B);
    for (int g0 = 0; g0 < nv; g0 += kGsGroup) {
      const int ng = std::min(kGsGroup, nv - g0);
      stats.launches++;
#define B200_DOTS(EPV, NG) gs_dots_kernel<U, EPV, NG><<<grd, 256, 0, st_>>>(V, vs, ln, w, g0, ng, part, pstride(), poff + g0)
      if (vec_ok<U>(ln)) {
        constexpr int E = PackTraits<U>::EPV;
        if (ng == 1) B200_DOTS(E, 1); else if (ng == 2) B200_DOTS(E, 2); else if (ng <= 4) B200_DOTS(E, 4); else B200_DOTS(E, 8);
      } else {
        if (ng == 1) B200_DOTS(1, 1); else if (ng == 2) B200_DOTS(1, 2); else if (ng <= 4) B200_DOTS(1, 4); else B200_DOTS(1, 8);
      }
#undef B200_DOTS
    }
  }
  template <typename U>
  void k_update_dots(const U *V, size_t vs, size_t ln, U *w, int nv, const U *pin, int nch, U *pout, U *hexp, size_t hstride, int acc) {
    dim3 grd(nch, B);
    stats.launches++;
    if (vec_ok<U>(ln)) gs_update_dots_kernel<U, PackTraits<U>::EPV><<<grd, 256, 0, st_>>>(V, vs, ln, w, nv, pin, nch, pstride(), 0, pout, 0, hexp, hstride, 0, acc);
    else gs_update_dots_kernel<U, 1><<<grd, 256, 0, st_>>>(V, vs, ln, w, nv, pin, nch, pstride(), 0, pout, 0, hexp, hstride, 0, acc);
  }
  template <typename U>
  void k_update_norm(const U *V, size_t vs, size_t ln, U *w, int nv, const U *pin, int nch, U *pout, int do_norm, U *hexp, size_t hstride, int acc) {
    dim3 grd(nch, B);
    stats.launches++;
    if (vec_ok<U>(ln)) gs_update_norm_kernel<U, PackTraits<U>::EPV><<<grd, 256, 0, st_>>>(V, vs, ln, w, nv, pin, nch, pstride(), 0, pout, 0, do_norm, hexp, hstride, 0, acc);
    else gs_update_norm_kernel<U, 1><<<grd, 256, 0, st_>>>(V, vs, ln, w, nv, pin, nch, pstride(), 0, pout, 0, do_norm, hexp, hstride, 0, acc);
  }
  template <typename U>
  void k_scale(const U *w, U *y, U *y2, size_t ln, const U *pin, int nch, U *hexp, size_t hstride, int hoff) {
    dim3 grd((unsigned)stream_blocks(ln), B);  // few fat CTAs: every CTA pays the prologue reduction once
    stats.launches++;
    if (vec_ok<U>(ln)) gs_scale_kernel<U, PackTraits<U>::EPV><<<grd, 256, 0, st_>>>(w, y, y2, ln, pin, nch, pstride(), 0, hexp, hstride, hoff);
    else gs_scale_kernel<U, 1><<<grd, 256, 0, st_>>>(w, y, y2, ln, pin, nch, pstride(), 0, hexp, hstride, hoff);
  }
  // CGS2 of w against V_0..V_{nv-1}, normalised into dst (and dst2 if given).  Exports h_i (both passes summed) to
  // hexp[b*hstride + i] and ||w''||^2 to hexp[b*hstride + nv].  No host synchronisation.
  template <typename U>
  void gs_cgs2(const U *V, size_t vs, size_t ln, int nv, U *w, U *dst, U *dst2, U *hexp, size_t hstride) {
    U *P0 = gpart<U>(0), *P1 = gpart<U>(1), *P2 = gpart<U>(2);
    const int nch = gs_chunks(ln);
    if (nv <= kGsGroup) {
      k_dots<U>(V, vs, ln, w, nv, P0, 0, nch);
      k_update_dots<U>(V, vs, ln, w, nv, P0, nch, P1, hexp, hstride, 0);
      k_update_norm<U>(V, vs, ln, w, nv, P1, nch, P2, 1, hexp, hstride, 1);
    } else {
      k_dots<U>(V, vs, ln, w, nv, P0, 0, nch);
      k_update_norm<U>(V, vs, ln, w, nv, P0, nch, P2, 0, hexp, hstride, 0);
      k_dots<U>(V, vs, ln, w, nv, P1, 0, nch);
      k_update_norm<U>(V, vs, ln, w, nv, P1, nch, P2, 1, hexp, hstride, 1);
    }
    k_scale<U>(w, dst, dst2, ln, P2, nch, hexp, hstride, nv);
  }
  // outer (Krylov-Schur) orthonormalisation through the device kernels.  Classical Gram-Schmidt with the DGKS test
  // ARPACK uses (dgetv0/dnaitr: reorthogonalise when ||w'|| < 0.717 ||w||): the second pass -- two more reads of the
  // whole fp64 basis -- runs only when some active problem needs it.
  void orthonormalise_dev(const T *V, int nv, T *w, T *dst, std::vector<cd> &h, std::vector<double> &nrm, const std::vector<char> *skip = nullptr) {
    const int hs = hstride();
    T *P0 = gpart<T>(0), *P1 = gpart<T>(1), *P2 = gpart<T>(2);
    const int nch = gs_chunks(len);
    k_dots<T>(V, vstride, len, w, nv, P0, 0, nch);
    k_update_norm<T>(V, vstride, len, w, nv, P0, nch, P2, 1, hbuf_, (size_t)hs, 0);
    sum_partials_kernel<T><<<(B + 63) / 64, 64, 0, st_>>>(P2, nch, pstride(), 0, n2_dev_, B);
    stats.launches++;
    std::vector<double> n2(B);
    CUDA_CHECK(cudaMemcpyAsync(n2.data(), n2_dev_, B * sizeof(double), cudaMemcpyDeviceToHost, st_));
    fetch_h((size_t)B * hs);
    h.assign((size_t)B * nv, cd(0, 0));
    nrm.assign(B, 0.0);
    bool second = false;
    for (int b = 0; b < B; ++b) {
      double before = n2[b];
      for (int i = 0; i < nv; ++i) {
        h[(size_t)b * nv + i] = to_cd(hhost_[(size_t)b * hs + i]);
        before += std::norm(h[(size_t)b * nv + i]);
      }
      if (skip && (*skip)[b]) continue;
      if (!(n2[b] >= 0.5 * before)) second = true;  // ||w'|| < 0.707 ||w||
    }
    if (second || opt_.outer_dgks == 0) {
      k_dots<T>(V, vstride, len, w, nv, P1, 0, nch);
      k_update_norm<T>(V, vstride, len, w, nv, P1, nch, P2, 1, hbuf_, (size_t)hs, 1);
      stats.outer_second_pass++;
    }
    k_scale<T>(w, dst, nullptr, len, P2, nch, hbuf_, (size_t)hs, nv);
    if (second || opt_.outer_dgks == 0) {
      fetch_h((size_t)B * hs);
      for (int b = 0; b < B; ++b)
        for (int i = 0; i < nv; ++i) h[(size_t)b * nv + i] = to_cd(hhost_[(size_t)b * hs + i]);
      for (int b = 0; b < B; ++b) nrm[b] = std::sqrt(std::max(0.0, to_cd(hhost_[(size_t)b * hs + nv]).real()));
    } else {
      for (int b = 0; b < B; ++b) nrm[b] = std::sqrt(std::max(0.0, n2[b]));
    }
  }

  template <typename U>
  void apply_true_u(int mode, const U *x, const U *rhs, U *y) {
    if constexpr (std::is_same<U, T>::value) {
      apply_true(mode, x, rhs, y);
    } else {
      stats.stencil_applies++;
      launch_stencil<P, PC>(lv[0], mode, x, rhs, y, lv[0].fields, cx_true_p_, cy_true_p_, sigma_p_);
    }
  }
  // z = M^-1 v.  For the multigrid-precision path the input is expected in lv[0].b already (the kernels that produce
  // Krylov vectors store them there as well) and the V-cycle result is copied into the Z slot.
  template <typename U>
  void precondition_u(const U *v, U *z, bool input_staged) {
    if constexpr (std::is_same<U, T>::value) {
      precondition(v, z);
    } else {
      if (!input_staged) CUDA_CHECK(cudaMemcpyAsync(lv[0].b, v, vsE * sizeof(P), cudaMemcpyDeviceToDevice, st_));
      const int ncyc = mg_cycles_();
      if (graph_exec_) {
        CUDA_CHECK(cudaGraphLaunch(graph_exec_, st_));
        stats.launches += graph_nodes_;
        stats.stencil_applies += graph_fine_applies_;
      } else {
        precondition_body(lv[0].b, nullptr, ncyc);
        graph_result_ = ncyc == 1 ? lv[0].x : pre_b_;
      }
      CUDA_CHECK(cudaMemcpyAsync(z, graph_result_, vsE * sizeof(P), cudaMemcpyDeviceToDevice, st_));
    }
  }

  // One FGMRES cycle from the unit-norm residual sitting in slot 0 of the basis.  tol[b] < 0: problem inactive.
  // Returns the number of Arnoldi steps run; y (device, type U) holds the solution coefficients.
  template <typename U>
  int fgmres_cycle(const std::vector<double> &tol, std::vector<double> &res, std::vector<int> &jused, bool staged, int budget) {
    U *Vu = reinterpret_cast<U *>(Vg_), *Zu = reinterpret_cast<U *>(Zg_), *Hu = reinterpret_cast<U *>(Hd_);
    U *yu = reinterpret_cast<U *>(ydev_);
    const int ld = restart + 4;
    constexpr bool kStage = std::is_same<U, P>::value;
    CUDA_CHECK(cudaMemcpyAsync(tol_dev_, tol.data(), B * sizeof(double), cudaMemcpyHostToDevice, st_));
    double tmin = 1.0;
    for (int b = 0; b < B; ++b)
      if (tol[b] >= 0) tmin = std::min(tmin, tol[b]);
    const int cap = std::max(1, std::min(restart, budget));
    int target = (int)std::ceil(std::log(std::max(tmin, 1e-300)) / std::log(std::min(0.9, std::max(1e-3, rho_))));
    target = std::max(1, std::min(cap, target));
    int j = 0;
    res.assign(B, 0.0);
    jused.assign(B, 0);
    std::vector<double> hres(B);
    std::vector<int> hju(B);
    while (true) {
      for (; j < target; ++j) {
        U *vj = Vu + (size_t)j * vstride, *zj = Zu + (size_t)j * vstride, *w = Vu + (size_t)(j + 1) * vstride;
        precondition_u<U>(vj, zj, kStage && (j > 0 || staged));
        apply_true_u<U>(MODE_APPLY, zj, nullptr, w);
        gs_cgs2<U>(Vu, vstride, len, j + 1, w, w, kStage ? reinterpret_cast<U *>(lv[0].b) : nullptr, Hu + (size_t)j * ld, (size_t)restart * ld);
      }
      fgmres_lsq_kernel<U><<<(B + 31) / 32, 32, 0, st_>>>(Hu, restart, ld, j, tol_dev_, lsq_work_, yu, restart, res_dev_, jused_dev_, B);
      stats.launches++;
      CUDA_CHECK(cudaMemcpyAsync(hres.data(), res_dev_, B * sizeof(double), cudaMemcpyDeviceToHost, st_));
      CUDA_CHECK(cudaMemcpyAsync(hju.data(), jused_dev_, B * sizeof(int), cudaMemcpyDeviceToHost, st_));
      CUDA_CHECK(cudaStreamSynchronize(st_));
      stats.host_syncs++;
      bool all = true;
      int need = 0;
      for (int b = 0; b < B; ++b) {
        if (tol[b] < 0) continue;
        if (hres[b] > tol[b] && hju[b] == j) {  // not converged and no breakdown
          all = false;
          const double rate = std::min(0.95, std::max(1e-3, std::pow(std::max(hres[b], 1e-300), 1.0 / std::max(1, j))));
          need = std::max(need, (int)std::ceil(std::log(tol[b] / hres[b]) / std::log(rate)));
        }
      }
      if (all || j >= cap) break;
      target = std::min(cap, j + std::max(1, std::min(need, 8)));
    }
    double rmax = 1e-3;
    for (int b = 0; b < B; ++b) {
      res[b] = hres[b];
      jused[b] = hju[b];
      if (tol[b] >= 0 && hju[b] > 0) rmax = std::max(rmax, std::pow(std::max(hres[b], 1e-300), 1.0 / hju[b]));
    }
    rho_ = std::min(0.9, rmax);
    return j;
  }

  // xsol = (A - sigma)^-1 rhs for every problem not in `skip`, to the relative residuals tolv.  Returns the worst
  // final relative residual; iters_out = Arnoldi steps run (all cycles).
  double solve_op(const T *rhs, T *xsol, int &iters_out, const std::vector<char> *skip = nullptr, const std::vector<double> *tolv = nullptr) {
    // the tensorial path stays on the round-1 host-driven fp64 FGMRES: with no fp32 cycles to gain from, its adaptive
    // one-pass Gram-Schmidt is ~10 % faster than always-CGS2 device cycles (angled_64: 2 109 vs 2 322 ms)
    if (tensor_) return fgmres(rhs, xsol, iters_out, skip, tolv);
    auto tol_of = [&](int b) { return tolv ? (*tolv)[b] : opt_.inner_tol; };
    bool ir = !masked_ && opt_.inner_ir != 0;  // the fp32 twin of the operator keeps the PEC model: no masking
    std::vector<char> done(B, 0);
    if (skip) done = *skip;
    std::vector<unsigned char> hskip(B);
    std::vector<double> resrel(B, 1.0), bn2(B, 0.0), n2(B, 0.0), tolc(B), cres;
    std::vector<int> ju;
    CUDA_CHECK(cudaMemsetAsync(xsol, 0, vstride * sizeof(T), st_));
    const T *rcur = rhs;
    const int nch = gs_chunks(len);
    int total = 0, cyc = 0;
    bool verified = true;
    const dim3 egrd((unsigned)stream_blocks(len), B);
    while (true) {
      // ||r||^2 of the current residual (partials; reduced inside ir_begin)
      k_dots<T>(rcur, vstride, len, rcur, 1, gpart<T>(0), 0, nch);
      if (cyc > 0) {  // decide on the true fp64 residual
        sum_partials_kernel<T><<<(B + 63) / 64, 64, 0, st_>>>(gpart<T>(0), nch, pstride(), 0, n2_dev_, B);
        stats.launches++;
        CUDA_CHECK(cudaMemcpyAsync(n2.data(), n2_dev_, B * sizeof(double), cudaMemcpyDeviceToHost, st_));
        if (cyc == 1) CUDA_CHECK(cudaMemcpyAsync(bn2.data(), bn2_dev_, B * sizeof(double), cudaMemcpyDeviceToHost, st_));
        CUDA_CHECK(cudaStreamSynchronize(st_));
        stats.host_syncs++;
        bool all = true, stagnated = false;
        for (int b = 0; b < B; ++b) {
          if (done[b]) continue;
          const double r = bn2[b] > 0 ? std::sqrt(n2[b] / bn2[b]) : 0.0;
          if (ir && !(r < 0.5 * resrel[b])) stagnated = true;
          resrel[b] = r;
          if (r <= tol_of(b)) done[b] = 1; else all = false;
        }
        if (all || total >= opt_.gmres_maxit) break;
        if (stagnated || cyc >= 8) ir = false;  // finish in fp64
      }
      for (int b = 0; b < B; ++b) {
        hskip[b] = done[b] ? 1 : 0;
        const double want = 0.5 * tol_of(b) / std::max(resrel[b], 1e-300);
        tolc[b] = done[b] ? -1.0 : std::min(0.5, std::max(want, ir ? opt_.ir_floor : 0.0));
      }
      CUDA_CHECK(cudaMemcpyAsync(skip_dev_, hskip.data(), B, cudaMemcpyHostToDevice, st_));
      stats.launches++;
      double *n2cur = cyc == 0 ? bn2_dev_ : n2_dev_;  // ||r||^2 of this cycle (cycle 0: ||b||^2, kept for the relative residuals)
      int steps;
      if (ir) {
        P *Vp = reinterpret_cast<P *>(Vg_);
#define B200_IRB(E) ir_begin_kernel<T, P, E><<<egrd, 256, 0, st_>>>(rcur, Vp, lv[0].b, len, gpart<T>(0), nch, pstride(), 0, n2cur, skip_dev_)
        if (vec_ok<P>(len)) B200_IRB(PackTraits<P>::EPV); else B200_IRB(1);
#undef B200_IRB
        steps = fgmres_cycle<P>(tolc, cres, ju, true, opt_.gmres_maxit - total);
        int nvmax = 0;
        for (int b = 0; b < B; ++b) nvmax = std::max(nvmax, ju[b]);
        if (nvmax > 0) {
          stats.launches++;
          const P *Zp = reinterpret_cast<const P *>(Zg_), *yp = reinterpret_cast<const P *>(ydev_);
          if (vec_ok<P>(len)) ir_update_kernel<T, P, PackTraits<P>::EPV><<<egrd, 256, 0, st_>>>(Zp, vstride, len, yp, restart, nvmax, n2cur, xsol);
          else ir_update_kernel<T, P, 1><<<egrd, 256, 0, st_>>>(Zp, vstride, len, yp, restart, nvmax, n2cur, xsol);
        }
      } else {
#define B200_IRB(E) ir_begin_kernel<T, T, E><<<egrd, 256, 0, st_>>>(rcur, Vg_, nullptr, len, gpart<T>(0), nch, pstride(), 0, n2cur, skip_dev_)
        if (vec_ok<T>(len)) B200_IRB(PackTraits<T>::EPV); else B200_IRB(1);
#undef B200_IRB
        steps = fgmres_cycle<T>(tolc, cres, ju, false, opt_.gmres_maxit - total);
        int nvmax = 0;
        for (int b = 0; b < B; ++b) nvmax = std::max(nvmax, ju[b]);
        if (nvmax > 0) {
          stats.launches++;
          if (vec_ok<T>(len)) ir_update_kernel<T, T, PackTraits<T>::EPV><<<egrd, 256, 0, st_>>>(Zg_, vstride, len, ydev_, restart, nvmax, n2cur, xsol);
          else ir_update_kernel<T, T, 1><<<egrd, 256, 0, st_>>>(Zg_, vstride, len, ydev_, restart, nvmax, n2cur, xsol);
        }
      }
      total += steps;
      // estimates: res_cycle is relative to the residual the cycle started from
      bool all_est = true, trust = true;
      for (int b = 0; b < B; ++b) {
        if (done[b]) continue;
        const double est = cres[b] * resrel[b];
        if (est > tol_of(b)) all_est = false;
        if (ir && tolc[b] < opt_.ir_trust) trust = false;  // the fp32 estimate is good to ~1e-5 of the cycle's starting residual
        cres[b] = est;
      }
      ++cyc;
      if (all_est && trust) {  // fp64 cycles: the estimate is the true residual up to rounding; fp32: loose tolerances only
        for (int b = 0; b < B; ++b)
          if (!done[b]) resrel[b] = cres[b];
        verified = false;
        break;
      }
      if (total >= opt_.gmres_maxit && !ir) {
        for (int b = 0; b < B; ++b)
          if (!done[b]) resrel[b] = cres[b];
        break;
      }
      apply_true(MODE_RESID, xsol, rhs, rhs_);
      rcur = rhs_;
    }
    (void)verified;
    if (opt_.verbose >= 2) {
      double wr = 0.0;
      for (int b = 0; b < B; ++b)
        if (!skip || !(*skip)[b]) wr = std::max(wr, resrel[b]);
      fprintf(stderr, "[b200ms]   solve_op: cycles %d steps %d worst %.2e tol0 %.1e ir %d\n", cyc, total, wr, tol_of(0), (int)ir);
    }
    iters_out = total;
    stats.inner_iters += total;
    stats.inner_cycles += cyc;
    double worst = 0.0;
    for (int b = 0; b < B; ++b)
      if (!skip || !(*skip)[b]) worst = std::max(worst, resrel[b]);
    return worst;
  }

  // -- Krylov-Schur ---------------------------------------------------------------------------------
  struct EigResult {
    std::vector<cd> theta;      // [B][k] Ritz values of OP
    std::vector<int> nconv;     // [B]
    std::vector<double> resid;  // [B] max Ritz residual estimate relative to |theta|
    bool ok = true;
  };

  void init_start_vector(uint64_t seed) {
    // random start vector (the reference seeds numpy's PCG64 with 0, solver.py:846; converged eigenpairs do
    // not depend on it) with the PEC wall rows zeroed (solver.py:849-853)
    std::vector<T> hv(len);
    std::mt19937_64 rng(seed);
    std::uniform_real_distribution<double> U(0.0, 1.0);
    for (size_t e = 0; e < len; ++e) {
      cd v(U(rng), U(rng));
      hv[e] = from_cd<T>(v);
    }
    for (int c = 0; c < (int)(len / N); ++c)
      for (int i = 0; i < nx; ++i)
        for (int j = 0; j < ny; ++j)
          if ((nx > 1 && i == 0) || (ny > 1 && j == 0)) hv[c * N + (size_t)i * ny + j] = zero_of<T>();
    for (int b = 0; b < B; ++b)
      CUDA_CHECK(cudaMemcpyAsync(rhs_ + (size_t)b * len, hv.data(), len * sizeof(T), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaStreamSynchronize(st_));
    if (!tensor_) mask_E(rhs_, len);  // solver.py:507: vec_init = dnz * vec_init
    dots(rhs_, 1, rhs_, hbuf_, hstride(), 0, false);
    scale_inv_norm(rhs_, Vout_, hbuf_, hstride());
  }

  EigResult krylov_schur(bool real_arith) {
    EigResult out;
    out.theta.assign((size_t)B * k, cd(0, 0));
    out.nconv.assign(B, 0);
    out.resid.assign(B, 0.0);
    std::vector<CMat> Bm(B, CMat(m + 1, m));
    std::vector<char> done(B, 0);
    std::vector<CMat> Yfinal(B, CMat(m, k));
    std::vector<cd> h;
    std::vector<double> nrm;
    // inexact shift-invert: the inner tolerance is relaxed as the wanted Ritz pairs converge
    // (tol_j ~ eps / ||r_{j-1}||, Bouras & Fraysse / Simoncini); capped and with a safety factor
    std::vector<double> tolv(B, opt_.inner_tol);
    int nkeep = 0;
    const int keep_target = opt_.ks_keep > 0 ? std::min(m - 1, std::max(k + 1, opt_.ks_keep)) : std::min(m - 1, k + std::max(1, (m - k) / 2));
    for (int rst = 0; rst <= opt_.max_restarts; ++rst) {
      for (int j = nkeep; j < m; ++j) {
        T *vj = Vout_ + (size_t)j * vstride, *w = Vout_ + (size_t)(j + 1) * vstride;
        int its = 0;
        double worst = solve_op(vj, w, its, &done, &tolv);
        stats.op_applies++;
        if (!(worst <= 1e-3)) stats.inner_failures++;
        if (j + 2 < kGsMaxCoef) orthonormalise_dev(Vout_, j + 1, w, w, h, nrm, &done);
        else orthonormalise(Vout_, j + 1, w, w, h, nrm);
        for (int b = 0; b < B; ++b) {
          if (done[b]) continue;
          for (int i = 0; i <= j; ++i) Bm[b](i, j) += h[(size_t)b * (j + 1) + i];
          Bm[b](j + 1, j) = nrm[b];
        }
      }
      stats.restarts = rst;
      // Rayleigh-Ritz + restart matrices
      std::vector<T> qh((size_t)B * m * m, zero_of<T>());
      bool all_done = true;
      std::vector<int> newly;
      for (int b = 0; b < B; ++b) {
        if (done[b]) continue;
        CMat Tm(m, m), Q;
        for (int i = 0; i < m; ++i)
          for (int j = 0; j < m; ++j) Tm(i, j) = Bm[b](i, j);
        CMat Horig = Tm;
        if (!schur(Tm, Q)) {
          out.ok = false;
          done[b] = 1;
          continue;
        }
        // rank Ritz values by |theta| (ARPACK which='LM' on OP)
        std::vector<int> idx(m);
        for (int i = 0; i < m; ++i) idx[i] = i;
        std::stable_sort(idx.begin(), idx.end(), [&](int a, int c) { return std::abs(Tm(a, a)) > std::abs(Tm(c, c)); });
        std::vector<int> sel = select_closed(Tm, idx, keep_target, real_arith);
        // wanted k first (they are the first k of the ranking, inside sel)
        schur_reorder(Tm, Q, sel);
        const int keep = (int)sel.size();
        if (keep != keep_target) {
          out.ok = false;
          done[b] = 1;
          continue;
        }
        const cd hlast = Bm[b](m, m - 1);
        std::vector<cd> brow(keep);
        for (int i = 0; i < keep; ++i) brow[i] = hlast * Q(m - 1, i);
        CMat S = tri_eigvecs(Tm, keep);
        // Eigenvalue condition numbers in the projected problem.  ARPACK's test bounds the Ritz RESIDUAL; the error of a
        // Ritz value is that residual times kappa = 1/|y^H x|, which is ~1 for guided modes and in the hundreds for the
        // nearly defective pairs of PML modes (pml_none_128: two modes 1.2e-5 apart in n).  The contract is on n_eff, so the
        // residual is weighted by kappa (capped) before it is compared with eig_tol.
        std::vector<double> kappa = eig_condition(S, keep);
        // the k wanted = k largest |theta| among the kept
        std::vector<int> w(keep);
        for (int i = 0; i < keep; ++i) w[i] = i;
        std::stable_sort(w.begin(), w.end(), [&](int a, int c) { return std::abs(Tm(a, a)) > std::abs(Tm(c, c)); });
        int nconv = 0;
        double worst = 0.0;
        for (int q = 0; q < k; ++q) {
          const int i = w[q];
          cd acc = 0.0;
          for (int j = 0; j <= i; ++j) acc += brow[j] * S(j, i);
          double rel = std::abs(acc) / std::max(std::abs(Tm(i, i)), 1e-300);
          worst = std::max(worst, rel);
          if (rel * std::min(std::max(kappa[i], 1.0), opt_.kappa_cap) <= opt_.eig_tol) ++nconv;
          if (opt_.verbose >= 2 && b == 0)
            fprintf(stderr, "[b200ms]   restart %d ritz %d: theta (%.9e, %.9e) rel %.2e kappa %.2e tol_inner %.1e\n", rst, q, Tm(i, i).real(), Tm(i, i).imag(), rel,
                    kappa[i], tolv[b]);
        }
        out.nconv[b] = nconv;
        out.resid[b] = worst;
        // the first-order tensorial operator is far from normal (eigenvalue errors follow the residual linearly): its
        // shift-invert solves are not relaxed (measured on angled_phi_48: |dn| 4e-8 relaxed vs 1e-10 exact)
        // The relaxation bound of inexact Arnoldi carries the spectral gap of the wanted Ritz value as a factor (Simoncini
        // 2005): harmless for guided modes, fatal for a nearly degenerate non-normal pair (pml_none_128: two PML modes 3e-5
        // apart in theta; with the relaxed 1e-4 solves |dn| was 6e-5, with unrelaxed 1e-8 solves 4e-8).  A wanted Ritz value
        // closer than cluster_gap (relative) to any other Ritz value switches the relaxation off for that problem.
        double min_gap = 1e300;
        for (int q = 0; q < k; ++q) {
          const cd ti = Tm(w[q], w[q]);
          for (int j = 0; j < m; ++j)
            if (j != w[q]) min_gap = std::min(min_gap, std::abs(Tm(j, j) - ti) / std::max(std::abs(ti), 1e-300));
        }
        const bool clustered = min_gap < opt_.cluster_gap;
        if (clustered) tolv[b] = opt_.inner_tol;
        // Loosest tolerance: inner_relax_cap for real (lossless, no PML: near-normal, eigenvalue errors are second order in
        // the perturbation) problems; complex arithmetic (PML, bends, loss) is non-normal, the eigenvalue error is first
        // order in the inner residual (measured dn ~ 0.6 x cap on pml_none_128), so the cap is tied to the base tolerance.
        const double cap = real_arith ? opt_.inner_relax_cap : std::min(opt_.inner_relax_cap, opt_.inner_relax_complex * opt_.inner_tol);
        if (opt_.inner_relax > 0 && !tensor_ && !clustered)
          tolv[b] = std::min(cap, std::max(opt_.inner_tol, opt_.inner_relax * opt_.inner_tol / std::max(worst, 1e-300)));
        if (nconv == k || rst == opt_.max_restarts) {
          done[b] = 1;
          newly.push_back(b);
          for (int q = 0; q < k; ++q) {
            const int i = w[q];
            out.theta[(size_t)b * k + q] = Tm(i, i);
            if (real_arith && std::abs(Tm(i, i).imag()) > 1e-7 * std::abs(Tm(i, i))) out.ok = false;  // complex pair in real arithmetic
            for (int r = 0; r < m; ++r) {
              cd acc = 0.0;
              for (int j = 0; j <= i; ++j) acc += Q(r, j) * S(j, i);
              Yfinal[b](r, q) = acc;
            }
          }
          continue;
        }
        all_done = false;
        // restart matrices
        CMat Qk(m, keep);
        if (real_arith) {
          CMat Qc(m, keep);
          for (int r = 0; r < m; ++r)
            for (int i = 0; i < keep; ++i) Qc(r, i) = Q(r, i);
          int rank = real_basis(Qc, Qk);
          if (rank < keep) {
            out.ok = false;
            done[b] = 1;
            continue;
          }
        } else {
          for (int r = 0; r < m; ++r)
            for (int i = 0; i < keep; ++i) Qk(r, i) = Q(r, i);
        }
        CMat Bn(m + 1, m);
        if (real_arith) {
          // B_new = Qk^T H Qk (full), b_new = h * Qk[m-1, :]
          CMat HQ = matmul(Horig, Qk);
          for (int i = 0; i < keep; ++i)
            for (int j = 0; j < keep; ++j) {
              cd acc = 0.0;
              for (int r = 0; r < m; ++r) acc += std::conj(Qk(r, i)) * HQ(r, j);
              Bn(i, j) = acc;
            }
        } else {
          for (int i = 0; i < keep; ++i)
            for (int j = i; j < keep; ++j) Bn(i, j) = Tm(i, j);
        }
        for (int j = 0; j < keep; ++j) Bn(keep, j) = hlast * Qk(m - 1, j);
        Bm[b] = Bn;
        for (int r = 0; r < m; ++r)
          for (int i = 0; i < keep; ++i) qh[((size_t)b * m + r) * m + i] = from_cd<T>(Qk(r, i));
      }
      // Ritz vectors of the problems that converged in this cycle must be formed now: their basis is not
      // maintained once they are frozen
      if (!newly.empty()) extract_ritz(newly, Yfinal, real_arith);
      if (all_done) break;
      // V[:, :keep] <- V Q ; V[keep] <- V[m]      (Zg_ is free between inner solves: scratch)
      const int keep = keep_of(keep_target);
      CUDA_CHECK(cudaMemcpyAsync(qbuf_, qh.data(), qh.size() * sizeof(T), cudaMemcpyHostToDevice, st_));
      {
        dim3 grd(vec_blocks(), B);
        lincomb_kernel<T><<<grd, 256, (size_t)m * m * sizeof(T), st_>>>(Vout_, vstride, len, qbuf_, m, keep, m, Zg_, vstride);
      }
      CUDA_CHECK(cudaMemcpyAsync(Vout_, Zg_, (size_t)keep * vstride * sizeof(T), cudaMemcpyDeviceToDevice, st_));
      CUDA_CHECK(cudaMemcpyAsync(Vout_ + (size_t)keep * vstride, Vout_ + (size_t)m * vstride, vstride * sizeof(T),
                                 cudaMemcpyDeviceToDevice, st_));
      CUDA_CHECK(cudaStreamSynchronize(st_));
      nkeep = keep;
    }
    return out;
  }

  // Ritz vectors X = V Y (unit norm) for the listed problems -> ritz_ slots; real arithmetic: Y is made real
  // (phase fix) for real eigenvalues
  void extract_ritz(const std::vector<int> &which, const std::vector<CMat> &Yfinal, bool real_arith) {
    std::vector<T> yh((size_t)B * m * k, zero_of<T>());
    for (int b : which)
      for (int q = 0; q < k; ++q) {
        cd ph(1, 0);
        if (real_arith) {
          int best = 0;
          for (int r = 1; r < m; ++r)
            if (std::abs(Yfinal[b](r, q)) > std::abs(Yfinal[b](best, q))) best = r;
          cd v = Yfinal[b](best, q);
          if (std::abs(v) > 0) ph = std::conj(v) / std::abs(v);
        }
        double nn = 0.0;
        for (int r = 0; r < m; ++r) {
          cd v = Yfinal[b](r, q) * ph;
          if (real_arith) v = cd(v.real(), 0.0);
          nn += std::norm(v);
        }
        nn = nn > 0 ? 1.0 / std::sqrt(nn) : 0.0;
        for (int r = 0; r < m; ++r) {
          cd v = Yfinal[b](r, q) * ph;
          if (real_arith) v = cd(v.real(), 0.0);
          yh[((size_t)b * m + r) * k + q] = from_cd<T>(v * nn);
        }
      }
    CUDA_CHECK(cudaMemcpyAsync(qbuf_, yh.data(), yh.size() * sizeof(T), cudaMemcpyHostToDevice, st_));
    {
      dim3 grd(vec_blocks(), B);
      lincomb_kernel<T><<<grd, 256, (size_t)m * k * sizeof(T), st_>>>(Vout_, vstride, len, qbuf_, m, k, k, Zg_, vstride);
    }
    for (int b : which)
      for (int q = 0; q < k; ++q)
        CUDA_CHECK(cudaMemcpyAsync(ritz_ + (size_t)q * vstride + (size_t)b * len, Zg_ + (size_t)q * vstride + (size_t)b * len,
                                   len * sizeof(T), cudaMemcpyDeviceToDevice, st_));
    CUDA_CHECK(cudaStreamSynchronize(st_));
  }

  // -- relative mode solver (solver.py:750-776): Rayleigh-Ritz of A in the span of a supplied basis ----------
  // basis[b]: host [2][N][k] complex (mode fastest).  Returns eigenvalues of Q^H A Q, [B][k]; Ritz vectors -> ritz_.
  std::vector<cd> solve_relative(const std::vector<const cd *> &basis) {
    std::vector<T> hv(len);
    for (int q = 0; q < k; ++q)
      for (int b = 0; b < B; ++b) {
        for (size_t e = 0; e < len; ++e) hv[e] = from_cd<T>(basis[b][e * k + q]);
        CUDA_CHECK(cudaMemcpy(Vout_ + (size_t)q * vstride + (size_t)b * len, hv.data(), len * sizeof(T), cudaMemcpyHostToDevice));
      }
    std::vector<cd> h;
    std::vector<double> nrm;
    for (int q = 0; q < k; ++q) {  // orthonormal basis (the reference uses numpy's QR: same span)
      T *w = Vout_ + (size_t)q * vstride;
      if (q == 0) {
        dots(w, 1, w, hbuf_, hstride(), 0, false);
        scale_inv_norm(w, w, hbuf_, hstride());
      } else {
        orthonormalise(Vout_, q, w, w, h, nrm);
      }
    }
    std::vector<cd> zero(B, cd(0, 0));
    set_sigma(zero);
    std::vector<CMat> Hm(B, CMat(k, k));
    for (int j = 0; j < k; ++j) {
      T *wj = Zg_ + (size_t)j * vstride;
      apply_true(MODE_APPLY, Vout_ + (size_t)j * vstride, nullptr, wj);
      dots(Vout_, k, wj, hbuf_, hstride(), 0, false);
      fetch_h((size_t)B * hstride());
      for (int b = 0; b < B; ++b)
        for (int i = 0; i < k; ++i) Hm[b](i, j) = to_cd(hhost_[(size_t)b * hstride() + i]);
    }
    set_sigma(sig_host_);
    std::vector<cd> vals((size_t)B * k);
    std::vector<T> yh((size_t)B * k * k, zero_of<T>());
    for (int b = 0; b < B; ++b) {
      CMat Q;
      schur(Hm[b], Q);
      CMat S = tri_eigvecs(Hm[b], k);
      CMat Y = matmul(Q, S);
      for (int q = 0; q < k; ++q) {
        vals[(size_t)b * k + q] = Hm[b](q, q);
        for (int r = 0; r < k; ++r) yh[((size_t)b * k + r) * k + q] = from_cd<T>(Y(r, q));
      }
    }
    CUDA_CHECK(cudaMemcpyAsync(qbuf_, yh.data(), yh.size() * sizeof(T), cudaMemcpyHostToDevice, st_));
    {
      dim3 grd(vec_blocks(), B);
      lincomb_kernel<T><<<grd, 256, (size_t)k * k * sizeof(T), st_>>>(Vout_, vstride, len, qbuf_, k, k, k, ritz_, vstride);
    }
    CUDA_CHECK(cudaStreamSynchronize(st_));
    return vals;
  }

  // true eigen-residuals ||A x - lambda x|| / (|lambda| ||x||) for Ritz vector slot q, per problem
  std::vector<double> eigen_residuals(int q, const std::vector<cd> &lambda) {
    set_sigma(lambda);
    T *x = ritz_ + (size_t)q * vstride;
    apply_true(MODE_APPLY, x, nullptr, rhs_);
    dots(rhs_, 1, rhs_, hbuf_, hstride(), 0, false);
    dots(x, 1, x, hbuf_, hstride(), 1, false);
    fetch_h((size_t)B * hstride());
    std::vector<double> r(B);
    for (int b = 0; b < B; ++b) {
      double rn = std::sqrt(std::max(0.0, to_cd(hhost_[(size_t)b * hstride()]).real()));
      double xn = std::sqrt(std::max(0.0, to_cd(hhost_[(size_t)b * hstride() + 1]).real()));
      r[b] = rn / std::max(1e-300, xn * std::abs(lambda[b]));
    }
    set_sigma(sig_host_);
    return r;
  }

  // reorder Ritz vector slots: ritz_[new q] = old slot order[b][q] is per problem -> done through lincomb
  // with permutation matrices; here slots are shared by the batch so we permute per problem on the fly
  // in the epilogue via `perm`.
  void epilogue(const std::vector<cd> &ncomplex_sorted, const std::vector<int> &perm, const std::vector<const ProblemSetup *> &ps,
                cplx *host_dst_per_problem[], bool want_fields) {
    // permute Ritz vectors so that slot q holds mode q (descending n_eff) for every problem
    std::vector<T> ph((size_t)B * k * k, zero_of<T>());
    for (int b = 0; b < B; ++b)
      for (int q = 0; q < k; ++q) ph[((size_t)b * k + perm[(size_t)b * k + q]) * k + q] = from_real<T>(1.0);
    CUDA_CHECK(cudaMemcpyAsync(qbuf_, ph.data(), ph.size() * sizeof(T), cudaMemcpyHostToDevice, st_));
    {
      dim3 grd(vec_blocks(), B);
      lincomb_kernel<T><<<grd, 256, (size_t)k * k * sizeof(T), st_>>>(ritz_, vstride, len, qbuf_, k, k, k, Zg_, vstride);
    }
    if (!want_fields) {
      CUDA_CHECK(cudaStreamSynchronize(st_));
      return;
    }
    std::vector<cplx> nh((size_t)B * k);
    for (size_t i = 0; i < nh.size(); ++i) nh[i] = mk(ncomplex_sorted[i].real(), ncomplex_sorted[i].imag());
    CUDA_CHECK(cudaMemcpyAsync(ncomplex_, nh.data(), nh.size() * sizeof(cplx), cudaMemcpyHostToDevice, st_));
    const ProblemSetup &p0 = *ps[0];
    int jz_len = 0;
    if (p0.jz_axis >= 0) {
      jz_len = (int)p0.jz_e.size();
      std::vector<double> je((size_t)B * jz_len), jh((size_t)B * jz_len);
      for (int b = 0; b < B; ++b)
        for (int i = 0; i < jz_len; ++i) {
          je[(size_t)b * jz_len + i] = ps[b]->jz_e[i];
          jh[(size_t)b * jz_len + i] = ps[b]->jz_h[i];
        }
      CUDA_CHECK(cudaMemcpyAsync(jz_, je.data(), je.size() * sizeof(double), cudaMemcpyHostToDevice, st_));
      CUDA_CHECK(cudaMemcpyAsync(jz_ + (size_t)B * jz_len, jh.data(), jh.size() * sizeof(double), cudaMemcpyHostToDevice, st_));
      CUDA_CHECK(cudaStreamSynchronize(st_));
    }
    if constexpr (std::is_same<T, cplx>::value) {
      if (tensor_) {
        TensorEpilogueArgs<C> t;
        t.nx = nx; t.ny = ny; t.num_modes = k; t.vec = Zg_; t.vstride = vstride;
        t.ft = ft_; t.ft_bstride = shared_fields ? 0 : 18 * N; t.cx = lv[0].cx_true; t.cy = lv[0].cy_true;
        t.jz_e = jz_; t.jz_h = jz_ + (size_t)B * jz_len; t.jz_axis = p0.jz_axis; t.jz_len = jz_len;
        t.jac_a = p0.jac_a; t.jac_b = p0.jac_b;
        t.conj_flip = (!p0.eps_complex && p0.direction < 0) ? 1 : 0;
        t.h_scale = 1.0 / eta0(); t.out = fields_out_; t.single = single_out_ ? 1 : 0;
        dim3 blk(64, 4), grd((ny + 63) / 64, (nx + 3) / 4, B * k);
        tensor_epilogue_kernel<C><<<grd, blk, 0, st_>>>(t);
        CUDA_CHECK(cudaGetLastError());
        return;
      }
    }
    EpilogueArgs<T, C> a;
    a.nx = nx; a.ny = ny; a.num_modes = k; a.vec = Zg_; a.vstride = vstride;
    a.fields = lv[0].fields_true; a.field_bstride = lv[0].fbstride; a.cx = lv[0].cx_true; a.cy = lv[0].cy_true;
    a.ncomplex = ncomplex_; a.jz_e = jz_; a.jz_h = jz_ + (size_t)B * jz_len; a.jz_axis = p0.jz_axis; a.jz_len = jz_len;
    a.direction = p0.direction; a.h_scale = 1.0 / eta0(); a.out = fields_out_; a.single = single_out_ ? 1 : 0;
    dim3 blk(64, 4), grd((ny + 63) / 64, (nx + 3) / 4, B * k);
    if (has_mu) epilogue_kernel<T, C, true><<<grd, blk, 0, st_>>>(a);
    else epilogue_kernel<T, C, false><<<grd, blk, 0, st_>>>(a);
    CUDA_CHECK(cudaGetLastError());
  }
  // dn/deps of every mode of the problems with dst[b] != nullptr (device buffers, [M][3][nx][ny] complex128), from the Ritz
  // vectors epilogue() left in mode order; ncomplex_sorted as passed to epilogue() (csrc/sensitivity.cuh)
  void sensitivity(const std::vector<cd> &ncomplex_sorted, const std::vector<const ProblemSetup *> &ps, const std::vector<cplx *> &dst) {
    sensitivity_upload(ncomplex_sorted, ps, dst);
    sensitivity_launch();
    CUDA_CHECK(cudaStreamSynchronize(st_));
  }
  void sensitivity_upload(const std::vector<cd> &ncomplex_sorted, const std::vector<const ProblemSetup *> &ps, const std::vector<cplx *> &dst) {
    if (!sens_part_) {
      sens_part_ = arena_.get<cplx>((size_t)B * k * kSensChunks);
      sens_len_ = arena_.get<cplx>((size_t)B * 2 * (nx + ny));
      sens_out_ = arena_.get<cplx *>((size_t)B);
    }
    std::vector<cplx> nh((size_t)B * k), lens((size_t)B * 2 * (nx + ny));
    for (size_t i = 0; i < nh.size(); ++i) nh[i] = mk(ncomplex_sorted[i].real(), ncomplex_sorted[i].imag());
    for (int b = 0; b < B; ++b)
      for (int a = 0; a < 2; ++a) {
        const Axis &A = ps[b]->ax[a];
        cplx *l = lens.data() + (a == 0 ? (size_t)b * 2 * nx : (size_t)B * 2 * nx + (size_t)b * 2 * ny);
        for (int i = 0; i < A.n; ++i) {
          l[i] = mk(A.lf[i].real(), A.lf[i].imag());
          l[A.n + i] = mk(A.lb[i].real(), A.lb[i].imag());
        }
        if (A.pmc && A.n > 1) l[A.n] = 0.5 * l[A.n];  // the PMC row of Db is 2 / lb[0]: half a dual cell
      }
    CUDA_CHECK(cudaMemcpyAsync(ncomplex_, nh.data(), nh.size() * sizeof(cplx), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaMemcpyAsync(sens_len_, lens.data(), lens.size() * sizeof(cplx), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaMemcpyAsync(sens_out_, dst.data(), (size_t)B * sizeof(cplx *), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaStreamSynchronize(st_));  // the host vectors above must outlive the copies
  }
  // the two gradient kernels on the vectors in gmres_z() (epilogue() leaves the Ritz vectors there in mode order)
  void sensitivity_launch() {
    SensArgs<T, C> a;
    a.nx = nx; a.ny = ny; a.num_modes = k; a.vec = Zg_; a.vstride = vstride;
    a.fields = lv[0].fields_true; a.field_bstride = lv[0].fbstride; a.has_mu = has_mu ? 1 : 0;
    a.cx = lv[0].cx_true; a.cy = lv[0].cy_true; a.len_x = sens_len_; a.len_y = sens_len_ + (size_t)B * 2 * nx;
    a.ncomplex = ncomplex_; a.out = sens_out_;
    sens_scan_kernel<T, C><<<dim3(kSensChunks, B * k), 256, 0, st_>>>(a, sens_part_);
    CUDA_CHECK(cudaGetLastError());
    const unsigned nblk = (unsigned)std::min<size_t>((N + 255) / 256, 1024);
    sens_write_kernel<T, C><<<dim3(nblk, B * k), 256, 0, st_>>>(a, sens_part_);
    CUDA_CHECK(cudaGetLastError());
    stats.launches += 2;
  }
  T *scratch_vec(int i) { return i == 0 ? xsol_ : rhs_; }
  T *basis0() { return Vout_; }
  T *gmres_z() { return Zg_; }
  T *gmres_v() { return Vg_; }
  void set_output(cplx *buf) { fields_out_ = buf; }  // device buffer for the packed fields (owned by the caller)
  size_t output_bytes_per_problem() const { return (size_t)6 * N * k * (single_out_ ? sizeof(cplxf) : sizeof(cplx)); }
  T *hessenberg() { return Hd_; }
  T *ritz_ptr() { return ritz_; }

 private:
  static void transfer_sizes(const AxisTransfer &t, size_t &ints, size_t &dbls) {
    for (const Transfer1D *q : {&t.node, &t.edge}) {
      ints += q->p_i0.size() * 2 + q->r_ptr.size() + q->r_idx.size() + 256;
      dbls += q->p_w0.size() * 2 + q->r_w.size() + 256;
      dbls += q->p_w0.size() + 4 * q->r_ptr.size() + 192;  // fp32 prolongation weights (2 x n floats) and the packed restriction lists (32 B per coarse index)
    }
  }
  template <typename U>
  const U *up(const std::vector<U> &v) {
    U *d = arena_.get<U>(std::max<size_t>(v.size(), 1));
    if (!v.empty()) CUDA_CHECK(cudaMemcpyAsync(d, v.data(), v.size() * sizeof(U), cudaMemcpyHostToDevice, st_));
    CUDA_CHECK(cudaStreamSynchronize(st_));
    return d;
  }
  void upload_transfer(const Transfer1D &h, Transfer1DDev &d) {
    d.p_i0 = up(h.p_i0); d.p_i1 = up(h.p_i1); d.p_w0 = up(h.p_w0); d.p_w1 = up(h.p_w1);
    d.r_ptr = up(h.r_ptr); d.r_idx = up(h.r_idx); d.r_w = up(h.r_w);
    std::vector<float> w0f(h.p_w0.begin(), h.p_w0.end()), w1f(h.p_w1.begin(), h.p_w1.end());
    d.p_w0f = up(w0f); d.p_w1f = up(w1f);
    // packed restriction lists (csrc/kernels.cuh restrict4_kernel): possible when no coarse index gathers more than four fine ones
    const int nc = (int)h.r_ptr.size() - 1;
    bool ok = nc > 0;
    for (int I = 0; I < nc && ok; ++I) ok = h.r_ptr[I + 1] - h.r_ptr[I] <= 4;
    d.r4 = nullptr;
    if (ok) {
      std::vector<RList4> packed(nc);
      for (int I = 0; I < nc; ++I) {
        const int k0 = h.r_ptr[I], cnt = h.r_ptr[I + 1] - k0;
        for (int q = 0; q < 4; ++q) {
          packed[I].idx[q] = cnt > 0 ? h.r_idx[k0 + std::min(q, cnt - 1)] : 0;
          packed[I].w[q] = q < cnt ? (float)h.r_w[k0 + q] : 0.0f;
        }
      }
      d.r4 = up(packed);
    }
  }
  int keep_of(int keep_target) const { return keep_target; }

  // choose `count` Ritz values (indices into diag(T)) in ranking order such that, in real arithmetic,
  // the set is closed under complex conjugation
  static std::vector<int> select_closed(const CMat &Tm, const std::vector<int> &ranked, int count, bool real_arith) {
    std::vector<int> sel;
    if (!real_arith) {
      sel.assign(ranked.begin(), ranked.begin() + count);
      return sel;
    }
    const int mtot = (int)ranked.size();
    std::vector<char> used(mtot, 0);
    auto is_cplx = [&](int i) { return std::abs(Tm(i, i).imag()) > 1e-10 * std::max(1e-300, std::abs(Tm(i, i))); };
    auto partner = [&](int i) {
      int best = -1;
      double bd = 1e300;
      for (int j = 0; j < mtot; ++j) {
        if (j == i || used[j]) continue;
        double d = std::abs(Tm(j, j) - std::conj(Tm(i, i)));
        if (d < bd) { bd = d; best = j; }
      }
      return best;
    };
    for (int r = 0; r < mtot && (int)sel.size() < count; ++r) {
      int i = ranked[r];
      if (used[i]) continue;
      if (!is_cplx(i)) {
        used[i] = 1;
        sel.push_back(i);
      } else if ((int)sel.size() + 2 <= count) {
        used[i] = 1;
        int p = partner(i);
        sel.push_back(i);
        if (p >= 0) { used[p] = 1; sel.push_back(p); }
      }
    }
    // top up with the best remaining real Ritz values if pairs were skipped
    for (int r = 0; r < mtot && (int)sel.size() < count; ++r) {
      int i = ranked[r];
      if (!used[i] && !is_cplx(i)) { used[i] = 1; sel.push_back(i); }
    }
    for (int r = 0; r < mtot && (int)sel.size() < count; ++r) {
      int i = ranked[r];
      if (!used[i]) { used[i] = 1; sel.push_back(i); }
    }
    return sel;
  }

  Arena &arena_;
  cudaStream_t st_;
  b200ms_options opt_;
  HierarchyPlan plan_;
  int mask_x_ = 0, mask_y_ = 0;
  T *Vout_ = nullptr, *Vg_ = nullptr, *Zg_ = nullptr, *xsol_ = nullptr, *rhs_ = nullptr, *ritz_ = nullptr;
  T *partial_ = nullptr, *hbuf_ = nullptr, *qbuf_ = nullptr, *sigma_ = nullptr;
  P *sigma_p_ = nullptr, *pre_a_ = nullptr, *pre_b_ = nullptr;
  C *ft_ = nullptr;
  T *tb_[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cplx *tcoef_ = nullptr;
  std::vector<cd> sig_mg_host_;
  bool dinv_ready_ = false;
  std::map<long, int> m2_resident_;  // pair-marching kernel: resident CTAs on the device per (mode, TMA or registers, CTA width)
  cudaGraphExec_t graph_exec_ = nullptr;
  P *graph_result_ = nullptr;
  long graph_nodes_ = 0, graph_fine_applies_ = 0;
  cplx *ncomplex_ = nullptr, *fields_out_ = nullptr;
  double *jz_ = nullptr;
  bool coarse_krylov_ = false;
  int kc_ = 16;
  P *cV_ = nullptr, *cZ_ = nullptr, *cH_ = nullptr, *cH2_ = nullptr, *cy_ = nullptr, *cbeta_ = nullptr, *cone_ = nullptr;
  std::vector<T> hhost_;
  std::vector<cd> sig_host_;
  // round-2 inner solver state
  cplx *sens_part_ = nullptr, *sens_len_ = nullptr;
  cplx **sens_out_ = nullptr;
  P *cx_true_p_ = nullptr, *cy_true_p_ = nullptr;  // reference-operator difference coefficients in the multigrid precision
  T *Hd_ = nullptr, *ydev_ = nullptr, *gpart_ = nullptr;
  cplx *lsq_work_ = nullptr;
  double *tol_dev_ = nullptr, *res_dev_ = nullptr, *n2_dev_ = nullptr, *bn2_dev_ = nullptr;
  int *jused_dev_ = nullptr;
  unsigned char *skip_dev_ = nullptr;
  int fused_l0_ = -1;      // first level of the fused multigrid tail (-1: none)
  size_t fused_smem_ = 0;
  double rho_ = 0.2;  // convergence factor per Arnoldi step seen in the last cycle (plans the next one)
};

}  // namespace b200ms
