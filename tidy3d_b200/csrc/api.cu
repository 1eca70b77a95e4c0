// C ABI of libb200ms.so (see include/b200ms.h for the reference interfaces each entry point replaces).
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <future>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only; a no-op unless a profiler (ncu / nsys) injects itself

#include "../../include/b200ms.h"
#include "post.cuh"
#include "solver.cuh"

using namespace b200ms;

// Named ranges for profilers (SURVEY 5: the phases of one b200ms_solve_batch call on the timeline, one range stack per thread:
// the upload and delivery helpers run on their own threads).  `ncu --nvtx --nvtx-include "b200ms:eigen-iteration/"` restricts a
// capture to the kernels of one phase.
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange &) = delete;
  NvtxRange &operator=(const NvtxRange &) = delete;
};

// grow-only device buffer
struct DevBuf {
  unsigned char *p = nullptr;
  size_t cap = 0;
  void reserve(size_t n) {
    if (n <= cap) return;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    CUDA_CHECK(cudaMalloc(&p, n));
    cap = n;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct b200ms_handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t io_stream = nullptr;  // uploads of raw media (+ scan kernels)
  cudaStream_t dl_stream = nullptr;  // delivery of packed fields
  Arena arena;
  DevBuf raw[2];      // raw eps/mu of a window of problems (+ bend factors), double-buffered
  DevBuf out[2];      // packed fields of a window, double-buffered
  DevBuf scan;        // reduction scratch + per-medium results of prepare_window
  DevBuf refs;        // MediumRef array of the batch being built
  DevBuf post;        // interpolation tables / partials / results of the on-device post-processing
  b200ms_options opt;
  std::string err;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  unsigned char *flush_buf = nullptr;
  size_t flush_bytes = 0;
  b200ms_stats stats;
};

extern "C" int b200ms_version(void) { return B200MS_VERSION; }

extern "C" void b200ms_default_options(b200ms_options *o) {
  o->eig_tol = kFpEps;   // the reference's ARPACK tolerance (TOL_EIGS = fp_eps, solver.py:20)
  o->inner_tol = 1e-8;
  o->ncv = 0;
  o->max_restarts = 500;  // scipy: maxiter = 10 n restarts; the PML-cluster case needs ~80-110
  o->gmres_restart = 40;
  o->gmres_maxit = 400;
  o->mg_nu = 2;
  o->mg_min_size = 12;
  o->mg_coarse_iters = 16;
  o->max_batch = 64;
  o->mg_omega = 0.8;
  o->mg_ppw = 4.0;
  o->verbose = 0;
  o->mg_pml_phase = 0.7853981633974483;
  o->mg_cycles = 1;
  o->use_graph = 1;
  o->mg_nu_growth = 0;
  o->gmres_cgs2 = 2;
  o->inner_relax = 1.0;
  o->inner_relax_cap = 1e-4;
  o->inner_ir = 1;
  o->ir_floor = 1e-4;
  o->ir_trust = 3e-5;
  o->inner_relax_complex = 50.0;
  o->cluster_gap = 1e-3;
  o->mg_fuse_first = 1;
  o->ks_keep = 0;
  o->mg_fused_tail = 1;
  o->kappa_cap = 1e4;
  o->outer_dgks = 1;
  o->stencil_pair = 1;
  o->stencil_pair_rows = 0;
  o->transfer_vec = 3;
  o->tensor_mg_cycles = 3;
}

extern "C" int b200ms_create(int device, b200ms_handle **out) {
  if (!out) return B200MS_ERR_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return B200MS_ERR_CUDA;  // no CPU fallback
  if (device < 0) {
    if (cudaGetDevice(&device) != cudaSuccess) return B200MS_ERR_CUDA;
  }
  if (device >= count || cudaSetDevice(device) != cudaSuccess) return B200MS_ERR_CUDA;
  auto *h = new b200ms_handle();
  h->device = device;
  b200ms_default_options(&h->opt);
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->io_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->dl_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess) {
    delete h;
    return B200MS_ERR_CUDA;
  }
  *out = h;
  return B200MS_OK;
}

extern "C" int b200ms_destroy(b200ms_handle *h) {
  if (!h) return B200MS_OK;
  cudaSetDevice(h->device);
  h->arena.release();
  for (int q = 0; q < 2; ++q) {
    h->raw[q].release();
    h->out[q].release();
  }
  h->scan.release();
  h->refs.release();
  h->post.release();
  if (h->io_stream) cudaStreamDestroy(h->io_stream);
  if (h->dl_stream) cudaStreamDestroy(h->dl_stream);
  if (h->flush_buf) cudaFree(h->flush_buf);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return B200MS_OK;
}

extern "C" void *b200ms_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
extern "C" void b200ms_host_free(void *ptr) {
  if (ptr) cudaFreeHost(ptr);
}

extern "C" int b200ms_set_options(b200ms_handle *h, const b200ms_options *opt) {
  if (!h || !opt) return B200MS_ERR_ARG;
  h->opt = *opt;
  return B200MS_OK;
}

extern "C" const char *b200ms_last_error(b200ms_handle *h) { return h ? h->err.c_str() : "null handle"; }

extern "C" int b200ms_get_stats(b200ms_handle *h, b200ms_stats *out) {
  if (!h || !out) return B200MS_ERR_ARG;
  *out = h->stats;
  return B200MS_OK;
}

namespace {

struct GroupKey {
  int nx, ny, k, kind, has_mu, sx, sy, jz_axis, dir, rel, tens, prec, masked;
  double theta, phi;
  bool operator<(const GroupKey &o) const {
    return std::tie(nx, ny, k, kind, has_mu, sx, sy, jz_axis, dir, rel, tens, prec, masked, theta, phi) <
           std::tie(o.nx, o.ny, o.k, o.kind, o.has_mu, o.sx, o.sy, o.jz_axis, o.dir, o.rel, o.tens, o.prec, o.masked, o.theta, o.phi);
  }
};
struct MediumKey {
  const double *eps, *mu, *cx, *cy;
  int nx, ny, p0, p1, bend_axis, incidence;
  double bend_radius, theta, phi;
  bool operator==(const MediumKey &o) const {
    auto same = [](double a, double b) { return (std::isnan(a) && std::isnan(b)) || a == b; };
    return eps == o.eps && mu == o.mu && cx == o.cx && cy == o.cy && nx == o.nx && ny == o.ny && p0 == o.p0 && p1 == o.p1 &&
           bend_axis == o.bend_axis && incidence == o.incidence && same(bend_radius, o.bend_radius) && theta == o.theta && phi == o.phi;
  }
};
// kind: 0 real, 1 complex vectors + real fields, 2 all complex
int kind_of(const ProblemSetup &s) { return !s.is_complex ? 0 : (s.coef_complex ? 2 : 1); }

inline size_t align256(size_t n) { return (n + 255) & ~size_t(255); }

// A window of consecutive problems whose raw media are resident on the device: set-up stages A-C of host_setup.hpp with
// the per-cell work (reductions) done by medium_scan_kernel.
struct Window {
  int i0 = 0, i1 = 0;
  std::vector<ProblemSetup> setups;  // one per problem of the window
  std::vector<MediumRef> refs;       // one per problem (device pointers into the raw buffer)
  std::vector<int> slot;             // medium slot of each problem (problems sharing eps/mu/geometry share a slot)
  size_t h2d_bytes = 0;
};

// bytes of the raw buffer one geometric cross-section takes on the device (every array in its own 256-byte aligned sub-buffer)
size_t section_device_bytes(const b200ms_section &sec, int nx, int ny) {
  const int nv = (sec.poly_start && sec.nrect > 0) ? sec.poly_start[sec.nrect] : 0;
  size_t b = align256((size_t)sec.nrect * 4 * sizeof(double)) + align256((size_t)sec.nrect * sizeof(int)) + align256((size_t)sec.nmedia * 9 * sizeof(cplx)) +
             align256((size_t)(nx + 1) * sizeof(double)) + align256((size_t)(ny + 1) * sizeof(double));
  if (sec.shape) b += align256((size_t)sec.nrect * sizeof(int));
  if (nv > 0) b += align256((size_t)(sec.nrect + 1) * sizeof(int)) + align256((size_t)nv * 2 * sizeof(double));
  if (sec.site_medium) b += align256((size_t)3 * nx * ny * sizeof(unsigned short));
  return b;
}

void prepare_window(b200ms_handle *h, const b200ms_problem *prob, int i0, int i1, DevBuf &raw, cudaStream_t st, Window &W) {
  const int n = i1 - i0;
  W.i0 = i0;
  W.i1 = i1;
  W.setups.assign(n, ProblemSetup());
  W.refs.assign(n, MediumRef());
  W.slot.assign(n, -1);
  W.h2d_bytes = 0;
  std::vector<std::pair<MediumKey, int>> seen;  // key -> first problem with that medium
  std::vector<size_t> off_eps(n, 0), off_mu(n, 0), off_d(n, 0), off_sec(n, 0);
  size_t total = 0;
  for (int q = 0; q < n; ++q) {
    const b200ms_problem &p = prob[i0 + q];
    ProblemSetup &s = W.setups[q];
    setup_geometry(p, s);
    if (s.status != B200MS_OK) continue;
    MediumKey mk{p.eps ? p.eps : reinterpret_cast<const double *>(p.section), p.mu, p.coords_x, p.coords_y, p.nx, p.ny, p.num_pml[0], p.num_pml[1], p.bend_axis, p.incidence ? 1 : 0,
                 p.bend_radius, p.angle_theta, p.angle_phi};
    auto it = std::find_if(seen.begin(), seen.end(), [&](const std::pair<MediumKey, int> &e) { return e.first == mk; });
    if (it != seen.end()) {
      W.slot[q] = W.slot[it->second];
      continue;
    }
    W.slot[q] = (int)seen.size();
    seen.push_back({mk, q});
    const size_t N = (size_t)p.nx * p.ny;
    off_eps[q] = total;
    total += align256(9 * N * sizeof(cplx));
    if (p.mu) {
      off_mu[q] = total;
      total += align256(9 * N * sizeof(cplx));
    }
    if (s.jz_axis >= 0) {
      off_d[q] = total;
      total += align256(2 * s.jz_e.size() * sizeof(double));
    }
    if (!p.eps) {  // geometric cross-section: shapes, medium ids, eps table, cell boundaries (+ shape kinds, polygon vertices, site map)
      off_sec[q] = total;
      total += section_device_bytes(*p.section, p.nx, p.ny);
    }
  }
  const int nslot = (int)seen.size();
  raw.reserve(std::max<size_t>(total, 256));
  // scan scratch: [kScanBlocks][kScanSlots] partials, then nslot result rows
  h->scan.reserve(align256((size_t)kScanBlocks * kScanSlots * sizeof(double)) + align256((size_t)std::max(nslot, 1) * kScanSlots * sizeof(double)) +
                  4096);
  double *d_partial = reinterpret_cast<double *>(h->scan.p);
  double *d_res = reinterpret_cast<double *>(h->scan.p + align256((size_t)kScanBlocks * kScanSlots * sizeof(double)));
  std::vector<MediumRef> slot_ref(nslot);
  for (auto &e : seen) {
    const int q = e.second;
    const b200ms_problem &p = prob[i0 + q];
    const ProblemSetup &s = W.setups[q];
    const size_t N = (size_t)p.nx * p.ny;
    MediumRef r;
    r.eps = reinterpret_cast<const cplx *>(raw.p + off_eps[q]);
    if (p.eps) {
      CUDA_CHECK(cudaMemcpyAsync(raw.p + off_eps[q], p.eps, 9 * N * sizeof(cplx), cudaMemcpyDefault, st));
      W.h2d_bytes += 9 * N * sizeof(cplx);
    } else {  // rasterise the geometric cross-section on the device (f-2: replaces nine epsilon_on_grid calls + a 9N upload)
      const b200ms_section &sec = *p.section;
      unsigned char *cur = raw.p + off_sec[q];
      auto put = [&](const void *src, size_t bytes) -> unsigned char * {  // 256-byte aligned sub-buffer, filled from host memory
        unsigned char *dst = cur;
        if (bytes) CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        cur += align256(bytes);
        W.h2d_bytes += bytes;
        return dst;
      };
      const int nv = (sec.poly_start && sec.nrect > 0) ? sec.poly_start[sec.nrect] : 0;
      double *d_rects = reinterpret_cast<double *>(put(sec.rects, (size_t)sec.nrect * 4 * sizeof(double)));
      int *d_med = reinterpret_cast<int *>(put(sec.medium, (size_t)sec.nrect * sizeof(int)));
      cplx *d_tab = reinterpret_cast<cplx *>(put(sec.eps_table, (size_t)sec.nmedia * 9 * sizeof(cplx)));
      double *d_x = reinterpret_cast<double *>(put(p.coords_x, (size_t)(p.nx + 1) * sizeof(double)));
      double *d_y = reinterpret_cast<double *>(put(p.coords_y, (size_t)(p.ny + 1) * sizeof(double)));
      const int *d_shape = sec.shape ? reinterpret_cast<const int *>(put(sec.shape, (size_t)sec.nrect * sizeof(int))) : nullptr;
      const int *d_pstart = nv > 0 ? reinterpret_cast<const int *>(put(sec.poly_start, (size_t)(sec.nrect + 1) * sizeof(int))) : nullptr;
      const double *d_pxy = nv > 0 ? reinterpret_cast<const double *>(put(sec.poly_xy, (size_t)nv * 2 * sizeof(double))) : nullptr;
      const unsigned short *d_site = sec.site_medium ? reinterpret_cast<const unsigned short *>(put(sec.site_medium, 3 * N * sizeof(unsigned short))) : nullptr;
      SectionDev sd{sec.nrect, d_rects, d_med, d_tab, d_x, d_y, sec.nmedia, d_shape, d_pstart, d_pxy, d_site};
      section_raster_kernel<<<(unsigned)std::min<size_t>((N + 255) / 256, 2048), 256, 0, st>>>(sd, p.nx, p.ny, const_cast<cplx *>(r.eps));
    }
    r.mu = nullptr;
    if (p.mu) {
      r.mu = reinterpret_cast<const cplx *>(raw.p + off_mu[q]);
      CUDA_CHECK(cudaMemcpyAsync(raw.p + off_mu[q], p.mu, 9 * N * sizeof(cplx), cudaMemcpyDefault, st));
      W.h2d_bytes += 9 * N * sizeof(cplx);
    }
    const double *d_de = nullptr, *d_dh = nullptr;
    if (s.jz_axis >= 0) {
      const size_t nn = s.jz_e.size();
      double *dd = reinterpret_cast<double *>(raw.p + off_d[q]);
      CUDA_CHECK(cudaMemcpyAsync(dd, s.jz_e.data(), nn * sizeof(double), cudaMemcpyHostToDevice, st));
      CUDA_CHECK(cudaMemcpyAsync(dd + nn, s.jz_h.data(), nn * sizeof(double), cudaMemcpyHostToDevice, st));
      d_de = dd;
      d_dh = dd + nn;
    }
    r.p = medium_params(s, p, d_de, d_dh);
    const int nb = (int)std::min<size_t>(kScanBlocks, (N + 255) / 256);
    medium_scan_kernel<<<nb, 256, 0, st>>>(r.eps, r.mu, r.p, d_partial);
    medium_scan_final_kernel<<<1, 32, 0, st>>>(d_partial, nb, d_res + (size_t)W.slot[q] * kScanSlots);
    slot_ref[W.slot[q]] = r;
  }
  std::vector<MediumScan> scans(std::max(nslot, 1));
  if (nslot > 0) CUDA_CHECK(cudaMemcpyAsync(scans.data(), d_res, (size_t)nslot * kScanSlots * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_CHECK(cudaStreamSynchronize(st));
  CUDA_CHECK(cudaGetLastError());
  for (int q = 0; q < n; ++q) {
    if (W.setups[q].status != B200MS_OK) continue;
    W.refs[q] = slot_ref[W.slot[q]];
    W.setups[q].medium = W.slot[q];
    finish_setup(prob[i0 + q], W.setups[q], scans[W.slot[q]]);
  }
}

// device array of MediumRef for a batch (fB entries)
const MediumRef *upload_refs(b200ms_handle *h, const std::vector<MediumRef> &refs, cudaStream_t st) {
  h->refs.reserve(align256(refs.size() * sizeof(MediumRef)) + 4096);
  MediumRef *d = reinterpret_cast<MediumRef *>(h->refs.p);
  CUDA_CHECK(cudaMemcpyAsync(d, refs.data(), refs.size() * sizeof(MediumRef), cudaMemcpyHostToDevice, st));
  return d;
}


// ---- on-device post-processing (csrc/post.cuh) ----------------------------------------------------------------------
// 1-D tables of one axis: colocation points = interior cell boundaries, plus the symmetry plane itself when the min wall is one
// (mode_solver.py:494-502), linear interpolation from the centre / boundary Yee sites of the SYMMETRY-EXPANDED data
// (mode_solver.py:504-507 interpolates mode_solver_data.symmetry_expanded; monitor_data.py:237-282 mirrors the half domain
// with the factor sym_val * symmetry_eigenvalue), trapezoid weights (monitor_data.py:425-467).
struct HostAxisTables {
  std::vector<int> ci0, ci1, bi0, bi1;
  std::vector<double> cw0, cw1, bw0, bw1, area;
  int P = 0;
};
void interp_row(const std::vector<double> &src, double d, int &i0, double &w0, int &i1, double &w1) {
  const int n = (int)src.size();
  int hi = (int)(std::lower_bound(src.begin(), src.end(), d) - src.begin());
  i0 = std::min(std::max(hi - 1, 0), n - 1);
  i1 = std::min(std::max(hi, 0), n - 1);
  w1 = src[i1] > src[i0] ? (d - src[i0]) / (src[i1] - src[i0]) : 0.0;
  if (d == src[i1]) {
    w0 = 0.0;
    w1 = 1.0;
  } else {
    w0 = 1.0 - w1;
  }
  if (d < src.front() || d > src.back()) w0 = w1 = 0.0;  // only the symmetry-plane point of the centre sites; axis_tables sets it
}
void axis_tables(const double *coords, int n, int sym, HostAxisTables &t, const double *bounds = nullptr) {
  std::vector<double> pts;
  if (n + 1 > 2) {
    for (int i = (sym == 0 ? 1 : 0); i < n; ++i) pts.push_back(coords[i]);
  }
  t.P = pts.empty() ? 1 : (int)pts.size();
  t.ci0.assign(t.P, 0); t.ci1.assign(t.P, 0); t.bi0.assign(t.P, 0); t.bi1.assign(t.P, 0);
  t.cw0.assign(t.P, 1.0); t.cw1.assign(t.P, 0.0); t.bw0.assign(t.P, 1.0); t.bw1.assign(t.P, 0.0); t.area.assign(t.P, 1.0);
  if (pts.empty()) return;  // a one-cell axis is not interpolated and has unit size
  std::vector<double> cen(n), bnd(n);
  for (int i = 0; i < n; ++i) {
    cen[i] = 0.5 * (coords[i] + coords[i + 1]);
    bnd[i] = coords[i];
  }
  for (int p = 0; p < t.P; ++p) {
    interp_row(cen, pts[p], t.ci0[p], t.cw0[p], t.ci1[p], t.cw1[p]);
    interp_row(bnd, pts[p], t.bi0[p], t.bw0[p], t.bi1[p], t.bw1[p]);
  }
  if (sym != 0) {
    // the first point is the symmetry plane: a centre-site component there is the mean of its first value v and the mirror
    // image s v, s = sym_val * symmetry_eigenvalue (components/data/dataset.py:210-220).  The components that sit on centre
    // sites along an axis (x: Ex, Hy, Hz; y: Ey, Hx, Hz) all have eigenvalue -1 along it, so s = -sym: the value itself at a
    // PEC plane (sym = -1, even components), zero at a PMC plane (sym = +1, odd components)
    t.ci0[0] = t.ci1[0] = 0;
    t.cw0[0] = sym < 0 ? 1.0 : 0.0;
    t.cw1[0] = 0.0;
  }
  if (t.P == 1) return;
  for (int p = 0; p < t.P; ++p) {
    double lo = p == 0 ? pts[0] : 0.5 * (pts[p - 1] + pts[p]);
    double hi = p == t.P - 1 ? pts[t.P - 1] : 0.5 * (pts[p] + pts[p + 1]);
    if (bounds) {  // finite plane: cell sizes truncated to the part the plane covers (monitor_data.py:450-455)
      lo = std::min(std::max(lo, bounds[0]), bounds[1]);
      hi = std::min(std::max(hi, bounds[0]), bounds[1]);
    }
    t.area[p] = hi - lo;
  }
}

// Finite-grid correction factors of the modes of one problem (mode_solver.py:847-904, see b200ms_problem.grid_correction):
// primal multiplies the tangential E, dual the tangential H.  n_complex: num_modes complex (re,im).
using zc = std::complex<double>;  // (post_batch / post_overlaps have locals called cd)
void grid_factors(const b200ms_problem &p, const double *n_complex, std::vector<zc> &primal, std::vector<zc> &dual) {
  const int M = p.num_modes;
  primal.assign(M, zc(1.0, 0.0));
  dual.assign(M, zc(1.0, 0.0));
  if (!p.grid_correction || !n_complex) return;
  const double *g = p.grid_correction;
  const double scale = 2.0 * M_PI * p.freq / kC0 / std::cos(p.angle_theta) * (p.direction < 0 ? -1.0 : 1.0);
  for (int m = 0; m < M; ++m) {
    const zc ik = zc(0.0, 1.0) * (scale * zc(n_complex[2 * m], n_complex[2 * m + 1]));
    primal[m] = g[1] * std::exp(ik * g[0]) + g[3] * std::exp(ik * g[2]);
    dual[m] = g[5] * std::exp(ik * g[4]) + g[7] * std::exp(ik * g[6]);
  }
}

struct PostBatch {  // device-side description of the problems of one device batch (kept until the window's overlaps are done)
  std::vector<PostProblem> pp;
};

// Gauge / flux / normalisation of the B problems whose packed fields start at `region` (stride `per` bytes).
void post_batch(b200ms_handle *h, const std::vector<int> &ids, const Window &W, const b200ms_problem *prob, b200ms_result *res,
                unsigned char *region, size_t per) {
  const int B = (int)ids.size();
  const b200ms_problem &p0 = prob[W.i0 + ids[0]];
  const int nx = p0.nx, ny = p0.ny, M = p0.num_modes;
  bool any = false;
  for (int b = 0; b < B; ++b)
    if (prob[W.i0 + ids[b]].post || res[W.i0 + ids[b]].flux || res[W.i0 + ids[b]].te_fraction) any = true;
  if (!any) return;
  if (M > kPostMaxModes) throw std::invalid_argument("post-processing supports at most 64 modes");
  // pack the tables of all problems into one upload
  std::vector<HostAxisTables> tx(B), ty(B);
  size_t ints = 0, dbls = 0;
  for (int b = 0; b < B; ++b) {
    const b200ms_problem &p = prob[W.i0 + ids[b]];
    axis_tables(p.coords_x, nx, p.symmetry[0], tx[b], p.plane_bounds);
    axis_tables(p.coords_y, ny, p.symmetry[1], ty[b], p.plane_bounds ? p.plane_bounds + 2 : nullptr);
    ints += 4 * (size_t)(tx[b].P + ty[b].P);
    dbls += 5 * (size_t)(tx[b].P + ty[b].P);
  }
  const size_t off_d = align256(ints * sizeof(int)), off_pp = off_d + align256(dbls * sizeof(double));
  const size_t off_part = off_pp + align256((size_t)B * sizeof(PostProblem));
  const size_t off_flux = off_part + align256((size_t)B * kPostChunks * M * kPostSlots * sizeof(double));
  const size_t off_scal = off_flux + align256((size_t)2 * B * M * sizeof(double));
  const size_t off_gc = off_scal + align256((size_t)B * M * sizeof(cplx));
  const size_t total = off_gc + align256((size_t)B * M * sizeof(cplx));
  h->post.reserve(total + 4096);
  // grid-correction factors: flux = 0.5 Re(primal conj(dual) int (E1 H2* - E2 H1*) dS); problems without them get 1
  bool any_gc = false;
  for (int b = 0; b < B; ++b) any_gc = any_gc || prob[W.i0 + ids[b]].grid_correction != nullptr;
  std::vector<cplx> hgc;
  if (any_gc) {
    hgc.resize((size_t)B * M);
    std::vector<zc> gp, gd;
    for (int b = 0; b < B; ++b) {
      grid_factors(prob[W.i0 + ids[b]], res[W.i0 + ids[b]].n_complex, gp, gd);
      for (int m = 0; m < M; ++m) {
        const zc g = gp[m] * std::conj(gd[m]);
        hgc[(size_t)b * M + m] = mk(g.real(), g.imag());
      }
    }
  }
  std::vector<int> hi(ints);
  std::vector<double> hd(dbls);
  std::vector<PostProblem> pp(B);
  size_t ci = 0, cd = 0;
  int *di = reinterpret_cast<int *>(h->post.p);
  double *dd = reinterpret_cast<double *>(h->post.p + off_d);
  auto put = [&](const HostAxisTables &t, PostAxis &a) {
    a.P = t.P;
    auto pi = [&](const std::vector<int> &v) { const int *r = di + ci; std::copy(v.begin(), v.end(), hi.begin() + ci); ci += v.size(); return r; };
    auto pd = [&](const std::vector<double> &v) { const double *r = dd + cd; std::copy(v.begin(), v.end(), hd.begin() + cd); cd += v.size(); return r; };
    a.c_i0 = pi(t.ci0); a.c_i1 = pi(t.ci1); a.b_i0 = pi(t.bi0); a.b_i1 = pi(t.bi1);
    a.c_w0 = pd(t.cw0); a.c_w1 = pd(t.cw1); a.b_w0 = pd(t.bw0); a.b_w1 = pd(t.bw1); a.area = pd(t.area);
  };
  int do_gauge = 0, do_norm = 0;
  for (int b = 0; b < B; ++b) {
    const b200ms_problem &p = prob[W.i0 + ids[b]];
    put(tx[b], pp[b].ax);
    put(ty[b], pp[b].ay);
    pp[b].fields = region + (size_t)b * per;
    pp[b].mult = (p.symmetry[0] != 0 ? 2.0 : 1.0) * (p.symmetry[1] != 0 ? 2.0 : 1.0);
    pp[b].flags = p.post;
    pp[b].ct = std::cos(p.angle_theta); pp[b].st = std::sin(p.angle_theta);
    pp[b].cp = std::cos(p.angle_phi); pp[b].sp = std::sin(p.angle_phi);
    pp[b].symx = p.symmetry[0]; pp[b].symy = p.symmetry[1];
    do_gauge |= p.post & 1;
    do_norm |= p.post & 2;
  }
  cudaStream_t st = h->stream;
  CUDA_CHECK(cudaMemcpyAsync(di, hi.data(), ints * sizeof(int), cudaMemcpyHostToDevice, st));
  CUDA_CHECK(cudaMemcpyAsync(dd, hd.data(), dbls * sizeof(double), cudaMemcpyHostToDevice, st));
  PostProblem *dpp = reinterpret_cast<PostProblem *>(h->post.p + off_pp);
  CUDA_CHECK(cudaMemcpyAsync(dpp, pp.data(), (size_t)B * sizeof(PostProblem), cudaMemcpyHostToDevice, st));
  double *dpart = reinterpret_cast<double *>(h->post.p + off_part), *dflux = reinterpret_cast<double *>(h->post.p + off_flux);
  cplx *dscal = reinterpret_cast<cplx *>(h->post.p + off_scal);
  cplx *dgc = nullptr;
  if (any_gc) {
    dgc = reinterpret_cast<cplx *>(h->post.p + off_gc);
    CUDA_CHECK(cudaMemcpyAsync(dgc, hgc.data(), hgc.size() * sizeof(cplx), cudaMemcpyHostToDevice, st));
  }
  const bool single = p0.precision == 1;
  const int nch = (int)std::min<size_t>(kPostChunks, ((size_t)2 * nx * ny + 255) / 256);
  dim3 g1(nch, B);
  if (any_gc) {
    if (single) post_scan_kernel<cplxf, true><<<g1, 256, 0, st>>>(dpp, nx, ny, M, dpart);
    else post_scan_kernel<cplx, true><<<g1, 256, 0, st>>>(dpp, nx, ny, M, dpart);
  } else {
    if (single) post_scan_kernel<cplxf, false><<<g1, 256, 0, st>>>(dpp, nx, ny, M, dpart);
    else post_scan_kernel<cplx, false><<<g1, 256, 0, st>>>(dpp, nx, ny, M, dpart);
  }
  post_final_kernel<<<B, std::max(32, ((M + 31) / 32) * 32), 0, st>>>(dpp, dpart, nch, M, dflux, dscal, dflux + (size_t)B * M, dgc);
  if (do_gauge || do_norm) {
    dim3 g2((unsigned)std::min<size_t>(((size_t)6 * nx * ny * M + 255) / 256, 2048), B);
    if (single) post_apply_kernel<cplxf><<<g2, 256, 0, st>>>(dpp, (size_t)6 * nx * ny, M, dscal);
    else post_apply_kernel<cplx><<<g2, 256, 0, st>>>(dpp, (size_t)6 * nx * ny, M, dscal);
  }
  std::vector<double> hflux((size_t)2 * B * M);
  CUDA_CHECK(cudaMemcpyAsync(hflux.data(), dflux, hflux.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_CHECK(cudaStreamSynchronize(st));
  CUDA_CHECK(cudaGetLastError());
  h->stats.launches += 3;
  for (int b = 0; b < B; ++b)
  {
    if (res[W.i0 + ids[b]].flux) std::copy(hflux.begin() + (size_t)b * M, hflux.begin() + (size_t)(b + 1) * M, res[W.i0 + ids[b]].flux);
    if (res[W.i0 + ids[b]].te_fraction)
      std::copy(hflux.begin() + (size_t)(B + b) * M, hflux.begin() + (size_t)(B + b + 1) * M, res[W.i0 + ids[b]].te_fraction);
  }
}

// Modal overlaps between consecutive problems of the call (result.overlap_prev) for the problems [i0, i1); dev_fields[i] is
// the device address of the packed fields of problem i (null if not produced).
void post_overlaps(b200ms_handle *h, const b200ms_problem *prob, b200ms_result *res, int i0, int i1, const std::vector<const void *> &dev_fields) {
  struct Job { int i; };
  std::vector<int> todo;
  for (int i = i0; i < i1; ++i) {
    if (!res[i].overlap_prev || res[i].status != B200MS_OK) continue;
    const int M = prob[i].num_modes;
    std::fill(res[i].overlap_prev, res[i].overlap_prev + (size_t)2 * M * M, 0.0);
    if (i == 0 || !dev_fields[i] || !dev_fields[i - 1]) continue;
    const b200ms_problem &a = prob[i - 1], &b = prob[i];
    if (a.nx != b.nx || a.ny != b.ny || a.num_modes != b.num_modes || (a.precision == 1) != (b.precision == 1) || M > 32) continue;
    todo.push_back(i);
  }
  // one launch per (shape, precision) run of jobs; jobs are few and small, so they are simply processed one shape at a time
  size_t k = 0;
  while (k < todo.size()) {
    const b200ms_problem &p0 = prob[todo[k]];
    size_t e = k;
    while (e < todo.size() && prob[todo[e]].nx == p0.nx && prob[todo[e]].ny == p0.ny && prob[todo[e]].num_modes == p0.num_modes &&
           (prob[todo[e]].precision == 1) == (p0.precision == 1))
      ++e;
    const int np = (int)(e - k), nx = p0.nx, ny = p0.ny, M = p0.num_modes;
    std::vector<HostAxisTables> tx(np), ty(np);
    size_t ints = 0, dbls = 0;
    for (int q = 0; q < np; ++q) {
      const b200ms_problem &p = prob[todo[k + q]];
      axis_tables(p.coords_x, nx, p.symmetry[0], tx[q], p.plane_bounds);
      axis_tables(p.coords_y, ny, p.symmetry[1], ty[q], p.plane_bounds ? p.plane_bounds + 2 : nullptr);
      ints += 4 * (size_t)(tx[q].P + ty[q].P);
      dbls += 5 * (size_t)(tx[q].P + ty[q].P);
    }
    const size_t off_d = align256(ints * sizeof(int)), off_pp = off_d + align256(dbls * sizeof(double));
    const size_t off_pairs = off_pp + align256((size_t)np * sizeof(PostProblem));
    bool any_gc = false;  // grid-correction factors on either side of a pair: keep the two cross products apart
    for (int q = 0; q < np; ++q) any_gc = any_gc || prob[todo[k + q]].grid_correction || prob[todo[k + q] - 1].grid_correction;
    const int E = (any_gc ? 2 : 1) * M * M;
    const size_t off_part = off_pairs + align256((size_t)np * sizeof(PostPair));
    const size_t off_out = off_part + align256((size_t)np * kPostChunks * E * sizeof(cplx));
    h->post.reserve(off_out + align256((size_t)np * E * sizeof(cplx)) + 4096);
    std::vector<int> hi(ints);
    std::vector<double> hd(dbls);
    std::vector<PostProblem> pp(np);
    std::vector<PostPair> pairs(np);
    size_t ci = 0, cd = 0;
    int *di = reinterpret_cast<int *>(h->post.p);
    double *dd = reinterpret_cast<double *>(h->post.p + off_d);
    auto put = [&](const HostAxisTables &t, PostAxis &a) {
      a.P = t.P;
      auto pi = [&](const std::vector<int> &v) { const int *r = di + ci; std::copy(v.begin(), v.end(), hi.begin() + ci); ci += v.size(); return r; };
      auto pd = [&](const std::vector<double> &v) { const double *r = dd + cd; std::copy(v.begin(), v.end(), hd.begin() + cd); cd += v.size(); return r; };
      a.c_i0 = pi(t.ci0); a.c_i1 = pi(t.ci1); a.b_i0 = pi(t.bi0); a.b_i1 = pi(t.bi1);
      a.c_w0 = pd(t.cw0); a.c_w1 = pd(t.cw1); a.b_w0 = pd(t.bw0); a.b_w1 = pd(t.bw1); a.area = pd(t.area);
    };
    for (int q = 0; q < np; ++q) {
      const int i = todo[k + q];
      put(tx[q], pp[q].ax);
      put(ty[q], pp[q].ay);
      pp[q].fields = const_cast<void *>(dev_fields[i]);
      pp[q].mult = (prob[i].symmetry[0] != 0 ? 2.0 : 1.0) * (prob[i].symmetry[1] != 0 ? 2.0 : 1.0);
      pp[q].flags = 0;
      pp[q].ct = pp[q].cp = 1.0;
      pp[q].st = pp[q].sp = 0.0;
      pp[q].symx = pp[q].symy = 0;
      pairs[q].a = dev_fields[i - 1];
      pairs[q].b = dev_fields[i];
      pairs[q].prob = q;
    }
    cudaStream_t st = h->stream;
    CUDA_CHECK(cudaMemcpyAsync(di, hi.data(), ints * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_CHECK(cudaMemcpyAsync(dd, hd.data(), dbls * sizeof(double), cudaMemcpyHostToDevice, st));
    PostProblem *dpp = reinterpret_cast<PostProblem *>(h->post.p + off_pp);
    PostPair *dpairs = reinterpret_cast<PostPair *>(h->post.p + off_pairs);
    CUDA_CHECK(cudaMemcpyAsync(dpp, pp.data(), (size_t)np * sizeof(PostProblem), cudaMemcpyHostToDevice, st));
    CUDA_CHECK(cudaMemcpyAsync(dpairs, pairs.data(), (size_t)np * sizeof(PostPair), cudaMemcpyHostToDevice, st));
    cplx *dpart = reinterpret_cast<cplx *>(h->post.p + off_part), *dout = reinterpret_cast<cplx *>(h->post.p + off_out);
    const int nch = (int)std::min<size_t>(kPostChunks, ((size_t)nx * ny + 255) / 256);
    dim3 g(nch, np, M * M);
    if (any_gc) {
      if (p0.precision == 1) post_dot_kernel<cplxf, true><<<g, 256, 0, st>>>(dpp, dpairs, nx, ny, M, dpart);
      else post_dot_kernel<cplx, true><<<g, 256, 0, st>>>(dpp, dpairs, nx, ny, M, dpart);
    } else {
      if (p0.precision == 1) post_dot_kernel<cplxf, false><<<g, 256, 0, st>>>(dpp, dpairs, nx, ny, M, dpart);
      else post_dot_kernel<cplx, false><<<g, 256, 0, st>>>(dpp, dpairs, nx, ny, M, dpart);
    }
    post_dot_final_kernel<<<np, std::min(1024, std::max(32, ((M * M + 31) / 32) * 32)), 0, st>>>(dpart, nch, E, dout);
    std::vector<cplx> hout((size_t)np * E);
    CUDA_CHECK(cudaMemcpyAsync(hout.data(), dout, hout.size() * sizeof(cplx), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    CUDA_CHECK(cudaGetLastError());
    h->stats.launches += 2;
    if (!any_gc) {
      for (int q = 0; q < np; ++q) std::memcpy(res[todo[k + q]].overlap_prev, hout.data() + (size_t)q * M * M, (size_t)M * M * sizeof(cplx));
    } else {  // dot = conj(primal_a) dual_b (1/4 int Ea* x Hb) - conj(dual_a) primal_b (1/4 int Ha* x Eb)   (monitor_data.py:488-503, 680-697)
      std::vector<zc> pa, da, pb, db;
      for (int q = 0; q < np; ++q) {
        const int i = todo[k + q];
        grid_factors(prob[i - 1], res[i - 1].n_complex, pa, da);
        grid_factors(prob[i], res[i].n_complex, pb, db);
        const cplx *i1 = hout.data() + (size_t)q * E, *i2 = i1 + (size_t)M * M;
        for (int ma = 0; ma < M; ++ma)
          for (int mb = 0; mb < M; ++mb) {
            const size_t e = (size_t)ma * M + mb;
            const zc v = std::conj(pa[ma]) * db[mb] * zc(i1[e].re, i1[e].im) - std::conj(da[ma]) * pb[mb] * zc(i2[e].re, i2[e].im);
            res[i].overlap_prev[2 * e] = v.real();
            res[i].overlap_prev[2 * e + 1] = v.imag();
          }
      }
    }
    k = e;
  }
}

struct FieldCopy {  // one pending delivery of packed fields: device region -> caller memory (host or device)
  void *dst;
  const void *src;
  size_t bytes;
};

// Why the permittivity gradient (b200ms_result.grad_eps) is not available for a problem; nullptr when it is (csrc/sensitivity.cuh)
const char *grad_unsupported(const b200ms_problem &p, const ProblemSetup &s) {
  if (s.tensorial) return "grad_eps: tensorial (angled or off-diagonal eps) problems are not supported";
  if (!std::isnan(p.bend_radius)) return "grad_eps: bent waveguides are not supported";
  if (p.mu || p.incidence) return "grad_eps: mu_cross / split_curl_scaling are not supported";
  if (s.relative) return "grad_eps: the relative mode solver (basis fields) is not supported";
  if (s.has_pec) return "grad_eps: problems with PEC-valued cells are not supported";
  return nullptr;
}

template <typename T, typename C, typename P, typename PC>
void solve_group(b200ms_handle *h, const std::vector<int> &ids, const Window &W, const b200ms_problem *prob, b200ms_result *res,
                 unsigned char *out_region, const std::vector<cplx *> &grad_dst, std::vector<FieldCopy> &copies) {
  // ids index into the window (global problem index = W.i0 + id)
  const int B = (int)ids.size();
  std::vector<const ProblemSetup *> ps(B);
  std::vector<MediumRef> refs(B);
  bool share = true;
  for (int b = 0; b < B; ++b) {
    ps[b] = &W.setups[ids[b]];
    refs[b] = W.refs[ids[b]];
    refs[b].p.incidence = ps[b]->masked ? 1 : 0;  // zero-markers only where the diagonal path really removes unknowns
    if (W.slot[ids[b]] != W.slot[ids[0]]) share = false;
  }
  if (share) refs.resize(1);
  BatchSolver<T, C, P, PC> S(h->arena, h->stream, h->opt);
  auto wall0 = std::chrono::steady_clock::now();
  S.single_out_ = prob[W.i0 + ids[0]].precision == 1;
  const MediumRef *d_refs = upload_refs(h, refs, h->stream);
  {
    NvtxRange r("b200ms:build (hierarchy, coefficient fields, graph capture)");
    S.build(ps, share, d_refs);
  }
  S.set_output(reinterpret_cast<cplx *>(out_region));
  h->stats.setup_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
  CUDA_CHECK(cudaEventRecord(h->ev0, h->stream));  // inputs are resident in HBM from here on
  const bool real_arith = std::is_same<T, double>::value;
  const bool relative = ps[0]->relative;
  const int k = S.k;
  typename BatchSolver<T, C, P, PC>::EigResult eig;
  std::vector<cd> rel_vals;
  if (relative) {
    std::vector<const cd *> basis(B);
    for (int b = 0; b < B; ++b) basis[b] = reinterpret_cast<const cd *>(prob[W.i0 + ids[b]].basis_e);
    rel_vals = S.solve_relative(basis);
    eig.nconv.assign(B, k);
    eig.resid.assign(B, 0.0);
  } else {
    S.init_start_vector(0);
    NvtxRange r("b200ms:eigen-iteration");
    eig = S.krylov_schur(real_arith);
  }
  // eigenvalues of A: lambda = sigma + 1/theta; n = sqrt(-lambda) (principal root, solver.py:884)
  std::vector<cd> nsorted((size_t)B * k), lam((size_t)B * k);
  std::vector<int> perm((size_t)B * k);
  for (int b = 0; b < B; ++b) {
    std::vector<cd> nn(k), ll(k);
    for (int q = 0; q < k; ++q) {
      if (relative) {
        ll[q] = rel_vals[(size_t)b * k + q];
      } else {
        cd th = eig.theta[(size_t)b * k + q];
        ll[q] = (S.tensor_ ? ps[b]->sigma_t : ps[b]->sigma) + (std::abs(th) > 0 ? 1.0 / th : cd(0, 0));
      }
      if (S.tensor_) {
        nn[q] = ll[q];  // the first-order operator's eigenvalue is n_eff + i k_eff itself (solver.py:879-880)
      } else {
        nn[q] = std::sqrt(-ll[q]);
        if (nn[q].real() < 0) nn[q] = -nn[q];
      }
    }
    std::vector<int> o(k);
    for (int q = 0; q < k; ++q) o[q] = q;
    std::stable_sort(o.begin(), o.end(), [&](int a, int c) { return nn[a].real() > nn[c].real(); });  // solver.py:559
    for (int q = 0; q < k; ++q) {
      perm[(size_t)b * k + q] = o[q];
      nsorted[(size_t)b * k + q] = nn[o[q]];
      lam[(size_t)b * k + q] = ll[o[q]];
    }
  }
  bool want_fields = false;
  for (int b = 0; b < B; ++b) {
    const b200ms_result &rb = res[W.i0 + ids[b]];
    if (rb.fields || rb.flux || rb.te_fraction || rb.overlap_prev || prob[W.i0 + ids[b]].post) want_fields = true;  // post-processing needs them in HBM
  }
  S.epilogue(nsorted, perm, ps, nullptr, want_fields);
  if (std::any_of(grad_dst.begin(), grad_dst.end(), [](cplx *p) { return p != nullptr; })) {
    NvtxRange r("b200ms:permittivity gradient");
    S.sensitivity(nsorted, ps, grad_dst);
  }
  // true residuals on the sorted Ritz vectors (they sit in the FGMRES Z scratch after the permutation)
  std::vector<double> maxres(B, 0.0);
  {
    CUDA_CHECK(cudaMemcpyAsync(S.ritz_ptr(), S.gmres_z(), (size_t)k * S.vstride * sizeof(T), cudaMemcpyDeviceToDevice, h->stream));
    for (int q = 0; q < k; ++q) {
      std::vector<cd> lq(B);
      for (int b = 0; b < B; ++b) lq[b] = lam[(size_t)b * k + q];
      auto r = S.eigen_residuals(q, lq);
      for (int b = 0; b < B; ++b) maxres[b] = std::max(maxres[b], r[b]);
    }
  }
  CUDA_CHECK(cudaEventRecord(h->ev1, h->stream));
  CUDA_CHECK(cudaEventSynchronize(h->ev1));
  float ms = 0.f;
  CUDA_CHECK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  const size_t per = S.output_bytes_per_problem();
  if (want_fields)
    for (int b = 0; b < B; ++b)
      if (res[W.i0 + ids[b]].fields) copies.push_back({res[W.i0 + ids[b]].fields, out_region + (size_t)b * per, per});
  for (int b = 0; b < B; ++b)
    if (grad_dst[b]) copies.push_back({res[W.i0 + ids[b]].grad_eps, grad_dst[b], (size_t)3 * S.N * k * sizeof(cplx)});
  h->stats.device_ms += ms;
  h->stats.launches += S.stats.launches;
  h->stats.inner_iters += (long long)S.stats.inner_iters * B;
  h->stats.op_applies += (long long)S.stats.op_applies * B;
  h->stats.host_syncs += S.stats.host_syncs;
  h->stats.device_batches += 1;
  const double total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
  for (int b = 0; b < B; ++b) {
    b200ms_result &r = res[W.i0 + ids[b]];
    for (int q = 0; q < k; ++q) {
      cd n = nsorted[(size_t)b * k + q] * ps[b]->knorm;  // solver.py:262-263
      r.n_complex[2 * q] = n.real();
      r.n_complex[2 * q + 1] = n.imag();
    }
    r.eps_spec = ps[b]->eps_spec;
    r.converged = eig.nconv[b];
    r.outer_iters = S.stats.restarts;
    r.op_applies = S.stats.op_applies;
    r.inner_iters = S.stats.inner_iters;
    r.stencil_applies = (int)std::min<long>(S.stats.launches, 2147483647L);
    r.is_complex = real_arith ? 0 : 1;
    r.solve_ms = ms;
    r.total_ms = total_ms;
    r.max_residual = maxres[b];
    // converged == Ritz residuals of OP below eig_tol (ARPACK's criterion).  The residual with respect to A itself is
    // reported for information: it is amplified by ||A - sigma|| ~ 1/(k0 dl)^2 (and by 1e8 next to PEC cells) and only
    // screened for garbage (O(1)) here.
    // With PEC-valued cells (|eps| = 1e8) that amplification makes the figure meaningless at the reference's tolerance
    // (measured 0.25 on pec_block_40 with |dn| < 1e-8), so the screen is skipped there.
    r.status = (relative || (eig.nconv[b] == k && eig.ok && (maxres[b] < 1e-1 || ps[b]->has_pec) && S.stats.inner_failures == 0)) ? B200MS_OK : B200MS_ERR_NOCONV;
    if (h->opt.verbose)
      fprintf(stderr, "[b200ms] prob %d: conv %d/%d ok %d restarts %d op %d inner %d cycles %d syncs %ld reorth %d innerfail %d res %.2e ms %.1f\n", W.i0 + ids[b],
              eig.nconv[b], k, (int)eig.ok, S.stats.restarts, S.stats.op_applies, S.stats.inner_iters, S.stats.inner_cycles, S.stats.host_syncs,
              S.stats.outer_second_pass, S.stats.inner_failures, maxres[b], ms);
  }
}

// device memory one problem of a batch needs in the solver arena (Krylov bases dominate)
size_t bytes_per_problem(const ProblemSetup &s, const b200ms_options &opt) {
  const size_t N = (size_t)s.nx * s.ny;
  const size_t len = (s.tensorial ? 4 : 2) * N;
  const size_t sv = s.is_complex ? 16 : 8;
  const int m = opt.ncv > 0 ? opt.ncv : std::max(2 * s.num_modes + 1, 20);
  size_t vecs = (m + 1) + (2 * opt.gmres_restart + 1) + 4 + s.num_modes;
  size_t bytes = vecs * len * sv;
  bytes += (size_t)7 * 2 * N * sv * 4 / 3;            // multigrid level work vectors (x, b, r, tmp, dinv + coarse levels)
  bytes += (size_t)(s.has_mu ? 6 : 3) * N * 16 * 2;   // coefficient fields in both precisions
  if (s.tensorial) bytes += (size_t)18 * N * 16 + (size_t)6 * 2 * N * sv;  // derived tensor fields + preconditioner scratch
  return bytes;
}

template <typename... A>
void dispatch_group(int kind, A &&...a) {
  switch (kind) {
    case 0: solve_group<double, double, float, float>(std::forward<A>(a)...); break;
    case 1: solve_group<cplx, double, cplxf, float>(std::forward<A>(a)...); break;
    default: solve_group<cplx, cplx, cplxf, cplxf>(std::forward<A>(a)...); break;
  }
}

}  // namespace

extern "C" int b200ms_solve_batch(b200ms_handle *h, int nprob, const b200ms_problem *prob, b200ms_result *res) {
  if (!h || nprob < 0 || (nprob > 0 && (!prob || !res))) return B200MS_ERR_ARG;
  if (cudaSetDevice(h->device) != cudaSuccess) return B200MS_ERR_CUDA;
  h->err.clear();
  std::memset(&h->stats, 0, sizeof(h->stats));
  h->stats.nprob = nprob;
  const auto call0 = std::chrono::steady_clock::now();
  int first_err = B200MS_OK;
  try {
    // Windows of consecutive problems: a window's raw media are uploaded and scanned together, then its problems are
    // grouped by (shape, arithmetic kind, ...) and solved in device batches.  Three things run concurrently: the solve of
    // window w (this thread, h->stream), the upload + scan of window w+1 and the delivery of the fields of window w-1
    // (helper threads, h->io_stream); raw media and packed fields are double-buffered.
    const int wsize = std::max(1, h->opt.max_batch);
    const int nwin = (nprob + wsize - 1) / wsize;
    const int dev = h->device;
    Window Wn[2];
    auto upload = [h, prob, nprob, wsize, dev](int wi, Window *W) {
      if (cudaSetDevice(dev) != cudaSuccess) throw std::runtime_error("cudaSetDevice failed in the upload thread");
      const auto t0 = std::chrono::steady_clock::now();
      NvtxRange r("b200ms:upload + set-up of a window");
      prepare_window(h, prob, wi * wsize, std::min(nprob, (wi + 1) * wsize), h->raw[wi & 1], h->io_stream, *W);
      return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    auto download = [h, dev](std::vector<FieldCopy> copies) {
      if (cudaSetDevice(dev) != cudaSuccess) throw std::runtime_error("cudaSetDevice failed in the download thread");
      const auto t0 = std::chrono::steady_clock::now();
      NvtxRange r("b200ms:delivery of a window's fields");
      for (const FieldCopy &c : copies) CUDA_CHECK(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDefault, h->dl_stream));
      CUDA_CHECK(cudaStreamSynchronize(h->dl_stream));
      return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    std::future<double> up_f, dl_f;
    std::vector<const void *> dev_fields(nprob, nullptr);  // device address of each problem's packed fields (this + previous window)
    if (nwin > 0) h->stats.setup_ms += upload(0, &Wn[0]);
    size_t free_b = 0, total_b = 0;
    for (int wi = 0; wi < nwin; ++wi) {
      const int i0 = wi * wsize, i1 = std::min(nprob, i0 + wsize);
      Window &W = Wn[wi & 1];
      if (wi + 1 < nwin) up_f = std::async(std::launch::async, upload, wi + 1, &Wn[(wi + 1) & 1]);
      try {
        for (int i = i0; i < i1; ++i) {
          res[i].status = res[i].n_complex ? B200MS_OK : B200MS_ERR_ARG;
          res[i].converged = 0;
        }
        std::map<GroupKey, std::vector<int>> groups;
        size_t out_bytes = 0, grad_bytes = 0;
        for (int q = 0; q < i1 - i0; ++q) {
          const int i = i0 + q;
          const ProblemSetup &s = W.setups[q];
          if (res[i].status == B200MS_OK) res[i].status = s.status;
          res[i].eps_spec = s.eps_spec;
          res[i].is_complex = s.is_complex;
          const char *no_grad = (res[i].status == B200MS_OK && res[i].grad_eps) ? grad_unsupported(prob[i], s) : nullptr;
          if (no_grad) res[i].status = B200MS_ERR_UNSUPPORTED;
          if (res[i].status != B200MS_OK) {
            if (first_err == B200MS_OK) {
              first_err = res[i].status;
              h->err = no_grad ? no_grad : s.error.empty() ? "bad result buffers" : s.error;
            }
            continue;
          }
          GroupKey key{s.nx, s.ny, s.num_modes, kind_of(s), s.has_mu ? 1 : 0, prob[i].symmetry[0], prob[i].symmetry[1],
                       s.jz_axis, s.direction, s.relative ? 1 : 0, s.tensorial ? (s.eps_complex ? 2 : 1) : 0, prob[i].precision == 1 ? 1 : 0,
                       s.masked ? 1 : 0, prob[i].angle_theta, prob[i].angle_phi};
          groups[key].push_back(q);
          out_bytes += align256((size_t)6 * s.nx * s.ny * s.num_modes * (prob[i].precision == 1 ? 8 : 16));
          if (res[i].grad_eps) grad_bytes += align256((size_t)3 * s.nx * s.ny * s.num_modes * sizeof(cplx));
        }
        DevBuf &ob = h->out[wi & 1];  // last read by the delivery of window wi-2, which has completed (see below)
        ob.reserve(std::max<size_t>(out_bytes + grad_bytes + 4096, 4096));
        size_t gcursor = out_bytes;  // permittivity gradients follow the packed fields
        CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
        free_b += h->arena.cap;
        std::vector<FieldCopy> copies;
        size_t cursor = 0;
        for (auto &kv : groups) {
          const std::vector<int> &all = kv.second;
          const size_t per = bytes_per_problem(W.setups[all[0]], h->opt);
          int bmax = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(1, h->opt.max_batch), (size_t)(0.8 * free_b) / per));
          for (size_t s0 = 0; s0 < all.size();) {
            std::vector<int> ids(all.begin() + s0, all.begin() + std::min(all.size(), s0 + bmax));
            const ProblemSetup &sg = W.setups[ids[0]];
            const size_t pb = (size_t)6 * sg.nx * sg.ny * sg.num_modes * (prob[i0 + ids[0]].precision == 1 ? 8 : 16);
            unsigned char *region = ob.p + cursor;
            if (cursor + pb * ids.size() > ob.cap) throw std::runtime_error("output buffer accounting error");
            std::vector<cplx *> grad_dst(ids.size(), nullptr);
            size_t gc = gcursor;
            for (size_t b = 0; b < ids.size(); ++b)
              if (res[i0 + ids[b]].grad_eps) {
                grad_dst[b] = reinterpret_cast<cplx *>(ob.p + gc);
                gc += align256((size_t)3 * sg.nx * sg.ny * sg.num_modes * sizeof(cplx));
              }
            if (gc > ob.cap) throw std::runtime_error("output buffer accounting error");
            try {
              dispatch_group(kv.first.kind, h, ids, W, prob, res, region, grad_dst, copies);
            } catch (const DeviceOutOfMemory &) {
              // bytes_per_problem is an estimate (other processes, fragmentation): the arena is reserved before anything else
              // of the batch happens, so the same problems are simply solved in smaller device batches
              if (ids.size() == 1) throw;
              bmax = std::max<int>(1, (int)ids.size() / 2);
              h->arena.release();
              if (h->opt.verbose) fprintf(stderr, "[b200ms] solver arena does not fit: device batch reduced to %d problems\n", bmax);
              continue;
            }
            s0 += ids.size();
            gcursor = gc;
            {
              NvtxRange r("b200ms:post-processing in HBM");
              post_batch(h, ids, W, prob, res, region, pb);  // gauge / flux / normalisation in HBM, before delivery
            }
            for (size_t b = 0; b < ids.size(); ++b) {
              const int id = ids[b];
              dev_fields[i0 + id] = region + b * pb;
              if (res[i0 + id].status != B200MS_OK && first_err == B200MS_OK) {
                first_err = res[i0 + id].status;
                h->err = "eigen-iteration did not converge";
              }
            }
            cursor += align256(pb * ids.size());
          }
        }
        {
          NvtxRange r("b200ms:modal overlaps");
          post_overlaps(h, prob, res, i0, i1, dev_fields);  // modal overlaps between consecutive problems (fields still in HBM)
        }
        // deliver the fields of this window (destination may be host or device memory) while the next window is solved;
        // at most one delivery is in flight, so out[wi & 1] is free again by the time window wi + 2 writes it
        if (dl_f.valid()) h->stats.download_ms += dl_f.get();
        if (!copies.empty()) dl_f = std::async(std::launch::async, download, std::move(copies));
      } catch (...) {
        if (up_f.valid()) try { up_f.get(); } catch (...) {}
        if (dl_f.valid()) try { dl_f.get(); } catch (...) {}
        throw;
      }
      if (up_f.valid()) h->stats.setup_ms += up_f.get();
    }
    if (dl_f.valid()) h->stats.download_ms += dl_f.get();
  } catch (const std::invalid_argument &e) {
    h->err = e.what();
    return B200MS_ERR_ARG;
  } catch (const std::exception &e) {  // CUDA runtime failures, device memory exhaustion
    h->err = e.what();
    return B200MS_ERR_CUDA;
  }
  h->stats.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - call0).count();
  return first_err;
}

// ---- benchmark hook -----------------------------------------------------------------------------------
// mode 0: the fp64 operator apply of the Krylov iteration (true PML);  mode 1: the production smoother sweep
// (stored-diagonal Jacobi in the multigrid precision, fp32 by default)
template <typename T, typename C, typename P, typename PC>
static void bench_group(b200ms_handle *h, const Window &W, int nbatch, int mode, int nrep, int flush_l2,
                        const double *x, double *y, double *ms_out, double *bytes_out) {
  std::vector<const ProblemSetup *> ps(nbatch, &W.setups[0]);
  std::vector<MediumRef> refs(nbatch, W.refs[0]);
  BatchSolver<T, C, P, PC> S(h->arena, h->stream, h->opt);
  S.build(ps, false, upload_refs(h, refs, h->stream));
  const size_t len = S.len;
  std::vector<T> hx(len);
  std::vector<P> hp(len);
  std::mt19937_64 rng(7);
  std::uniform_real_distribution<double> U(-1.0, 1.0);
  for (size_t e = 0; e < len; ++e) {
    cd v = x ? cd(x[2 * e], x[2 * e + 1]) : cd(U(rng), U(rng));
    hx[e] = from_cd<T>(v);
    hp[e] = from_cd<P>(v);
  }
  T *dx = S.basis0(), *dy = S.basis0() + S.vstride, *drhs = S.basis0() + 2 * S.vstride;
  P *px = reinterpret_cast<P *>(S.basis0() + 3 * S.vstride), *py = px + S.vstride, *prhs = px + 2 * S.vstride;
  for (int b = 0; b < nbatch; ++b) {
    CUDA_CHECK(cudaMemcpyAsync(dx + (size_t)b * len, hx.data(), len * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(drhs + (size_t)b * len, hx.data(), len * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(px + (size_t)b * len, hp.data(), len * sizeof(P), cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(prhs + (size_t)b * len, hp.data(), len * sizeof(P), cudaMemcpyHostToDevice, h->stream));
  }
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (flush_l2 && !h->flush_buf) {
    h->flush_bytes = (size_t)256 << 20;
    CUDA_CHECK(cudaMalloc(&h->flush_buf, h->flush_bytes));
  }
  // mode 2: one fused CGS2 step in the multigrid precision against 4 basis vectors (slots 0..3 of the FGMRES basis)
  P *gsV = reinterpret_cast<P *>(S.gmres_v()), *gsW = gsV + 4 * S.vstride;
  if (mode == 2)
    for (int q = 0; q < 5; ++q)
      for (int b = 0; b < nbatch; ++b)
        CUDA_CHECK(cudaMemcpyAsync(gsV + (size_t)q * S.vstride + (size_t)b * len, hp.data(), len * sizeof(P), cudaMemcpyHostToDevice, h->stream));
  // mode 3: the permittivity-gradient kernels, every mode slot holding the random vector, n = 2 for every mode
  cplx *gdst = nullptr;
  if (mode == 3) {
    for (int q = 0; q < S.k; ++q)
      for (int b = 0; b < nbatch; ++b)
        CUDA_CHECK(cudaMemcpyAsync(S.gmres_z() + (size_t)q * S.vstride + (size_t)b * len, hx.data(), len * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMalloc(&gdst, (size_t)nbatch * S.k * 3 * S.N * sizeof(cplx)));
    std::vector<cplx *> dst(nbatch);
    for (int b = 0; b < nbatch; ++b) dst[b] = gdst + (size_t)b * S.k * 3 * S.N;
    S.sensitivity_upload(std::vector<cd>((size_t)nbatch * S.k, cd(2.0, 0.0)), ps, dst);
  }
  auto run = [&]() {
    if (mode == 3) S.sensitivity_launch();
    else if (mode == 2) S.template gs_cgs2<P>(gsV, S.vstride, len, 4, gsW, gsW, nullptr, reinterpret_cast<P *>(S.hessenberg()), (size_t)S.restart * (S.restart + 4));
    else if (mode == 1) S.apply(0, MODE_JACOBI, px, prhs, py);
    else S.apply_true(MODE_APPLY, dx, drhs, dy);
  };
  for (int w = 0; w < 3; ++w) run();
  double total = 0.0;
  if (flush_l2) {
    for (int r = 0; r < nrep; ++r) {
      CUDA_CHECK(cudaMemsetAsync(h->flush_buf, r & 0xff, h->flush_bytes, h->stream));
      CUDA_CHECK(cudaEventRecord(h->ev0, h->stream));
      run();
      CUDA_CHECK(cudaEventRecord(h->ev1, h->stream));
      CUDA_CHECK(cudaEventSynchronize(h->ev1));
      float ms = 0.f;
      CUDA_CHECK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
      total += ms;
    }
  } else {
    CUDA_CHECK(cudaEventRecord(h->ev0, h->stream));
    for (int r = 0; r < nrep; ++r) run();
    CUDA_CHECK(cudaEventRecord(h->ev1, h->stream));
    CUDA_CHECK(cudaEventSynchronize(h->ev1));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    total = ms;
  }
  CUDA_CHECK(cudaGetLastError());
  if (gdst) CUDA_CHECK(cudaFree(gdst));
  if (ms_out) *ms_out = total / nrep;
  // algorithmic bytes (SURVEY 8(d)): apply = read v (2) + write Av (2) + nf coefficient fields per cell;
  // smoother sweep = read x, rhs, omega/diag (6) + write x' (2) + nf coefficient fields per cell
  const double ncell = (double)S.N * nbatch;
  if (bytes_out && mode == 3)  // scan and write pass each read v (2) + exx, eyy, iez per cell and mode; write 3 complex128
    *bytes_out = ncell * S.k * (2.0 * (2.0 * sizeof(T) + 3.0 * sizeof(C)) + 3.0 * sizeof(cplx));
  else if (bytes_out && mode == 2)  // dots: 4+1 vectors; update+dots: 4 + r/w w; update+norm: 4 + r/w w; scale: r + w
    *bytes_out = (double)len * nbatch * sizeof(P) * 19.0;
  else if (bytes_out)
    *bytes_out = mode == 1 ? ncell * (8.0 * sizeof(P) + (double)S.nf * sizeof(PC)) : ncell * (4.0 * sizeof(T) + (double)S.nf * sizeof(C));
  if (y) {
    for (size_t e = 0; e < len; ++e) {
      cd v;
      if (mode == 1) {
        P t;
        CUDA_CHECK(cudaMemcpy(&t, py + e, sizeof(P), cudaMemcpyDeviceToHost));
        v = to_cd(t);
      } else {
        T t;
        CUDA_CHECK(cudaMemcpy(&t, dy + e, sizeof(T), cudaMemcpyDeviceToHost));
        v = to_cd(t);
      }
      y[2 * e] = v.real();
      y[2 * e + 1] = v.imag();
    }
  }
}

extern "C" int b200ms_bench_stencil(b200ms_handle *h, const b200ms_problem *prob, int nbatch, int mode, int nrep,
                                    int flush_l2, const double *x, double *y, double *ms_per_launch,
                                    double *bytes_per_apply) {
  if (!h || !prob || nbatch < 1 || nrep < 1) return B200MS_ERR_ARG;
  if (cudaSetDevice(h->device) != cudaSuccess) return B200MS_ERR_CUDA;
  try {
    Window W;
    prepare_window(h, prob, 0, 1, h->raw[0], h->stream, W);
    const ProblemSetup &s = W.setups[0];
    if (s.status != B200MS_OK) {
      h->err = s.error;
      return s.status;
    }
    switch (kind_of(s)) {
      case 0:
        bench_group<double, double, float, float>(h, W, nbatch, mode, nrep, flush_l2, x, y, ms_per_launch, bytes_per_apply);
        break;
      case 1:
        bench_group<cplx, double, cplxf, float>(h, W, nbatch, mode, nrep, flush_l2, x, y, ms_per_launch, bytes_per_apply);
        break;
      default:
        bench_group<cplx, cplx, cplxf, cplxf>(h, W, nbatch, mode, nrep, flush_l2, x, y, ms_per_launch, bytes_per_apply);
        break;
    }
  } catch (const std::exception &e) {
    h->err = e.what();
    return B200MS_ERR_CUDA;
  }
  return B200MS_OK;
}

// ---- host-only debug hooks ----------------------------------------------------------------------------
extern "C" int b200ms_debug_schur(int n, const double *a, double *t, double *q) {
  if (n < 1 || !a || !t || !q) return B200MS_ERR_ARG;
  CMat A(n, n), Q;
  for (int i = 0; i < n * n; ++i) A.a[i] = cd(a[2 * i], a[2 * i + 1]);
  bool ok = schur(A, Q);
  for (int i = 0; i < n * n; ++i) {
    t[2 * i] = A.a[i].real();
    t[2 * i + 1] = A.a[i].imag();
    q[2 * i] = Q.a[i].real();
    q[2 * i + 1] = Q.a[i].imag();
  }
  return ok ? B200MS_OK : B200MS_ERR_NOCONV;
}

extern "C" int b200ms_debug_sensitivity(const b200ms_problem *prob, const double *vec, const double *lambda, double *out) {
  if (!prob || !vec || !lambda || !out) return B200MS_ERR_ARG;
  ProblemSetup s;
  setup_problem(*prob, s);
  if (s.status != B200MS_OK) return s.status;
  if (grad_unsupported(*prob, s)) return B200MS_ERR_UNSUPPORTED;
  const int nx = s.nx, ny = s.ny;
  const size_t N = (size_t)nx * ny;
  // the device operands of sensitivity(): 1-D coefficients, exx, eyy, 1 / ezz (the host mirror stores ezz), Yee lengths
  std::vector<cplx> cx(4 * nx), cy(4 * ny), f(3 * N), len[2];
  for (int a = 0; a < 2; ++a) {
    std::vector<cd> c;
    s.ax[a].coefficients(c);
    cplx *dst = a == 0 ? cx.data() : cy.data();
    for (size_t i = 0; i < c.size(); ++i) dst[i] = mk(c[i].real(), c[i].imag());
    const Axis &A = s.ax[a];
    len[a].resize(2 * A.n);
    for (int i = 0; i < A.n; ++i) {
      len[a][i] = mk(A.lf[i].real(), A.lf[i].imag());
      len[a][A.n + i] = mk(A.lb[i].real(), A.lb[i].imag());
    }
    if (A.pmc && A.n > 1) len[a][A.n] = 0.5 * len[a][A.n];
  }
  for (size_t i = 0; i < N; ++i) {
    f[i] = mk(s.f(0)[i].real(), s.f(0)[i].imag());
    f[N + i] = mk(s.f(1)[i].real(), s.f(1)[i].imag());
    const cd iez = 1.0 / s.f(2)[i];
    f[2 * N + i] = mk(iez.real(), iez.imag());
  }
  const cplx *v = reinterpret_cast<const cplx *>(vec);
  const SensCell<cplx, cplx> c{nx, ny, v, v + N, f.data(), f.data() + N, f.data() + 2 * N, nullptr, cx.data(), cy.data()};
  cplx S = mk(0.0, 0.0);
  for (int i = 0; i < nx; ++i)
    for (int j = 0; j < ny; ++j) {
      cplx e1, e2, q1, q2, u, ax, ay, az;
      sens_cell(c, i, j, e1, e2, q1, q2, u);
      sens_areas(len[0].data(), len[1].data(), nx, ny, i, j, ax, ay, az);
      S += sens_flux_term(ax, ay, e1, e2, q1, q2);
    }
  cd n = std::sqrt(-cd(lambda[0], lambda[1]));  // n_complex of the mode (solver.py:884)
  if (n.real() < 0) n = -n;
  const cplx nc = mk(n.real(), n.imag()), inv2s = recip(2.0 * S);
  cplx *o = reinterpret_cast<cplx *>(out);
  for (int i = 0; i < nx; ++i)
    for (int j = 0; j < ny; ++j) {
      cplx e1, e2, q1, q2, u, ax, ay, az, g[3];
      sens_cell(c, i, j, e1, e2, q1, q2, u);
      sens_areas(len[0].data(), len[1].data(), nx, ny, i, j, ax, ay, az);
      sens_grad(nc, inv2s, ax, ay, az, e1, e2, u, g);
      const size_t t = (size_t)i * ny + j;
      for (int q = 0; q < 3; ++q) o[q * N + t] = g[q];
    }
  return B200MS_OK;
}

extern "C" int b200ms_debug_setup(const b200ms_problem *prob, double *sigma, int *flags, double *target, double *knorm,
                                  double *coef_x, double *coef_y, double *fields) {
  if (!prob) return B200MS_ERR_ARG;
  NvtxRange r("b200ms:debug set-up (host mirror)");  // also keeps the NVTX path exercised where there is no GPU
  ProblemSetup s;
  setup_problem(*prob, s);
  if (s.status != B200MS_OK && s.status != B200MS_ERR_UNSUPPORTED) return s.status;
  if (sigma) {
    sigma[0] = s.sigma.real();
    sigma[1] = s.sigma.imag();
  }
  if (flags) {
    flags[0] = s.is_complex;
    flags[1] = s.tensorial;
    flags[2] = s.has_mu;
    flags[3] = s.coef_complex;
  }
  if (target) *target = s.target;
  if (knorm) *knorm = s.knorm;
  for (int a = 0; a < 2; ++a) {
    double *dst = a == 0 ? coef_x : coef_y;
    if (!dst) continue;
    std::vector<cd> c;
    s.ax[a].coefficients(c);
    for (size_t i = 0; i < c.size(); ++i) {
      dst[2 * i] = c[i].real();
      dst[2 * i + 1] = c[i].imag();
    }
  }
  if (fields) {
    const size_t n = (size_t)s.nx * s.ny;
    for (int q = 0; q < 6; ++q)
      for (size_t i = 0; i < n; ++i) {
        fields[2 * (q * n + i)] = s.f(q)[i].real();
        fields[2 * (q * n + i) + 1] = s.f(q)[i].imag();
      }
  }
  return s.status;
}

extern "C" int b200ms_debug_hierarchy(const b200ms_problem *prob, const b200ms_options *opt, int max_levels, int *shapes) {
  if (!prob || !shapes) return -1;
  b200ms_options o;
  b200ms_default_options(&o);
  if (opt) o = *opt;
  ProblemSetup s;
  setup_problem(*prob, s);
  if (s.status != B200MS_OK && s.status != B200MS_ERR_UNSUPPORTED) return -1;
  double kh_limit = 0.0, kmax = 0.0;
  if (s.max_k2 > 1e-6 && o.mg_ppw > 0) {
    kmax = std::sqrt(s.max_k2);
    kh_limit = 2.0 * M_PI / o.mg_ppw;
  }
  HierarchyPlan plan;
  plan_hierarchy(s.ax, o.mg_min_size, 12, kh_limit, kmax, plan);
  int n = std::min<int>(max_levels, (int)plan.nx.size());
  for (int l = 0; l < n; ++l) {
    shapes[2 * l] = plan.nx[l];
    shapes[2 * l + 1] = plan.ny[l];
  }
  return (int)plan.nx.size();
}

extern "C" int b200ms_debug_march2_geometry(int nx, int ny, int nbatch, int resident_ctas, int *cta_width, int *nstrips, int *rows) {
  if (nx < 1 || ny < 2 || (ny & 1) || nbatch < 1 || !cta_width || !nstrips || !rows) return B200MS_ERR_ARG;
  march2_strips(ny, *cta_width, *nstrips);
  *rows = march2_rows(nx, *nstrips, nbatch, resident_ctas);
  return B200MS_OK;
}

extern "C" int b200ms_debug_grid_factors(const b200ms_problem *prob, const double *n_complex, double *primal, double *dual) {
  if (!prob || !n_complex || !primal || !dual || prob->num_modes < 1) return B200MS_ERR_ARG;
  std::vector<zc> gp, gd;
  grid_factors(*prob, n_complex, gp, gd);
  for (int m = 0; m < prob->num_modes; ++m) {
    primal[2 * m] = gp[m].real(); primal[2 * m + 1] = gp[m].imag();
    dual[2 * m] = gd[m].real(); dual[2 * m + 1] = gd[m].imag();
  }
  return B200MS_OK;
}

// |E1|^2, |E2|^2 at the px x py colocation points of an angled plane exactly as post_scan_kernel evaluates them (same functions):
// e = px x py x {Ex, Ey, Ez} complex (re,im), point (p, q) at e + 6 (p py + q); out = px x py x {te, tm}
extern "C" int b200ms_debug_te_terms(const double *e, int px, int py, double angle_theta, double angle_phi, int symx, int symy, double *out) {
  if (!e || !out || px < 0 || py < 0) return -1;
  const double ct = std::cos(angle_theta), st = std::sin(angle_theta), cp = std::cos(angle_phi), sp = std::sin(angle_phi);
  for (int p = 0; p < px; ++p)
    for (int q = 0; q < py; ++q) {
      const size_t i = (size_t)p * py + q;
      const double *v = e + 6 * i;
      double kxy, kxz, kyz;
      te_point_flags(symx, symy, p, q, kxy, kxz, kyz);
      te_tm_terms(mk(v[0], v[1]), mk(v[2], v[3]), mk(v[4], v[5]), ct, st, cp, sp, kxy, kxz, kyz, out[2 * i], out[2 * i + 1]);
    }
  return 0;
}

extern "C" int b200ms_debug_post_tables_bounded(const double *coords, int n, int sym, double lo, double hi, int max_points, int *idx,
                                                double *wgt, double *area);
extern "C" int b200ms_debug_post_tables(const double *coords, int n, int sym, int max_points, int *idx, double *wgt, double *area) {
  return b200ms_debug_post_tables_bounded(coords, n, sym, -HUGE_VAL, HUGE_VAL, max_points, idx, wgt, area);
}
extern "C" int b200ms_debug_post_tables_bounded(const double *coords, int n, int sym, double lo, double hi, int max_points, int *idx,
                                                double *wgt, double *area) {
  if (!coords || n < 1 || !idx || !wgt || !area) return -1;
  HostAxisTables t;
  const double bounds[2] = {lo, hi};
  axis_tables(coords, n, sym, t, bounds);
  if (t.P > max_points) return -1;
  for (int p = 0; p < t.P; ++p) {
    idx[4 * p] = t.ci0[p]; idx[4 * p + 1] = t.ci1[p]; idx[4 * p + 2] = t.bi0[p]; idx[4 * p + 3] = t.bi1[p];
    wgt[4 * p] = t.cw0[p]; wgt[4 * p + 1] = t.cw1[p]; wgt[4 * p + 2] = t.bw0[p]; wgt[4 * p + 3] = t.bw1[p];
    area[p] = t.area[p];
  }
  return t.P;
}

// ---- device debug hooks -------------------------------------------------------------------------------
namespace {
template <typename T, typename C, typename P, typename PC>
int debug_run(b200ms_handle *h, const Window &W, int what, int level, int mode, const double *in0, const double *in1,
              double *out, int *iters, double *relres) {
  std::vector<const ProblemSetup *> ps(1, &W.setups[0]);
  std::vector<MediumRef> refs(1, W.refs[0]);
  BatchSolver<T, C, P, PC> S(h->arena, h->stream, h->opt);
  S.build(ps, false, upload_refs(h, refs, h->stream));
  if (what == 0 && mode >= 16) {  // mode + 16: the multigrid operator (preconditioner precision) also on level 0
    mode -= 16;
    if (level == 0 && mode != 3) level = -1000;
  }
  if (what == 0 && (level > 0 || level == -1000 || mode == 3)) {  // multigrid operator of level `level` in preconditioner precision
    if (level == -1000) level = 0;
    if (level < 0 || level >= (int)S.lv.size()) return B200MS_ERR_ARG;
    const size_t n2 = 2 * S.lv[level].N;
    std::vector<P> a(n2), b(n2), o(n2);
    for (size_t e = 0; e < n2; ++e) {
      a[e] = from_cd<P>(cd(in0[2 * e], in0[2 * e + 1]));
      b[e] = in1 ? from_cd<P>(cd(in1[2 * e], in1[2 * e + 1])) : zero_of<P>();
    }
    P *d0 = reinterpret_cast<P *>(S.basis0()), *d1 = d0 + S.vstride, *d2 = d0 + 2 * S.vstride;
    CUDA_CHECK(cudaMemcpy(d0, a.data(), n2 * sizeof(P), cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(d1, b.data(), n2 * sizeof(P), cudaMemcpyHostToDevice));
    if (mode == 3) S.jacobi0(level, d1, d2);
    else S.apply(level, mode, d0, d1, d2);
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaMemcpy(o.data(), d2, n2 * sizeof(P), cudaMemcpyDeviceToHost));
    for (size_t e = 0; e < n2; ++e) {
      cd v = to_cd(o[e]);
      out[2 * e] = v.real();
      out[2 * e + 1] = v.imag();
    }
    return B200MS_OK;
  }
  if (level < 0 || level >= (int)S.lv.size()) return B200MS_ERR_ARG;
  const size_t n2 = what == 0 ? 2 * S.lv[level].N : S.len;
  std::vector<T> a(n2), b(n2);
  for (size_t e = 0; e < n2; ++e) {
    a[e] = from_cd<T>(cd(in0[2 * e], in0[2 * e + 1]));
    b[e] = in1 ? from_cd<T>(cd(in1[2 * e], in1[2 * e + 1])) : zero_of<T>();
  }
  T *d0 = S.basis0(), *d1 = S.basis0() + S.vstride, *d2 = S.basis0() + 2 * S.vstride;
  CUDA_CHECK(cudaMemcpy(d0, a.data(), n2 * sizeof(T), cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMemcpy(d1, b.data(), n2 * sizeof(T), cudaMemcpyHostToDevice));
  if (what == 0) {
    S.apply_true(mode, d0, d1, d2);
  } else if (what == 1) {
    S.precondition(d0, d2);
  } else {
    int it = 0;
    double rr = S.fgmres(d0, d2, it);
    if (iters) *iters = it;
    if (relres) *relres = rr;
  }
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  CUDA_CHECK(cudaGetLastError());
  std::vector<T> o(n2);
  CUDA_CHECK(cudaMemcpy(o.data(), d2, n2 * sizeof(T), cudaMemcpyDeviceToHost));
  for (size_t e = 0; e < n2; ++e) {
    cd v = to_cd(o[e]);
    out[2 * e] = v.real();
    out[2 * e + 1] = v.imag();
  }
  return B200MS_OK;
}

int debug_dispatch(b200ms_handle *h, const b200ms_problem *prob, int what, int level, int mode, const double *in0,
                   const double *in1, double *out, int *iters, double *relres) {
  if (!h || !prob || !in0 || !out) return B200MS_ERR_ARG;
  if (cudaSetDevice(h->device) != cudaSuccess) return B200MS_ERR_CUDA;
  try {
    Window W;
    prepare_window(h, prob, 0, 1, h->raw[0], h->stream, W);
    const ProblemSetup &s = W.setups[0];
    if (s.status != B200MS_OK) {
      h->err = s.error;
      return s.status;
    }
    switch (kind_of(s)) {
      case 0: return debug_run<double, double, float, float>(h, W, what, level, mode, in0, in1, out, iters, relres);
      case 1: return debug_run<cplx, double, cplxf, float>(h, W, what, level, mode, in0, in1, out, iters, relres);
      default: return debug_run<cplx, cplx, cplxf, cplxf>(h, W, what, level, mode, in0, in1, out, iters, relres);
    }
  } catch (const std::exception &e) {
    h->err = e.what();
    return B200MS_ERR_CUDA;
  }
}
}  // namespace

extern "C" int b200ms_debug_apply(b200ms_handle *h, const b200ms_problem *prob, int level, int mode, const double *x,
                                  const double *rhs, double *y) {
  return debug_dispatch(h, prob, 0, level, mode, x, rhs, y, nullptr, nullptr);
}
extern "C" int b200ms_debug_vcycle(b200ms_handle *h, const b200ms_problem *prob, const double *r, double *z) {
  return debug_dispatch(h, prob, 1, 0, 0, r, nullptr, z, nullptr, nullptr);
}
extern "C" int b200ms_debug_solve(b200ms_handle *h, const b200ms_problem *prob, const double *b, double *x, int *iters,
                                  double *relres) {
  return debug_dispatch(h, prob, 2, 0, 0, b, nullptr, x, iters, relres);
}
