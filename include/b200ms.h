/*
 * b200ms.h -- C ABI of the B200-native waveguide mode solver (libb200ms.so).
 *
 * Drop-in boundary for the hot path of flexcompute/tidy3d's local mode solver.  Every entry point
 * names the reference interface it replaces (paths relative to the tidy3d tree):
 *
 *   b200ms_solve_batch   <->  tidy3d/plugins/mode/solver.py:941 `compute_modes(eps_cross, coords,
 *                             freq, mode_spec, mu_cross, split_curl_scaling, symmetry, direction,
 *                             solver_basis_fields)` == EigSolver.compute_modes (solver.py:33-269),
 *                             called once per frequency by ModeSolver._solve_single_freq
 *                             (tidy3d/plugins/mode/mode_solver.py:725); a batch corresponds to the
 *                             frequency loop ModeSolver._solve_all_freqs (mode_solver.py:655-672).
 *   b200ms_problem       <->  the argument list above; mode_spec fields as read at
 *                             solver.py:86-90,198,204,247 (tidy3d/components/mode.py:18-209).
 *   b200ms_result        <->  the returned tuple (fields[2,3,Nx,Ny,1,M], n_complex[M], eps_spec)
 *                             (solver.py:257-269), plus what the reference does not return: on-device
 *                             post-processing results and the permittivity gradient dn/deps (grad_eps).
 *   error codes          <->  ValueError / RuntimeError raised at solver.py:107, 876, 901.
 *
 * Plain C types only (no torch, no C++).  Host pointers in and out; the library owns all device
 * memory and one CUDA stream per handle.  One handle per GPU; calls on one handle must not overlap.
 * There is no CPU fallback: without a usable CUDA device b200ms_create fails with B200MS_ERR_CUDA.
 */
#ifndef B200MS_H
#define B200MS_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200MS_VERSION 205

/* return codes */
enum {
  B200MS_OK = 0,
  B200MS_ERR_SHAPE = 1,       /* ValueError: "Mismatch between 'coords' and 'esp_cross' shapes." (solver.py:107).  Reserved for the
                                 language binding: the C arrays carry no lengths (nx, ny are stated once and every array is
                                 sized from them), so only the binding that still holds the caller's arrays can see a mismatch
                                 (tidy3d_b200/_cabi.py PackedProblem raises it before the call) */
  B200MS_ERR_NO_MODES = 2,    /* RuntimeError: "Could not find any eigenmodes for this waveguide." (solver.py:876: an EMPTY result of
                                 scipy's eigs).  Reserved: a shift-invert run that finds fewer than num_modes pairs reports
                                 B200MS_ERR_NOCONV, as scipy raises ArpackNoConvergence before the reference reaches :876 */
  B200MS_ERR_UNSUPPORTED = 3, /* combination the reference itself rejects (tensorial eps + basis fields, solver.py:357-361) or that is
                                 outside the built scope (basis fields together with removed PEC unknowns) */
  B200MS_ERR_CUDA = 4,        /* CUDA runtime failure or no device -- never falls back to the CPU */
  B200MS_ERR_NOCONV = 5,      /* eigen-iteration did not converge (scipy ArpackNoConvergence analogue) */
  B200MS_ERR_ARG = 6          /* bad argument (null pointer, num_modes < 1, ...) */
};

/* eps_spec values, solver.py:364,376,383 */
enum { B200MS_SPEC_DIAGONAL = 0, B200MS_SPEC_TENSORIAL_REAL = 1, B200MS_SPEC_TENSORIAL_COMPLEX = 2 };

typedef struct b200ms_handle b200ms_handle;

/* A cross-section described by geometry instead of a sampled permittivity array: what ModeSolver._solver_eps builds on the
 * host with nine Simulation.epsilon_on_grid calls per frequency (mode_solver.py:587-653, simulation.py:1135-1241) is
 * rasterised on the device.  epsilon_on_grid starts from the background medium and lets every structure, in order, overwrite
 * the Yee sites its geometry contains (simulation.py:1191-1226); eps_xx, eps_xy, eps_xz are sampled at the Ex site (cell
 * centre in x, lower boundary in y), eps_y* at the Ey site, eps_z* at the Ez site (simulation.py:1231-1236).  Two ways to say
 * where the media are, which may be combined:
 *   - a list of primitive shapes in the solver plane (the cuts of Box / Cylinder / Sphere / PolySlab structures), later
 *     entries override earlier ones;
 *   - `site_medium`, a per-site medium index the CALLER evaluated once per plane with the reference's own
 *     Geometry.inside_meshgrid (any geometry: the map does not depend on the frequency); the listed shapes then draw on
 *     top of it.  Either way only 9 numbers per medium change from one frequency to the next. */
enum {
  B200MS_SHAPE_RECT = 0,    /* row: center_x, center_y, size_x, size_y; inside when |x - cx| <= sx/2 and |y - cy| <= sy/2
                               (Box.inside, components/geometry/base.py:2042-2068) */
  B200MS_SHAPE_DISC = 1,    /* row: center_x, center_y, radius, dz; inside when |x-cx|^2 + |y-cy|^2 + dz^2 <= radius^2: the cut of a
                               Cylinder whose axis is the plane normal (dz = 0; Cylinder.inside, geometry/primitives.py:600-632) or
                               of a Sphere whose centre lies dz off the plane (Sphere.inside, primitives.py:44-70) */
  B200MS_SHAPE_POLYGON = 2  /* row unused; vertices poly_xy[poly_start[i] .. poly_start[i+1]): the cut of a PolySlab whose axis is the
                               plane normal (vertical side walls), or the trapezoid a slanted-wall slab shows in a plane containing
                               its axis.  Even-odd crossing rule; like the reference's matplotlib Path.contains_points
                               (polyslab.py:509-516) the result for a point exactly ON an edge is unspecified */
};
typedef struct {
  int nrect;               /* number of shapes */
  const double *rects;     /* nrect x 4 doubles, meaning per shape kind above */
  const int *medium;       /* nrect: row of eps_table used inside each shape */
  int nmedia;              /* rows of eps_table; row 0 is the background medium */
  const double *eps_table; /* nmedia x 9 complex128 (re,im): relative permittivity tensor (xx,xy,...,zz) of each medium AT THIS
                              PROBLEM'S FREQUENCY (dispersive media are evaluated by the caller: 9 numbers per medium) */
  /* ---- since version 201 (all may be NULL: a list of rectangles, as in version 200) ---- */
  const int *shape;        /* NULL (every shape is a rectangle) or nrect kinds B200MS_SHAPE_* */
  const int *poly_start;   /* NULL without polygons, else nrect + 1 offsets (in vertices) into poly_xy */
  const double *poly_xy;   /* polygon vertices, (x, y) pairs in plane coordinates */
  const unsigned short *site_medium; /* NULL, or 3*nx*ny medium indices [Ex sites | Ey sites | Ez sites], each C-order with y fastest:
                              the medium found at every Yee site before the listed shapes are drawn (replaces "background
                              everywhere").  Indices >= nmedia are a caller error (clamped to nmedia - 1 on the device) */
} b200ms_section;

/* One eigenproblem == one compute_modes call (one plane, one frequency). */
typedef struct {
  int nx, ny;            /* eps_cross[i].shape */
  int num_modes;         /* mode_spec.num_modes */
  int num_pml[2];        /* mode_spec.num_pml */
  int symmetry[2];       /* 0 none, +1 PMC, -1 PEC at the min wall (solver.py:184,197) */
  int bend_axis;         /* mode_spec.bend_axis, ignored when bend_radius is NaN */
  int direction;         /* +1 "+", -1 "-" */
  int precision;         /* mode_spec.precision: 0 double, 1 single.  single: result.fields is a complex64 buffer (solver.py:265-267);
                            the eigenproblem itself is always solved to the handle's tolerances */
  int incidence;         /* 1 when the caller passed mu_cross or split_curl_scaling (solver.py:93 enable_incidence_matrices): Ex/Ey
                            unknowns on PEC-valued cells are removed and 1/eps_zz is zeroed there (solver.py:441-449, 474-477,
                            506-508, 568-569); no effect without PEC-valued cells */
  int post;              /* on-device post-processing of the fields before delivery (ModeSolver.data_raw steps, solver-plane
                            coordinates): bit 0 = gauge (largest in-plane E entry real positive, mode_solver.py:802-810), bit 1 =
                            flux normalisation (fields / sqrt|flux|, mode_solver.py:517-521 with monitor_data.py:582-618) */
  double freq;           /* Hz */
  double target_neff;    /* NaN == None */
  double bend_radius;    /* NaN == None */
  double angle_theta, angle_phi;
  const double *eps;     /* 9*nx*ny complex128 as interleaved (re,im), component-major xx,xy,...,zz,
                            each component C-order with y fastest (solver.py:890-901); NULL when `section` is given */
  const double *coords_x; /* nx+1 */
  const double *coords_y; /* ny+1 */
  const double *mu;      /* NULL (identity), or the relative permeability `mu_cross` (solver.py:62-66, 128-136) in the same
                            9*nx*ny complex128 layout as eps */
  const b200ms_section *section; /* NULL, or the geometric description the permittivity is rasterised from (eps == NULL) */
  const double *basis_e; /* NULL, or the in-plane E part of `solver_basis_fields` (solver.py:219-236, 750-776):
                            2*nx*ny*num_modes complex128 (re,im) laid out [Ex|Ey][ix][iy][mode]; the modes are then
                            computed as linear combinations of this basis (relative mode solver) */
  const double *grid_correction; /* since version 202.  NULL (factors 1), or 8 doubles {dp0, wp0, dp1, wp1, dd0, wd0, dd1, wd1} from which the
                            finite-grid correction factors of ModeSolver._grid_correction (mode_solver.py:847-904) are formed for every
                            mode once its n_complex is known: with k = 2 pi n_complex freq / C_0 / cos(angle_theta) (negated for
                            direction "-"), primal = wp0 exp(i k dp0) + wp1 exp(i k dp1) multiplies the tangential E, dual (dd*, wd*)
                            the tangential H in the flux and in the modal overlaps (monitor_data.py:488-503).  dp* / dd*: offsets
                            along the plane normal (um) from the mode plane to the two simulation-grid boundaries / centres that
                            bracket it, w*: the linear interpolation weights (one grid point only: {d, 1, 0, 0}).  Only the
                            post-processing results (post bit 1, flux, overlap_prev) depend on it; the fields themselves do not */
  const double *plane_bounds; /* since version 203.  NULL (nothing is truncated), or 4 doubles {xmin, xmax, ymin, ymax}: the extent of a
                            finite mode plane in plane coordinates (of the full, mirrored plane when a symmetry wall is present).
                            The trapezoid weights of flux, TE fraction and modal overlaps are then truncated to the part of each
                            cell the plane covers, like the reference's _diff_area (monitor_data.py:437-455: mid-points and end
                            points clipped to monitor.bounds).  Only the post-processing results depend on it */
} b200ms_problem;

typedef struct {
  double *fields;        /* caller-allocated 2*3*nx*ny*1*num_modes complex128 (re,im) -- complex64 when precision == 1 --, reference
                            layout [E/H][comp][ix][iy][0][mode]; HOST or DEVICE memory (unified addressing; a device buffer
                            keeps the fields in HBM for an NCCL gather or on-device post-processing); NULL skips the fields */
  double *n_complex;     /* caller-allocated num_modes complex128 (re,im): n_eff + i k_eff */
  double *flux;          /* NULL, or caller-allocated num_modes doubles: flux of every mode BEFORE normalisation (colocated
                            tangential fields, trapezoid weights; monitor_data.py:523-539, 425-467, 582-618) */
  double *te_fraction;   /* NULL, or caller-allocated num_modes doubles: TE polarisation fraction int|E1|^2 / int(|E1|^2+|E2|^2) of the
                            colocated field (ModeData.pol_fraction, monitor_data.py:1625-1652), the input of the filter_pol re-ordering
                            (mode_solver.py:523-549); for angle_theta / angle_phi != 0 the field is first rotated to the propagation
                            axes like the reference does (monitor_data.py:1603-1607) and, with a symmetry wall, the integral is
                            that over the symmetry-expanded plane: products of components of opposite parity, which the rotation
                            creates, cancel between a point and its mirror image and are left out (except on the wall itself) */
  double *overlap_prev;  /* NULL, or caller-allocated num_modes^2 complex128 (re,im), row-major [m_prev][m]: modal overlap
                            dot(mode m_prev of the PREVIOUS problem of this call, mode m of this one) (monitor_data.py:640-697,
                            after gauge/normalisation), the input of overlap_sort (monitor_data.py:1295-1375).  Zeros when
                            there is no previous problem or its shape / num_modes / precision differ */
  int eps_spec;          /* out: B200MS_SPEC_* */
  int status;            /* out: per-problem B200MS_* code */
  int converged;         /* out: number of converged modes */
  int outer_iters;       /* out: Krylov-Schur restarts */
  int op_applies;        /* out: shift-invert (OP^-1) applications */
  int inner_iters;       /* out: total preconditioned GMRES iterations */
  int stencil_applies;   /* out: kernels launched for this batch (all kinds) */
  int is_complex;        /* out: 1 if the eigenproblem was solved in complex arithmetic (solver.py:389-411) */
  double solve_ms;       /* out: device time (CUDA events) of the eigen-solve + field recovery of the batch this problem
                            was in, operator data already resident in HBM, results still on the device */
  double total_ms;       /* out: host wall time of that batch incl. upload of the operator and download of the fields */
  double max_residual;   /* out: max_i ||A v_i - lambda_i v_i|| / (|lambda_i| ||v_i||) */
  /* ---- since version 205 ---- */
  double *grad_eps;      /* NULL, or caller-allocated num_modes*3*nx*ny complex128 (re,im), HOST or DEVICE memory like `fields`:
                            d n_complex[m] / d eps_cc[ix][iy] for c = xx, yy, zz, layout [mode][c][ix][iy] (y fastest), from the
                            left eigenvector of the diagonal operator (DESIGN.md section 10; no extra solve, works without
                            `fields`).  Diagonal problems only: a problem that asks for it and is tensorial / angled, bent, has
                            mu / split_curl_scaling (incidence), basis fields or PEC-valued cells gets status
                            B200MS_ERR_UNSUPPORTED before it is solved; the other problems of the call are unaffected */
} b200ms_result;

/* Tunables (all have defaults; see DESIGN.md). */
typedef struct {
  double eig_tol;        /* relative Ritz residual tolerance; default 1.19e-7 = the reference's ARPACK tol (solver.py:20,745);
                            the "tight" setting used by the parity tests is 1e-9 */
  double inner_tol;      /* relative residual of the shift-invert solves before relaxation (default 1e-8; tight 1e-10) */
  int ncv;               /* Krylov subspace size, 0 = max(2k+1, 20) like scipy (solver.py:744) */
  int max_restarts;      /* default 500 */
  int gmres_restart;     /* default 40 */
  int gmres_maxit;       /* default 400 */
  int mg_nu;             /* Jacobi pre/post sweeps (default 2) */
  int mg_min_size;       /* stop coarsening below this many cells per axis (default 12) */
  int mg_coarse_iters;   /* Krylov iterations on the coarsest level (default 16) */
  int max_batch;         /* problems solved concurrently on the device (default 64: 5120 CTAs of the fp64 apply = 4.94 waves on 148 SMs) */
  double mg_omega;       /* Jacobi damping (default 0.8) */
  double mg_ppw;         /* indefinite problems: keep >= this many cells per local wavelength (default 4) */
  int verbose;
  double mg_pml_phase;   /* multigrid operator: clamp |arg| of the PML stretch to this (default pi/4; <=0: off) */
  double inner_relax;    /* inexact shift-invert: inner tol = clamp(inner_relax * inner_tol / ritz_residual); 0 = off (default 1.0) */
  double inner_relax_cap; /* loosest inner tolerance allowed (default 1e-4) */
  int gmres_cgs2;        /* inner FGMRES Gram-Schmidt: 1 always two passes (CGS2); 0 one pass (+ a second on cancellation; measured 3x more
                            iterations at tol 1e-10); 2 (default) one pass while all residuals are > 3e-6, CGS2 below */
  int mg_nu_growth;      /* extra Jacobi sweeps per coarser level (variable V-cycle), default 0 */
  int use_graph;         /* 1 (default): replay the multigrid V-cycle as one CUDA graph */
  int mg_cycles;         /* V-cycles per preconditioner application (default 1) */
  int inner_ir;          /* 1 (default): run the FGMRES cycles in the multigrid precision (fp32) inside an fp64 iterative
                            refinement (diagonal path); 0: fp64 cycles */
  double ir_floor;       /* smallest residual reduction asked of one fp32 cycle (default 1e-4) */
  double ir_trust;       /* solves whose tolerance is >= this accept the fp32 residual estimate without an fp64 check (3e-5) */
  double inner_relax_complex; /* complex-arithmetic problems: loosest inner tolerance = this x inner_tol (default 50) */
  int mg_fuse_first;     /* 1 (default): the first two pre-smoothing sweeps (from the zero guess) run as one kernel pass */
  int ks_keep;           /* Krylov-Schur: Ritz vectors kept at a restart; 0 (default) = k + (ncv - k) / 2 */
  double cluster_gap;    /* a wanted Ritz value closer than this (relative) to another Ritz value disables the relaxation of the inner
                            tolerance for that problem (default 1e-3) */
  int mg_fused_tail;     /* 1 (default): the multigrid levels that fit in shared memory together (<= 64^2 cells) run as one kernel, one
                            CTA per problem (csrc/coarse_kernel.cuh); 0: one kernel per operation on every level */
  double kappa_cap;      /* the Ritz residual of a wanted pair is weighted by min(kappa, kappa_cap), kappa = condition number of the
                            Ritz value in the projected problem, before the comparison with eig_tol (default 1e4; 1 = ARPACK's test) */
  int outer_dgks;        /* 1 (default): Krylov-Schur orthogonalisation reorthogonalises only when ARPACK's DGKS test asks for it;
                            0: always two Gram-Schmidt passes */
  int stencil_pair;      /* 1 (default): pair-marching stencil kernels for the real fp32 multigrid operators on even-width levels (two columns
                            per thread, 64-bit accesses, CTA width fitted to the row, six-fold unrolled row loop): rows staged by TMA bulk
                            copies (cp.async.bulk + mbarrier, ring of three stages, csrc/march2_tma.cuh) where ny % 4 == 0 outside the fused
                            first sweeps, prefetched into two sets of registers (csrc/march2.cuh) elsewhere; 0: the one-column marching
                            kernel everywhere */
  int stencil_pair_rows; /* rows marched per CTA by the pair kernel (rounded to 6 m - 3); 0 (default) = chosen per level from the
                            number of resident CTAs */
  int transfer_vec;      /* multigrid transfers: bit 0 = the prolongation reads / writes its four fine values as one 128-bit access (fp32 vectors,
                            nyf % 4 == 0); bit 1 = the restriction reads each fine row of its patch as aligned 64-bit pairs when the patch is
                            contiguous */
  int tensor_mg_cycles;  /* tensorial path: V-cycles (defect correction on the multigrid operator) per application of the E-block inverse inside
                            the block preconditioner; 0 = mg_cycles.  Default 3 (see csrc/solver.cuh mg_cycles_ and tools/proto_tensor.py) */
} b200ms_options;

/* Counters of the most recent b200ms_solve_batch call on a handle (all its device batches together). */
typedef struct {
  double device_ms;      /* sum over device batches of the CUDA-event window "operator resident in HBM -> results in HBM" */
  double setup_ms;       /* host wall time spent on upload + problem set-up + hierarchy build */
  double download_ms;    /* host wall time spent delivering the fields */
  double total_ms;       /* host wall time of the whole call */
  long long launches;    /* kernels launched (CUDA-graph nodes counted individually) */
  long long inner_iters; /* sum over problems of the FGMRES iterations each went through */
  long long op_applies;  /* sum over problems of shift-invert applications */
  long long host_syncs;  /* stream synchronisations inside the inner solves, summed over device batches */
  int device_batches;    /* how many device batches the call was split into */
  int nprob;
} b200ms_stats;

int b200ms_version(void);
void b200ms_default_options(b200ms_options *opt);
/* device < 0: use cudaGetDevice() */
int b200ms_create(int device, b200ms_handle **out);
int b200ms_destroy(b200ms_handle *h);
int b200ms_set_options(b200ms_handle *h, const b200ms_options *opt);
const char *b200ms_last_error(b200ms_handle *h);
int b200ms_get_stats(b200ms_handle *h, b200ms_stats *out);

/* Page-locked host memory for result buffers (optional): fields written into memory from b200ms_host_alloc are copied
 * device->host at full PCIe/C2C speed instead of through the driver's pageable staging path. */
void *b200ms_host_alloc(size_t bytes);
void b200ms_host_free(void *ptr);

/* Solve nprob independent eigenproblems.  Problems with identical (nx, ny, arithmetic) are batched on
 * the device.  Returns B200MS_OK if every problem succeeded, else the first failing status (each
 * result carries its own status). */
int b200ms_solve_batch(b200ms_handle *h, int nprob, const b200ms_problem *prob, b200ms_result *res);

/* Benchmark / roofline hook: run one of the two hot stencil kernels `nrep` times on `nbatch` device-resident copies
 * of the operator of `prob` and return the mean kernel time (CUDA events on the library stream).
 * mode 0: y = (A - sigma) x, the fp64 operator apply of the Krylov iteration; mode 1: the production smoother sweep
 * (stored-diagonal Jacobi in the multigrid precision); mode 2: one fused CGS2 Gram-Schmidt step of the inner solver against
 * four basis vectors in the multigrid precision (gs_dots, gs_update_dots, gs_update_norm, gs_scale: 19 vector passes); mode 3: the two
 * permittivity-gradient kernels (csrc/sensitivity.cuh) for prob.num_modes modes, N*M*(2*(2*s_v + 3*s_c) + 48) bytes per problem.  x (2*nx*ny complex128 (re,im)) may be NULL (random); y may be
 * NULL.  bytes_per_apply returns the algorithmic bytes of one launch (SURVEY 8(d)): N*(4*s_v + nf*s_c) per problem for
 * the apply, N*(8*s_v + nf*s_c) for the sweep. */
int b200ms_bench_stencil(b200ms_handle *h, const b200ms_problem *prob, int nbatch, int mode, int nrep,
                         int flush_l2, const double *x, double *y, double *ms_per_launch,
                         double *bytes_per_apply);

/* ---- host-only debug hooks (no GPU needed; used by the CPU test-suite) ---------------------- */
/* complex Schur decomposition A = Q T Q^H of an n x n row-major complex matrix (re,im) */
int b200ms_debug_schur(int n, const double *a, double *t, double *q);
/* problem set-up as the solver sees it: writes sigma (re,im), flags[4] = {is_complex, tensorial,
 * has_mu, eps_is_complex}, target, knorm, 1-D coefficient vectors coef_x[8*nx] / coef_y[8*ny]
 * (f0,f1,b0,bm complex) and fields[6*nx*ny] complex (exx,eyy,ezz,mxx,myy,mzz). NULL outputs skipped. */
int b200ms_debug_setup(const b200ms_problem *prob, double *sigma, int *flags, double *target,
                       double *knorm, double *coef_x, double *coef_y, double *fields);
/* the permittivity gradient of one mode of `prob` from a given eigenvector, by the functions the device kernel calls
 * (csrc/sensitivity.cuh): vec = 2*nx*ny complex (re,im) [Ex|Ey] in solver units, lambda = its eigenvalue (re,im) of A = P Q
 * (-n^2), out = 3*nx*ny complex (re,im) dn/deps_{xx,yy,zz}.  B200MS_ERR_UNSUPPORTED outside the scope of grad_eps */
int b200ms_debug_sensitivity(const b200ms_problem *prob, const double *vec, const double *lambda, double *out);
/* multigrid hierarchy shapes for a problem: writes up to max_levels (nx,ny) pairs, returns count */
int b200ms_debug_hierarchy(const b200ms_problem *prob, const b200ms_options *opt, int max_levels,
                           int *shapes);

/* launch geometry of the pair-marching stencil kernels (csrc/march2.cuh) for an nx x ny level of `nbatch` problems on a device
 * that keeps `resident_ctas` of them resident: threads per CTA (column pairs per strip), strips per row, rows marched per CTA */
int b200ms_debug_march2_geometry(int nx, int ny, int nbatch, int resident_ctas, int *cta_width, int *nstrips, int *rows);

/* the finite-grid correction factors (b200ms_problem.grid_correction) the post-processing applies to the modes of `prob` given
 * their n_complex (num_modes complex (re,im)): primal / dual, num_modes complex (re,im) each */
int b200ms_debug_grid_factors(const b200ms_problem *prob, const double *n_complex, double *primal, double *dual);

/* the 1-D tables of the on-device post-processing for one axis of n cells (coords: n + 1 boundaries; sym: the problem's
 * symmetry value for that axis): colocation points (interior boundaries, plus the symmetry plane), and for each of them the
 * two source indices / weights of the linear interpolation from the centre sites and from the boundary sites of the
 * symmetry-expanded data, and its trapezoid weight.  idx / wgt: 4 per point {centre i0, centre i1, boundary i0, boundary i1};
 * returns the number of points, -1 on bad arguments or when max_points is too small */
int b200ms_debug_post_tables(const double *coords, int n, int sym, int max_points, int *idx, double *wgt, double *area);
/* |E1|^2 and |E2|^2 (the integrands of te_fraction) at the px x py colocation points of an angled plane, evaluated by the very
 * functions the device kernel calls: e = px x py x {Ex, Ey, Ez} complex (re,im), symx / symy the problem's symmetry values (the
 * first point along an axis with a symmetry wall is the wall itself), out = px x py x {te, tm} */
int b200ms_debug_te_terms(const double *e, int px, int py, double angle_theta, double angle_phi, int symx, int symy, double *out);
/* the same with the extent [lo, hi] of a finite mode plane along this axis (b200ms_problem.plane_bounds) */
int b200ms_debug_post_tables_bounded(const double *coords, int n, int sym, double lo, double hi, int max_points, int *idx, double *wgt,
                                     double *area);

/* ---- device debug hooks (GPU tests compare these against the numpy model) ------------------- */
/* y = (A - sigma) x on level `level` of the hierarchy of `prob`; x,y complex128 2*nxl*nyl */
int b200ms_debug_apply(b200ms_handle *h, const b200ms_problem *prob, int level, int mode,
                       const double *x, const double *rhs, double *y);
/* one multigrid V-cycle z = M^-1 r on the fine level */
int b200ms_debug_vcycle(b200ms_handle *h, const b200ms_problem *prob, const double *r, double *z);
/* x = (A - sigma)^-1 b by preconditioned FGMRES; returns iterations and relative residual */
int b200ms_debug_solve(b200ms_handle *h, const b200ms_problem *prob, const double *b, double *x,
                       int *iters, double *relres);

#ifdef __cplusplus
}
#endif
#endif /* B200MS_H */
