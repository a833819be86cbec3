/* libtemd — C ABI of the B200-native zonal-mean + TEM hot path (drop-in for jhollowed/PyTEMDiags).
 *
 * The reference is pure Python (no FFI); the entry points below are the operations its two public
 * classes perform on the hot path, i.e. what a ctypes binding inside the reference would call
 * (INTEGRATION.md shows that binding).  Reference citations are paths under PyTEMDiags/.
 *
 * Conventions
 *   - every array pointer is a DEVICE pointer (float64) unless the name ends in `_host`;
 *   - field layout is [row][ncol] with row = time*nlev + lev ("[time][lev][ncol]", ncol contiguous),
 *     leading dimension `ld` >= ncol in elements, `ld` even, base 16-byte aligned (TMA);
 *   - coefficient blocks are [field][row][lpad], lpad = temd_plan_lpad() (L+1 rounded up to 8);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises
 *     except temd_basis_build (one status read-back) and temd_check_finite;
 *   - return value 0 = ok, < 0 = argument / numerical error, > 0 = cudaError_t;
 *     temd_last_error() returns a thread-local description.
 *   - inputs are borrowed read-only; the plan owns only its basis and one split-K workspace per stream: entry points
 *     are stream-ordered and re-entrant per (device, stream); they run on the plan's device and restore the caller's
 *     current device before returning.
 */
#ifndef TEMD_H
#define TEMD_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct temd_plan temd_plan;

int temd_version(void);
const char* temd_last_error(void);

/* sph_zonal_averager.__init__ (sph_zonal_mean.py:36-181): ncol = N native columns, L = max degree,
 * nlat_out = M output latitudes. */
int temd_plan_create(int device, int ncol, int L, int nlat_out, temd_plan** plan);
int temd_plan_destroy(temd_plan* plan);
int temd_plan_lpad(const temd_plan* plan);

/* Plan for temd_basis_build_min_norm: as temd_plan_create, but L+1 > ncol is allowed (a rank-deficient Y0 is then
 * certain; the de-duplicated plan lives on U < L+1 unique nodes whenever the grid has fewer latitudes than degrees). */
int temd_plan_create_min_norm(int device, int ncol, int L, int nlat_out, temd_plan** plan);

/* Number of whitened basis directions of the built plan: L+1 after temd_basis_build / _dedup / _weighted, the rank r
 * after temd_basis_build_min_norm; -1 if the basis is not built. */
int temd_plan_rank(const temd_plan* plan);

/* sph_zonal_averager.sph_compute_matrices (sph_zonal_mean.py:302-422): builds the Legendre basis at
 * x = cos(colatitude) of the native (x[N]) and output (x_out[M]) latitudes by three-term recurrence
 * (replaces sph_harm loops :359-370), the Gram matrix, its Cholesky factor, and the orthonormalised
 * basis that replaces Y0inv = lstsq(Y0, I) (:389).  Fails (<0) if Y0 is numerically rank-deficient.
 * sanity[0] = sum diag(Y0inv*Y0), sanity[1] = sum offdiag (the reference's logged check :393-398),
 * written to host memory if sanity_host != NULL. */
int temd_basis_build(temd_plan* plan, const double* x, const double* x_out, double* sanity_host, void* stream);

/* Minimum-norm least squares, for rank-deficient Y0 (e.g. more Legendre degrees than distinct latitudes): the result
 * is NumPy's np.linalg.lstsq(Y0, ., rcond=None), i.e. Y0inv = pinv(Y0) with singular values sigma_i <=
 * eps * max(N, L+1) * sigma_1 dropped (N = total column count, eps = 2^-52).  The rank decision comes from a one-sided
 * Jacobi SVD of Yw = diag(sqrt(mult)) Y0(x_unique) (same singular values and right singular vectors as Y0); the basis
 * is whitened with (V_r Sigma_r^-1)^T and re-orthonormalised by one Cholesky pass.  Coefficients r..lpad-1 are exactly
 * zero, so every other entry point runs unchanged at the plan's lpad.
 *   x        the plan's ncol nodes (dense plan), or NULL for a plan created on the unique nodes (the de-duplicated
 *            path: its basis is then the weighted unique grid of temd_basis_build_dedup, and nunique = ncol);
 *   x_unique, mult  the nunique distinct nodes and how many columns of the full grid share each (any order).
 * rank_host (nullable): r.  sanity_host as in temd_basis_build, with sanity[0] = r.  Fails (<0) if the Jacobi sweeps
 * do not converge or the rank-r whitened basis is not positive definite.  Works on any plan. */
int temd_basis_build_min_norm(temd_plan* plan, const double* x, const double* x_unique, const double* mult, int nunique,
                              const double* x_out, int* rank_host, double* sanity_host, void* stream);

/* Deprecated quadrature inverse of the reference, Y0inv = Y0^T diag(w) (sph_zonal_mean.py:72,180-181,383-386):
 * w[N] are the grid-cell area weights ALREADY multiplied by 4 pi.  temd_project / temd_synth_* then compute
 * Y (Y0^T diag(w)) A; temd_eddy_flux_project is not available in this mode. */
int temd_basis_build_weighted(temd_plan* plan, const double* x, const double* x_out, const double* w, void* stream);

/* Dense exports of the reference's attributes Y0 [N][L+1], Y0inv [L+1][N], Y0p [M][L+1]
 * (sph_zonal_mean.py:420-422); any pointer may be NULL. */
int temd_basis_export(temd_plan* plan, double* Y0, double* Y0inv, double* Y0p, void* stream);

/* Forward projection, first GEMM of sph_zonal_mean.py:251: coef[f][row][:] = Q^T fields[f][row][:].
 * fields_host: host array of nfields device pointers.  If lev_scale != NULL, rows of field
 * `scale_field` are multiplied by lev_scale[row % nlev] (theta = T*(p0/p)^k, tem_diagnostics.py:498). */
int temd_project(temd_plan* plan, const double* const* fields_host, int nfields, int rows, size_t ld,
                 const double* lev_scale, int scale_field, int nlev, double* coef, void* stream);

/* sph_zonal_mean (sph_zonal_mean.py:291-296): out[row][m] on the output latitudes, ld_out >= M, even. */
int temd_synth_out(temd_plan* plan, const double* coef, int rows, double* out, size_t ld_out, void* stream);

/* Optional Legendre-space latitude derivative (BASELINE.json north_star; NOT used by the reference, whose
 * lat_gradient is a finite difference, tem_util.py:154): out[row][m] = d/dphi of the zonal mean of sph_zonal_mean at the
 * output latitudes, per radian, = sum_l b_l dY_l/dphi(phi_m) with dY_l/dphi = cos(phi) Y_l'(sin phi) from the
 * differentiated three-term recurrence.  temd_basis_export_dlat writes the dense dY0p [M][L+1]. */
int temd_synth_out_dlat(temd_plan* plan, const double* coef, int rows, double* out, size_t ld_out, void* stream);
int temd_basis_export_dlat(temd_plan* plan, double* dY0p, void* stream);

/* sph_zonal_mean_native (sph_zonal_mean.py:285-290): out[row][n] on the native columns. */
int temd_synth_native(temd_plan* plan, const double* coef, int rows, double* out, size_t ld_out, void* stream);

/* On-demand native-grid eddy field of the reference's properties up, vp, thetap, wapp, qp
 * (tem_diagnostics.py:517-529,537): out[row][n] = lev_scale[row % nlev] * x[row][n] - (Q coef)[row][n]
 * (lev_scale NULL = 1).  Not on the hot path: the fused kernel below never materialises these. */
int temd_eddy_native(temd_plan* plan, const double* x, size_t ld_x, const double* coef, int rows,
                     const double* lev_scale, int nlev, double* out, size_t ld_out, void* stream);

/* Element-wise product out = a .* b on [rows][ncol] arrays (properties upvp, upwapp, vptp, :547-555). */
int temd_multiply(const double* a, size_t ld_a, const double* b, size_t ld_b, double* out, size_t ld_out,
                  int rows, int ncol, void* stream);

/* _decompose_zm_eddy + _compute_fluxes (tem_diagnostics.py:510-558), fused: per column tile forms the
 * native zonal means of u, v, T, omega from coef4 ([4][rows][lpad], order u,v,T,omega, T unscaled),
 * the eddies, the products u'v', u'omega', v'T' and projects them: coef_flux [3][rows][lpad]
 * (order upvp, upwapp, vptp).  coef4's theta block holds theta coefficients (already scaled) and the
 * kernel forms theta = lev_scale[row % nlev] * T on the fly.  Eddies and products never reach HBM. */
int temd_eddy_flux_project(temd_plan* plan, const double* u, const double* v, const double* t, const double* w,
                           int rows, size_t ld, const double* coef4, const double* lev_scale, int nlev,
                           double* coef_flux, void* stream);

/* Tracer eddy fluxes for TWO tracers at once (tem_diagnostics.py:532-538,560-570): coef4 = [4][rows][lpad] coefficient
 * blocks of (q1, q2, v, omega); coef_flux [4][rows][lpad] = projections of q1'v', q1'omega', q2'v', q2'omega'.  The
 * native means of v and omega are synthesised once for both tracers: 16 (L+1) flop per point per PAIR, against
 * 14 (L+1) per tracer when temd_eddy_flux_project is called on (q, v, T, omega). */
int temd_tracer_flux_project(temd_plan* plan, const double* q1, const double* q2, const double* v, const double* w,
                             int rows, size_t ld, const double* coef4, double* coef_flux, void* stream);

/* _compute_derivatives + the ten diagnostics methods (tem_diagnostics.py:574-797; tem_util.py:57-243).
 * zm: 7 zonal-mean arrays [nt][nlev][M] in the order ub, vb, thetab, wapb, upvpb, upwappb, vptpb.
 * gp/gl: np.gradient coefficient triplets (a,b,c) per level [3][nlev] / per latitude [3][M].
 * out: TEMD_NOUT arrays [nt][nlev][M] in the order of TEMD_OUT_* below (+2 planes kept for ABI compatibility with
 * v100, which staged F_phi cos(phi) / F_p there; no longer written). */
typedef struct temd_epilogue_args {
    int nt, nlev, nlat;
    size_t ld;              /* leading dimension (>= nlat) of every [nt*nlev][ld] plane */
    const double* zm;       /* [7][nt*nlev][ld] */
    const double* p;        /* [nlev] Pa */
    const double* latr;     /* [nlat] radians */
    const double* gp;       /* [3][nlev] interior np.gradient coefficients a, b, c */
    const double* gl;       /* [3][nlat] */
    int p_uniform, lat_uniform;   /* NumPy's exactly-uniform-spacing branch (then hp / hlat is the spacing) */
    double hp, hlat;
    const double* coslat;   /* [nlat] */
    const double* f;        /* [nlat] Coriolis parameter */
    double p0, a, H, g0, pi;
    double* out;            /* [TEMD_NOUT + 2][nt*nlev][ld]; the last two planes are unused (v100 scratch) */
} temd_epilogue_args;

enum {
    TEMD_OUT_DUB_DP = 0, TEMD_OUT_DTHETAB_DP, TEMD_OUT_UBCOSLAT, TEMD_OUT_DUBCOSLAT_DLAT, TEMD_OUT_PSI,
    TEMD_OUT_PSICOSLAT, TEMD_OUT_DPSICOSLAT_DLAT, TEMD_OUT_DPSI_DP, TEMD_OUT_INT_VBDP,
    TEMD_OUT_VTEM, TEMD_OUT_OMEGATEM, TEMD_OUT_WTEM, TEMD_OUT_PSITEM, TEMD_OUT_EPFY, TEMD_OUT_EPFZ,
    TEMD_OUT_EPDIV, TEMD_OUT_UTENDEPFD, TEMD_OUT_UTENDVTEM, TEMD_OUT_UTENDWTEM, TEMD_NOUT
};

int temd_tem_epilogue(temd_plan* plan, const temd_epilogue_args* args, void* stream);

/* Tracer TEM (tem_diagnostics.py:532-538,560-570,602-611 and the methods etfy/etfz/etdiv/qtendetfd/
 * qtendvtem/qtendwtem :801-991) for ONE tracer.  zmq: [3][nt*nlev][ld] = qb, qpvpb, qpwappb (obtained with
 * temd_project on q and temd_eddy_flux_project on (q, v, T, omega), whose first two products are then
 * q'v' and q'omega').  psi / vtem / omegatem: planes written by temd_tem_epilogue.
 * out: [TEMD_NTROUT + 2][nt*nlev][ld], last two planes unused (v100 scratch). */
typedef struct temd_tracer_args {
    int nt, nlev, nlat;
    size_t ld;
    const double* zmq;
    const double* psi;
    const double* vtem;
    const double* omegatem;
    const double* p;
    const double* latr;
    const double* gp;
    const double* gl;
    int p_uniform, lat_uniform;
    double hp, hlat;
    const double* coslat;
    double p0, a, H;
    double* out;
} temd_tracer_args;

enum {
    TEMD_TROUT_DQB_DP = 0, TEMD_TROUT_QBCOSLAT, TEMD_TROUT_DQBCOSLAT_DLAT, TEMD_TROUT_ETFY, TEMD_TROUT_ETFZ,
    TEMD_TROUT_ETDIV, TEMD_TROUT_QTENDETFD, TEMD_TROUT_QTENDVTEM, TEMD_TROUT_QTENDWTEM, TEMD_NTROUT
};

int temd_tracer_epilogue(temd_plan* plan, const temd_tracer_args* args, void* stream);

/* NaN screen of sph_zonal_mean.py:219-221 done on the small coefficient block (NaNs in a field
 * propagate into its coefficients): returns 0 if all n values are finite, -2 if a NaN was found, -6 if only
 * infinities were found (the reference screens NaN only).  Runs on the device that owns `data`; synchronises. */
int temd_check_finite(const double* data, size_t n, void* stream);

/* HOST helper (both pointers are host memory): multi-threaded memcpy used to stage pageable input arrays into
 * pinned buffers ahead of the asynchronous host->device copy.  No reference counterpart (the reference never leaves
 * the host). */
int temd_host_copy(void* dst_host, const void* src_host, size_t bytes, int nthreads);

/* ---- Structure-exploiting fast path (SURVEY.md §8f-4), opt-in -------------------------------------------------
 * Rows of Y0 depend on latitude only (sph_zonal_mean.py:361-363): columns with the same x = sin(lat) form a group
 * (a raveled lat-lon grid, tem_util.py:331, has NLAT groups of NLON columns).  The plan is created on the U unique
 * nodes and factorised with temd_basis_build_dedup (basis rows weighted by sqrt(multiplicity): same Gram matrix, same
 * coefficients as the dense path).  Group description, all device pointers: goff[U+1] offsets into the group-sorted
 * column list, perm[ncol] sorted position -> column (NULL when every group is a contiguous column range),
 * gid[ncol] column -> group, rsq[U] = 1/sqrt(multiplicity). */
int temd_basis_build_dedup(temd_plan* plan, const double* x_unique, const double* x_out, const double* mult,
                           double* sanity_host, void* stream);

/* One pass over the fields (HBM bound).  with_products = 0: out[f][row][u] = (sum_{i in u} fields[f][row][i]) * rsq[u]
 * for f < nfields <= 4 - the input of temd_project on the unique grid.  with_products = 1 (fields = u, v, T, omega;
 * lev_scale/scale_field as in temd_project turn T into theta): TEMD_GS_NPLANES planes [row][ld_out]:
 *   0-3 a0_f (first member of the group), 4-7 s_f = sum (x_f - a0_f), 8-10 sum (x_a - a0_a)(x_b - a0_b) for
 *   (a,b) = (u,v), (u,omega), (v,theta), 11-14 the weighted sums of with_products = 0.
 * max_count / min_count: largest / smallest multiplicity (selects the warp-per-group and thread-per-group kernels);
 * even_groups != 0: every goff[] entry is even (with perm == NULL this allows 16-byte loads). */
#define TEMD_GS_NPLANES 15
int temd_group_sums(const double* const* fields_host, int nfields, int rows, size_t ld, const int* perm,
                    const int* goff, int ngroups, int max_count, int min_count, int even_groups, const double* rsq,
                    const double* lev_scale, int scale_field, int nlev, int with_products, double* out,
                    size_t ld_out, void* stream);

/* Eddy-flux group sums about the spectral zonal means (tem_diagnostics.py:517-529,547-555 without materialising
 * eddies): means_w [4][rows][ld_m] = temd_synth_native of the four coefficient blocks on the unique grid
 * (= sqrt(n_u) * zonal mean); out [3][rows][ld_out] = rsq[u] * sum_{i in u} a'_i b'_i for u'v', u'omega', v'theta',
 * ready for temd_project on the unique grid. */
int temd_dedup_flux(const double* gsums, size_t ld_gs, const double* means_w, size_t ld_m, const int* goff,
                    const double* rsq, int rows, int ngroups, double* out, size_t ld_out, void* stream);

/* out[row][i] = alpha * lev_scale[row % nlev] * x[row][i] + beta * rsq[gid[i]] * means_w[row][gid[i]]
 * (x NULL: expanded native zonal mean, sph_zonal_mean.py:285-290; alpha 1, beta -1: eddy field). rsq NULL = 1. */
int temd_dedup_expand(const double* x, size_t ld_x, const double* lev_scale, int nlev, const double* means_w,
                      size_t ld_m, const int* gid, const double* rsq, double alpha, double beta, double* out,
                      size_t ld_out, int rows, int ncol, void* stream);

/* Multi-GPU (SURVEY.md §8e): time steps never interact (sph_zonal_mean.py:244-251, tem_util.py:154,192,232), so each
 * process owns a time slab and the only exchange is ONE all-gather of the stacked output planes at the end.
 * libnccl.so.2 is resolved at run time (dlopen); without it these three calls return -7 and everything else works.
 *   temd_comm_unique_id : rank 0 makes the 128-byte id and ships it to the other ranks by any side channel;
 *   temd_comm_init      : collective over all ranks (ncclCommInitRank) on `device`;
 *   temd_allgather_outputs : recv[r*count .. (r+1)*count) = rank r's send[0 .. count), enqueued on `stream`. */
typedef struct temd_comm temd_comm;
int temd_comm_unique_id(char* id128_host);
int temd_comm_init(int device, int nranks, int rank, const char* id128_host, temd_comm** comm);
int temd_comm_destroy(temd_comm* comm);
int temd_allgather_outputs(temd_comm* comm, const double* send, double* recv, size_t count, void* stream);

/* Synthetic benchmark/test fields (SURVEY.md §8d): out[t][lev][ncol], field 0..4 = ua, va, ta, wap, q. */
int temd_synth_fields(double* out, int field, int seed, int t0, int nt, int nlev, int ncol, size_t ld,
                      const double* lat_rad, const double* lon_rad, const double* plev_hpa, void* stream);

#ifdef __cplusplus
}
#endif
#endif
