// Internal (non-ABI) declarations shared by the temd translation units.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#define TEMD_MAX_FIELDS 8

namespace temd {

// error plumbing (temd_api.cu): records a thread-local message, returns `code`
int temd_set_error(int code, const char* fmt, ...);

// TMA descriptor for a row-major 2-D double array: dim0 = contiguous extent (elements), dim1 = rows,
// box = {box0 (<=16), box1 (<=256)}, 128-B swizzle, zero fill out of bounds.
int make_tma_2d(CUtensorMap* out, const void* base, uint64_t dim0, uint64_t dim1, uint64_t row_stride_bytes,
                uint32_t box0, uint32_t box1);

// ---- K4 project (temd_project.cu) ----
void project_lblocks(int lpad, int* ntb, int* lblocks);
int project_pick_split(int tiles, int nchunks, int sms, int max_split);
int launch_reduce_partials(const double* part, double* out, int nsplit, int nfields, int rows, int lpad,
                           const double* lev_scale, int scale_field, int nlev, cudaStream_t stream);
size_t project_workspace_doubles(int nfields, int rows, int lpad, int nsplit);
int launch_project(const double* const* x, int nfields, int rows, int ncol, size_t ld_x, const double* qt, int lpad,
                   size_t ld_q, double* out, double* part, int nsplit, const double* lev_scale, int scale_field,
                   int nlev, cudaStream_t stream);

int launch_project_products(const double* const* xpairs, int npairs, int rows, int ncol, size_t ld_x, const double* qt,
                            int lpad, size_t ld_q, double* out, double* part, int nsplit, cudaStream_t stream);

// ---- generic synthesis GEMM  S[row][n] = sum_l C[row][l] * B[l][n]  (temd_synth.cu) ----
int launch_synth(const double* c, int rows, int lpad, size_t ld_c, const double* b, int ncol, size_t ld_b, double* out,
                 size_t ld_out, cudaStream_t stream);

int launch_synth_eddy4(const double* coef4, int rows_total, int r0, int rows, int lpad, const double* b, int ncol, size_t ld_b,
                       const double* const* x, size_t ld_x, const double* lev_scale, int scale_field, int nlev,
                       double* const* out, size_t ld_out, cudaStream_t stream);

int launch_synth_resident(const double* c, int rows, int lpad, size_t ld_c, const double* b, int ncol, size_t ld_b,
                          double* out, size_t ld_out, int sms, cudaStream_t stream);

// ---- K1 basis + K3 Cholesky/inverse (temd_basis.cu) ----
int launch_basis(const double* x, int n, int L, const double* rec_a, const double* rec_b, double* qt, size_t ld,
                 int lpad, cudaStream_t stream);
int launch_basis_dlat(const double* x, int n, int L, const double* rec_a, const double* rec_b, double* dt, size_t ld,
                      int lpad, cudaStream_t stream);
int launch_chol_inv(const double* G, int ldg, int n, double* LT, double* Linv, int ldi, int lpad, int* status,
                    cudaStream_t stream);
int launch_matmul_small(const double* A, const double* B, double* C, int n, int ld, cudaStream_t stream);

// ---- one-sided Jacobi SVD for the minimum-norm build (temd_svd.cu) ----
int launch_identity(double* M, int n, int ld, cudaStream_t stream);
// Orthogonalises the k rows (length m) of A in place (Vt != NULL: accumulates the rotations into the k x k rows of Vt,
// which must hold the identity), then writes the truncated whitening matrix Wt [lpad][lpad] and the rank (device
// int).  sigma / sigma_sorted: k doubles each.  mult[nu]: node multiplicities (their sum is N in the cutoff).
// Synchronises once per sweep; fails if the sweeps do not converge.
int jacobi_svd_whitening(double* A, size_t lda, int m, int k, double* Vt, size_t ldv, int Lp, const double* mult,
                         int nu, double* Wt, int lpad, double* sigma, double* sigma_sorted, int* rank_dev,
                         unsigned long long* off_dev, int* sweeps_out, cudaStream_t stream);

// ---- K5 fused eddy / flux / projection (temd_eddy.cu) ----
int eddy_supported(int lpad);
int eddy_pick_split(int rows, int lpad, int nchunks, int sms, int nprod);
size_t eddy_workspace_doubles(int rows, int lpad, int nsplit, int nprod);
int launch_eddy_flux_project(const double* const* x4, int rows, int ncol, size_t ld_x, const double* qt, int lpad,
                             size_t ld_q, const double* coef4, double* coef_flux, double* part, int nsplit,
                             const double* lev_scale, int nlev, int nprod, cudaStream_t stream);

// ---- K6 stencil epilogue (temd_epilogue.cu) ----
struct EpilogueArgs;
int launch_tem_epilogue(const EpilogueArgs& a, cudaStream_t stream);

// ---- synthetic fields (temd_fields.cu) ----
int launch_synth_fields(double* out, int field, int seed, int t0, int nt, int nlev, int ncol, size_t ld,
                        const double* lat_rad, const double* lon_rad, const double* plev_hpa, cudaStream_t stream);

}  // namespace temd
