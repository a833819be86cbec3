// One-sided (Hestenes) Jacobi SVD of the weighted unique-node basis Yw = diag(sqrt(n)) Y_U, for the minimum-norm
// build (temd_basis_build_min_norm, DESIGN.md §2 "truncated whitening").
//
// Yw (U x (L+1)) has the Gram matrix of the full-grid Y0, hence its singular values and right singular vectors V.
// The k = min(U, L+1) <= 1024 vectors that are orthogonalised are
//   the columns of Yw when U >= L+1 (tall; V accumulates the rotations), or
//   the rows of Yw when U < L+1 (wide; converged row i is sigma_i v_i^T).
// The vectors are rows of a row-major [k][lda] array.  Pairs follow the round-robin (circle) ordering, k/2 disjoint
// pairs per launch; the ordering and every reduction are fixed, so results are reproducible run to run.  The rank
// follows NumPy's lstsq/pinv default cutoff: sigma_i > eps max(N, L+1) sigma_1, N = total column count.  Eigenvalues
// of the Gram matrix would not do: they resolve sigma / sigma_1 down to ~1e-8 only, and the cutoff sits near 1e-13.
#include <cmath>
#include <cstring>

#include "temd_common.cuh"
#include "temd_internal.h"

namespace temd {

static constexpr int kSvdThreads = 256;
static constexpr int kSvdMaxSweeps = 30;

// round-robin ordering of kk (even) slots: slot 0 stays, slots 1..kk-1 rotate by one position per step
__device__ __forceinline__ int rr_slot(int pos, int step, int kk) { return pos == 0 ? 0 : (pos - 1 + step) % (kk - 1) + 1; }

// sums of three per-thread values over the block; every thread gets the totals (fixed order: reproducible)
__device__ __forceinline__ void block_sum3(double& a, double& b, double& c) {
    __shared__ double s[3][kSvdThreads / 32];
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s[0][w] = a; s[1][w] = b; s[2][w] = c; }
    __syncthreads();
    a = b = c = 0.0;
    for (int i = 0; i < kSvdThreads / 32; i++) { a += s[0][i]; b += s[1][i]; c += s[2][i]; }
    __syncthreads();
}

// One step of a sweep: block t orthogonalises the pair in slots (t, kk-1-t).  `off` receives the largest
// |a_i^T a_j| / (|a_i| |a_j|) above `tol` seen (non-negative doubles order like their bit patterns).
__global__ void __launch_bounds__(kSvdThreads)
k_jacobi_step(double* __restrict__ A, size_t lda, int m, double* __restrict__ Vt, size_t ldv, int nv, int k, int kk,
              int step, double tol, unsigned long long* __restrict__ off) {
    int i = rr_slot(blockIdx.x, step, kk), j = rr_slot(kk - 1 - blockIdx.x, step, kk);
    if (i >= k || j >= k) return;                   // partner of the padding slot (odd k)
    if (i > j) { const int t = i; i = j; j = t; }
    double* ai = A + (size_t)i * lda;
    double* aj = A + (size_t)j * lda;
    double al = 0.0, be = 0.0, ga = 0.0;
    for (int e = threadIdx.x; e < m; e += kSvdThreads) {
        const double x = ai[e], y = aj[e];
        al = fma(x, x, al); be = fma(y, y, be); ga = fma(x, y, ga);
    }
    block_sum3(al, be, ga);
    if (!(al > 0.0) || !(be > 0.0)) return;
    const double rel = fabs(ga) / sqrt(al) / sqrt(be);
    if (!(rel > tol)) return;
    if (threadIdx.x == 0) atomicMax(off, (unsigned long long)__double_as_longlong(rel));
    // stable rotation (Rutishauser; Demmel & Veselic 1992): t = sign(zeta) / (|zeta| + sqrt(1 + zeta^2))
    const double zeta = (be - al) / (2.0 * ga);
    const double az = fabs(zeta);
    const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (az > 1e150 ? 2.0 * az : az + sqrt(1.0 + zeta * zeta));
    const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
    for (int e = threadIdx.x; e < m; e += kSvdThreads) {
        const double x = ai[e], y = aj[e];
        ai[e] = c * x - s * y;
        aj[e] = s * x + c * y;
    }
    if (Vt != nullptr) {
        double* vi = Vt + (size_t)i * ldv;
        double* vj = Vt + (size_t)j * ldv;
        for (int e = threadIdx.x; e < nv; e += kSvdThreads) {
            const double x = vi[e], y = vj[e];
            vi[e] = c * x - s * y;
            vj[e] = s * x + c * y;
        }
    }
}

// sigma[i] = |a_i|, one block per vector
__global__ void __launch_bounds__(kSvdThreads)
k_jacobi_norms(const double* __restrict__ A, size_t lda, int m, double* __restrict__ sigma) {
    const double* a = A + (size_t)blockIdx.x * lda;
    double s = 0.0, d1 = 0.0, d2 = 0.0;
    for (int e = threadIdx.x; e < m; e += kSvdThreads) s = fma(a[e], a[e], s);
    block_sum3(s, d1, d2);
    if (threadIdx.x == 0) sigma[blockIdx.x] = sqrt(s);
}

// Single block: rank decision and the truncated whitening matrix.  Kept vectors are ordered by decreasing sigma
// (ties by index); row p < r of Wt (lpad x lpad, zero elsewhere) is w_p^T, the p-th column of W = V_r Sigma_r^-1:
// v_i / sigma_i from Vt (tall) or a_i / sigma_i^2 (wide, a_i = sigma_i v_i^T).  sigma_sorted[p] = sorted sigma.
__global__ void __launch_bounds__(1024)
k_jacobi_finalize(const double* __restrict__ A, size_t lda, const double* __restrict__ Vt, size_t ldv,
                  const double* __restrict__ sigma, int k, int Lp, const double* __restrict__ mult, int nu,
                  double* __restrict__ Wt, int lpad, double* __restrict__ sigma_sorted, int* __restrict__ rank_out) {
    __shared__ int s_src[1024];
    __shared__ double s_red[32];
    __shared__ int s_rank;
    const int tid = threadIdx.x;
    // total column count N (multiplicities are integers: the sum is exact) and sigma_1
    double n = 0.0, smax = 0.0;
    for (int u = tid; u < nu; u += blockDim.x) n += mult[u];
    for (int i = tid; i < k; i += blockDim.x) smax = fmax(smax, sigma[i]);
    for (int o = 16; o > 0; o >>= 1) {
        n += __shfl_xor_sync(0xffffffffu, n, o);
        smax = fmax(smax, __shfl_xor_sync(0xffffffffu, smax, o));
    }
    if ((tid & 31) == 0) s_red[tid >> 5] = n;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += s_red[w];
        s_red[0] = t;
        s_rank = 0;
    }
    __syncthreads();
    n = s_red[0];
    __syncthreads();
    if ((tid & 31) == 0) s_red[tid >> 5] = smax;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t = fmax(t, s_red[w]);
        s_red[0] = t;
    }
    __syncthreads();
    const double cutoff = 2.220446049250313e-16 * fmax(n, (double)Lp) * s_red[0];
    for (int i = tid; i < k; i += blockDim.x) {
        const double si = sigma[i];
        int pos = 0;
        for (int j = 0; j < k; j++) {
            const double sj = sigma[j];
            pos += (sj > si || (sj == si && j < i)) ? 1 : 0;
        }
        s_src[pos] = i;
        sigma_sorted[pos] = si;
        if (si > cutoff) atomicAdd(&s_rank, 1);
    }
    __syncthreads();
    const int r = s_rank;
    for (size_t e = tid; e < (size_t)lpad * lpad; e += blockDim.x) {
        const int p = (int)(e / lpad), l = (int)(e % lpad);
        double v = 0.0;
        if (p < r && l < Lp) {
            const int i = s_src[p];
            const double si = sigma[i];
            v = (Vt != nullptr) ? Vt[(size_t)i * ldv + l] / si : A[(size_t)i * lda + l] / (si * si);
        }
        Wt[e] = v;
    }
    if (tid == 0) *rank_out = r;
}

__global__ void k_identity(double* __restrict__ M, int n, int ld) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)n * ld) return;
    M[e] = ((int)(e / ld) == (int)(e % ld)) ? 1.0 : 0.0;
}

int launch_identity(double* M, int n, int ld, cudaStream_t stream) {
    const size_t tot = (size_t)n * ld;
    k_identity<<<(unsigned)((tot + 255) / 256), 256, 0, stream>>>(M, n, ld);
    return (int)cudaGetLastError();
}

int jacobi_svd_whitening(double* A, size_t lda, int m, int k, double* Vt, size_t ldv, int Lp, const double* mult,
                         int nu, double* Wt, int lpad, double* sigma, double* sigma_sorted, int* rank_dev,
                         unsigned long long* off_dev, int* sweeps_out, cudaStream_t stream) {
    if (k < 1 || k > 1024) return temd_set_error(-1, "jacobi_svd: k = %d outside [1, 1024]", k);
    const int kk = k + (k & 1);
    // convergence: every pair's |a_i^T a_j| / (|a_i| |a_j|) below sqrt(m) eps (LAPACK dgesvj's tolerance), with a
    // factor 16 of headroom over the rounding floor of a length-m dot product
    const double tol = 16.0 * 2.220446049250313e-16 * std::sqrt((double)m);
    int sweep = 0;
    bool converged = (k == 1);
    unsigned long long off = 0;
    while (!converged && sweep < kSvdMaxSweeps) {
        cudaError_t e = cudaMemsetAsync(off_dev, 0, sizeof(unsigned long long), stream);
        if (e != cudaSuccess) return temd_set_error((int)e, "jacobi_svd: %s", cudaGetErrorString(e));
        for (int step = 0; step < kk - 1; step++)
            k_jacobi_step<<<kk / 2, kSvdThreads, 0, stream>>>(A, lda, m, Vt, ldv, Vt ? k : 0, k, kk, step, tol, off_dev);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(&off, off_dev, sizeof(off), cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return temd_set_error((int)e, "jacobi_svd: %s", cudaGetErrorString(e));
        sweep++;
        converged = (off == 0);
    }
    if (!converged) {
        double worst;
        memcpy(&worst, &off, sizeof(worst));
        return temd_set_error(-5, "jacobi_svd: no convergence in %d sweeps (k = %d vectors of length %d; largest relative "
                                  "off-diagonal of the last sweep %.3e, tolerance %.3e)", kSvdMaxSweeps, k, m, worst, tol);
    }
    if (sweeps_out) *sweeps_out = sweep;
    k_jacobi_norms<<<k, kSvdThreads, 0, stream>>>(A, lda, m, sigma);
    k_jacobi_finalize<<<1, 1024, 0, stream>>>(A, lda, Vt, ldv, sigma, k, Lp, mult, nu, Wt, lpad, sigma_sorted, rank_dev);
    return (int)cudaGetLastError();
}

}  // namespace temd
