// extern "C" entry points of libtemd (declared in include/temd.h) + plan management.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/temd.h"
#include "temd_common.cuh"
#include "temd_internal.h"

namespace temd {

static thread_local char g_err[512] = "";

int temd_set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define TEMD_CUDA(call)                                                                              \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return temd_set_error((int)e__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                                  __FILE__, __LINE__);                                               \
    } while (0)

// Every entry point runs on the plan's device and leaves the caller's current device untouched.
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
        else if (err == cudaSuccess) prev = -1;   // nothing to restore
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define TEMD_ON_DEVICE(dev)                 \
    DeviceGuard guard__(dev);               \
    TEMD_CUDA(guard__.err)

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

int make_tma_2d(CUtensorMap* out, const void* base, uint64_t dim0, uint64_t dim1, uint64_t row_stride_bytes,
                uint32_t box0, uint32_t box1) {
    PFN_encodeTiled enc = get_encode();
    if (enc == nullptr) return temd_set_error(-3, "cuTensorMapEncodeTiled entry point not available");
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (row_stride_bytes & 15))
        return temd_set_error(-1, "TMA operand must be 16-byte aligned with a 16-byte-multiple row stride "
                                  "(base %p, stride %llu B): use an even leading dimension",
                              base, (unsigned long long)row_stride_bytes);
    if (box0 * sizeof(double) > 128 || box1 > 256) return temd_set_error(-1, "TMA box too large");
    cuuint64_t gdim[2] = {dim0, dim1};
    cuuint64_t gstr[1] = {row_stride_bytes};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return temd_set_error(-3, "cuTensorMapEncodeTiled failed (CUresult %d; dims %llu x %llu, stride %llu, box %u x %u)",
                              (int)r, (unsigned long long)dim0, (unsigned long long)dim1,
                              (unsigned long long)row_stride_bytes, box0, box1);
    return 0;
}

// flag bit 0: a NaN was seen, bit 1: an infinity was seen
__global__ void k_check_finite(const double* __restrict__ d, size_t n, int* __restrict__ flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    int bad = 0;
    for (; i < n; i += stride) {
        const double v = d[i];
        bad |= (v != v) ? 1 : (isinf(v) ? 2 : 0);
    }
    if (bad) atomicOr(flag, bad);
}

__global__ void k_trace_offdiag(const double* __restrict__ G, int n, int ld, double* __restrict__ out2) {
    // single block: out2[0] = trace, out2[1] = sum of off-diagonal entries
    __shared__ double s_tr[256], s_off[256];
    double tr = 0.0, off = 0.0;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n, j = e % n;
        const double v = G[(size_t)i * ld + j];
        if (i == j) tr += v; else off += v;
    }
    s_tr[threadIdx.x] = tr; s_off[threadIdx.x] = off;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) { s_tr[threadIdx.x] += s_tr[threadIdx.x + w]; s_off[threadIdx.x] += s_off[threadIdx.x + w]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out2[0] = s_tr[0]; out2[1] = s_off[0]; }
}

// out[row][n] = scale[row % nlev] * x[row][n] - out[row][n]   (eddy X' = X - zonal mean; scale = theta factor or null)
__global__ void k_eddy_native(const double* __restrict__ x, size_t ld_x, const double* __restrict__ scale, int nlev,
                              double* __restrict__ out, size_t ld_out, int rows, int n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n) return;
    for (int r = blockIdx.y; r < rows; r += gridDim.y) {
        const double s = scale ? scale[r % nlev] : 1.0;
        out[(size_t)r * ld_out + i] = s * x[(size_t)r * ld_x + i] - out[(size_t)r * ld_out + i];
    }
}

// out = a .* b
__global__ void k_mul(const double* __restrict__ a, size_t ld_a, const double* __restrict__ b, size_t ld_b,
                      double* __restrict__ out, size_t ld_out, int rows, int n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n) return;
    for (int r = blockIdx.y; r < rows; r += gridDim.y) out[(size_t)r * ld_out + i] = a[(size_t)r * ld_a + i] * b[(size_t)r * ld_b + i];
}

__global__ void k_add_diag(double* __restrict__ G, int ld, int n, double s) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) G[(size_t)i * ld + i] += s;
}

// out[l][n] = in[l][n] * w[n]   (Y0inv = Y0^T diag(w), reference sph_zonal_mean.py:383-386)
__global__ void k_scale_cols(const double* __restrict__ in, const double* __restrict__ w, double* __restrict__ out,
                             int rows, int n, size_t ld) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int l = blockIdx.y;
    if (i >= ld || l >= rows) return;
    out[(size_t)l * ld + i] = (i < (size_t)n) ? in[(size_t)l * ld + i] * w[i] : 0.0;
}

// in[l][n] *= sqrt(m[n])   (weighted unique grid of the de-duplicated path)
__global__ void k_scale_cols_sqrt(double* __restrict__ q, const double* __restrict__ m, int rows, int n, size_t ld) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int l = blockIdx.y;
    if (i >= (size_t)n || l >= rows) return;
    q[(size_t)l * ld + i] *= sqrt(m[i]);
}

// out[i][j] = in[j][i]; in is [rows_in][ld_in], out is [cols_in][ld_out]  (dense exports only)
__global__ void k_transpose(const double* __restrict__ in, int rows_in, int cols_in, size_t ld_in,
                            double* __restrict__ out, size_t ld_out) {
    __shared__ double tile[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int rr = r0 + r, cc = c0 + threadIdx.x;
        tile[r][threadIdx.x] = (rr < rows_in && cc < cols_in) ? in[(size_t)rr * ld_in + cc] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int oc = r0 + threadIdx.x, orow = c0 + r;
        if (orow < cols_in && oc < rows_in) out[(size_t)orow * ld_out + oc] = tile[threadIdx.x][r];
    }
}

}  // namespace temd

using namespace temd;

struct temd_plan {
    int dev, N, L, Lp, lpad, M, sms;
    size_t ld_q, ld_p;
    double *qt, *qt_alt;     // whitened basis Q^T [lpad][ld_q] and ping-pong buffer
    double *qpt, *qpt_alt;   // whitened output-grid basis [lpad][ld_p]
    double *dqpt;            // whitened latitude-derivative basis on the output grid (lazy, temd_synth_out_dlat)
    bool dqpt_built;
    double *linv, *linv1, *linv2, *gram, *lt;   // [lpad][lpad] each
    double *rec_a, *rec_b;   // recurrence coefficients [L+1]
    double *x, *x_out;       // copies of the node coordinates (for exports)
    std::mutex* work_mu;     // split-K partials: one workspace per stream, so a plan is re-entrant per (device, stream)
    std::map<std::pair<cudaStream_t, int>, std::pair<double*, size_t>>* work;   // slot 0: split-K partials, 1: eddy scratch
    int* status;
    double* sanity;
    bool built;
    bool weighted;   // deprecated quadrature inverse Y0inv = Y0^T diag(w): qt = raw basis (synthesis), qt_alt = weighted (projection)
    int rank;        // number of whitened directions of the built basis (L+1 unless built by temd_basis_build_min_norm)
};

// Split-K workspace of `stream` (grown on demand).  Work already enqueued on that stream may still use the old
// buffer when it grows: cudaFree synchronises the device before releasing it.
static int ensure_work(temd_plan* p, cudaStream_t stream, size_t doubles, double** out, int slot = 0) {
    std::lock_guard<std::mutex> lock(*p->work_mu);
    auto& w = (*p->work)[std::make_pair(stream, slot)];
    if (doubles > w.second) {
        if (w.first) TEMD_CUDA(cudaFree(w.first));
        w.first = nullptr;
        w.second = 0;
        TEMD_CUDA(cudaMalloc(&w.first, doubles * sizeof(double)));
        w.second = doubles;
    }
    *out = w.first;
    return 0;
}

static size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

extern "C" int temd_version(void) { return 101; }
extern "C" const char* temd_last_error(void) { return g_err; }

static int plan_create_impl(int device, int ncol, int L, int nlat_out, bool min_norm, temd_plan** out) {
    if (out == nullptr) return temd_set_error(-1, "plan_create: null output");
    *out = nullptr;
    if (ncol < 1 || L < 0 || nlat_out < 1) return temd_set_error(-1, "plan_create: bad sizes (ncol %d, L %d, M %d)", ncol, L, nlat_out);
    if (L + 1 > 1024) return temd_set_error(-1, "plan_create: L = %d exceeds the supported maximum 1023", L);
    if (!min_norm && L + 1 > ncol) return temd_set_error(-1, "plan_create: L+1 = %d exceeds ncol = %d (Y0 would be rank-deficient: lower L; the reference's lstsq would return a minimum-norm solution here, this build does not)", L + 1, ncol);
    TEMD_ON_DEVICE(device);
    cudaDeviceProp prop;
    TEMD_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return temd_set_error(-4, "libtemd is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    temd_plan* p = new temd_plan();
    memset(p, 0, sizeof(*p));
    p->work_mu = new std::mutex();
    p->work = new std::map<std::pair<cudaStream_t, int>, std::pair<double*, size_t>>();
    p->dev = device; p->N = ncol; p->L = L; p->Lp = L + 1; p->M = nlat_out;
    p->rank = -1;
    p->lpad = (int)round_up(L + 1, 8);
    p->sms = prop.multiProcessorCount;
    p->ld_q = round_up(ncol, 16);
    p->ld_p = round_up(nlat_out, 16);
    const size_t lp = p->lpad;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](double** ptr, size_t n) { if (e == cudaSuccess) e = cudaMalloc(ptr, n * sizeof(double)); };
    alloc(&p->qt, lp * p->ld_q); alloc(&p->qt_alt, lp * p->ld_q);
    alloc(&p->qpt, lp * p->ld_p); alloc(&p->qpt_alt, lp * p->ld_p);
    alloc(&p->linv, lp * lp); alloc(&p->linv1, lp * lp); alloc(&p->linv2, lp * lp); alloc(&p->gram, lp * lp); alloc(&p->lt, lp * lp);
    alloc(&p->rec_a, lp); alloc(&p->rec_b, lp);
    alloc(&p->x, ncol); alloc(&p->x_out, nlat_out);
    alloc(&p->sanity, 2);
    if (e == cudaSuccess) e = cudaMalloc(&p->status, sizeof(int));
    if (e != cudaSuccess) {
        temd_plan_destroy(p);
        return temd_set_error((int)e, "plan_create: cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    *out = p;
    return 0;
}

extern "C" int temd_plan_create(int device, int ncol, int L, int nlat_out, temd_plan** out) {
    return plan_create_impl(device, ncol, L, nlat_out, false, out);
}

extern "C" int temd_plan_create_min_norm(int device, int ncol, int L, int nlat_out, temd_plan** out) {
    return plan_create_impl(device, ncol, L, nlat_out, true, out);
}

extern "C" int temd_plan_destroy(temd_plan* p) {
    if (p == nullptr) return 0;
    DeviceGuard guard(p->dev);
    double* bufs[] = {p->dqpt, p->qt, p->qt_alt, p->qpt, p->qpt_alt, p->linv, p->linv1, p->linv2, p->gram, p->lt,
                      p->rec_a, p->rec_b, p->x, p->x_out, p->sanity};
    for (double* b : bufs) if (b) cudaFree(b);
    if (p->work) for (auto& kv : *p->work) if (kv.second.first) cudaFree(kv.second.first);
    if (p->status) cudaFree(p->status);
    delete p->work;
    delete p->work_mu;
    delete p;
    return 0;
}

extern "C" int temd_plan_lpad(const temd_plan* p) { return p ? p->lpad : -1; }
extern "C" int temd_plan_rank(const temd_plan* p) { return (p && p->built) ? p->rank : -1; }

static int gram_of(temd_plan* p, const double* basis, cudaStream_t st) {
    int ntb, lblocks;
    project_lblocks(p->lpad, &ntb, &lblocks);
    const int tiles = (p->Lp + 127) / 128;
    const int nchunks = (p->N + 15) / 16;
    const int nsplit = project_pick_split(tiles * lblocks, nchunks, p->sms, 512);
    double* work = nullptr;
    int rc = ensure_work(p, st, project_workspace_doubles(1, p->Lp, p->lpad, nsplit), &work);
    if (rc) return rc;
    const double* xs[1] = {basis};
    return launch_project(xs, 1, p->Lp, p->N, p->ld_q, basis, p->lpad, p->ld_q, p->gram, work, nsplit, nullptr, -1, 1, st);
}

// Recurrence coefficients, copies of the nodes and the raw (transposed) basis on both grids in qt_alt / qpt_alt;
// `mult` (nullable) scales the native rows by sqrt(mult).  Runs on the caller's device and stream.
static int raw_basis(temd_plan* p, const double* x, const double* x_out, const double* mult, cudaStream_t st) {
    // recurrence coefficients: Y_l = a_l x Y_{l-1} - b_l Y_{l-2}
    std::vector<double> ra(p->lpad, 0.0), rb(p->lpad, 0.0);
    const double PI = 3.141592653589793238462643383279502884;
    ra[0] = std::sqrt(1.0 / (4.0 * PI));
    if (p->L >= 1) ra[1] = std::sqrt(3.0 / (4.0 * PI));
    for (int l = 2; l <= p->L; l++) {
        ra[l] = std::sqrt(4.0 * l * l - 1.0) / l;
        rb[l] = ((l - 1.0) / l) * std::sqrt((2.0 * l + 1.0) / (2.0 * l - 3.0));
    }
    TEMD_CUDA(cudaMemcpyAsync(p->rec_a, ra.data(), p->lpad * sizeof(double), cudaMemcpyHostToDevice, st));
    TEMD_CUDA(cudaMemcpyAsync(p->rec_b, rb.data(), p->lpad * sizeof(double), cudaMemcpyHostToDevice, st));
    TEMD_CUDA(cudaStreamSynchronize(st));   // ra/rb are stack-owned
    TEMD_CUDA(cudaMemcpyAsync(p->x, x, p->N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    TEMD_CUDA(cudaMemcpyAsync(p->x_out, x_out, p->M * sizeof(double), cudaMemcpyDeviceToDevice, st));
    int rc;
    // K1: raw basis (transposed) on both grids
    if ((rc = launch_basis(p->x, p->N, p->L, p->rec_a, p->rec_b, p->qt_alt, p->ld_q, p->lpad, st))) return temd_set_error(rc, "basis kernel launch failed");
    if ((rc = launch_basis(p->x_out, p->M, p->L, p->rec_a, p->rec_b, p->qpt_alt, p->ld_p, p->lpad, st))) return temd_set_error(rc, "basis kernel launch failed");
    if (mult != nullptr) {
        dim3 grid((unsigned)((p->ld_q + 255) / 256), p->lpad);
        k_scale_cols_sqrt<<<grid, 256, 0, st>>>(p->qt_alt, mult, p->lpad, p->N, p->ld_q);
        TEMD_CUDA(cudaGetLastError());
    }
    return 0;
}

// Optional sanity readback, then marks the whitened basis built with `rank` directions.
static int finish_build(temd_plan* p, double* sanity_host, int rank, cudaStream_t st) {
    int rc;
    if (sanity_host != nullptr) {
        // reference's logged check (sph_zonal_mean.py:393-398): Y0inv Y0 = L^-T (Q^T Q) L^T; we report Q^T Q
        if ((rc = gram_of(p, p->qt, st))) return rc;
        k_trace_offdiag<<<1, 256, 0, st>>>(p->gram, p->Lp, p->lpad, p->sanity);
        TEMD_CUDA(cudaGetLastError());
        TEMD_CUDA(cudaMemcpyAsync(sanity_host, p->sanity, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    TEMD_CUDA(cudaStreamSynchronize(st));
    p->built = true;
    p->weighted = false;
    p->dqpt_built = false;
    p->rank = rank;
    return 0;
}

// `mult` (nullable): multiplicity of every node.  The raw basis rows are then scaled by sqrt(mult) before the
// factorisation (weighted unique grid of the de-duplicated fast path, temd_dedup.cu): its Gram matrix is the Gram
// matrix of the full grid in which node u appears mult[u] times.
static int basis_build_impl(temd_plan* p, const double* x, const double* x_out, const double* mult, double* sanity_host,
                            void* stream) {
    if (p == nullptr || x == nullptr || x_out == nullptr) return temd_set_error(-1, "basis_build: null argument");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    int rc = raw_basis(p, x, x_out, mult, st);
    if (rc) return rc;
    // CholeskyQR2: G = Y^T Y = L L^T, Y <- Y L^-T, twice (the second pass removes the cond(Y0)^2 eps loss of
    // orthogonality of the first); L^-1 accumulates as L2^-1 L1^-1.  If the first factorisation breaks down
    // (cond(Y0) >~ 3e6), a shifted first pass (G + s I, s = 11 (N Lp + Lp(Lp+1)) eps trace(G), "shifted
    // CholeskyQR3") pre-conditions the basis and one more pass is run.  A breakdown after that means Y0 is
    // numerically rank-deficient (where LAPACK gelsd would truncate): fail loudly.
    int status = 0;
    int passes = 2;
    for (int pass = 0; pass < passes; pass++) {
        double* cur = (pass == 0) ? p->qt_alt : p->qt;       // pass 0 reads the raw basis from the alt buffers
        double* curp = (pass == 0) ? p->qpt_alt : p->qpt;
        if ((rc = gram_of(p, cur, st))) return rc;
        if ((rc = launch_chol_inv(p->gram, p->lpad, p->Lp, p->lt, p->linv2, p->lpad, p->lpad, p->status, st))) return temd_set_error(rc, "cholesky launch failed");
        TEMD_CUDA(cudaMemcpyAsync(&status, p->status, sizeof(int), cudaMemcpyDeviceToHost, st));
        TEMD_CUDA(cudaStreamSynchronize(st));
        if (status != 0 && pass == 0) {
            double tr[2] = {0.0, 0.0};
            k_trace_offdiag<<<1, 256, 0, st>>>(p->gram, p->Lp, p->lpad, p->sanity);
            TEMD_CUDA(cudaMemcpyAsync(tr, p->sanity, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
            TEMD_CUDA(cudaStreamSynchronize(st));
            const double shift = 11.0 * ((double)p->N * p->Lp + (double)p->Lp * (p->Lp + 1)) * 1.1102230246251565e-16 * tr[0];
            k_add_diag<<<(p->Lp + 127) / 128, 128, 0, st>>>(p->gram, p->lpad, p->Lp, shift);
            if ((rc = launch_chol_inv(p->gram, p->lpad, p->Lp, p->lt, p->linv2, p->lpad, p->lpad, p->status, st))) return temd_set_error(rc, "cholesky launch failed");
            TEMD_CUDA(cudaMemcpyAsync(&status, p->status, sizeof(int), cudaMemcpyDeviceToHost, st));
            TEMD_CUDA(cudaStreamSynchronize(st));
            passes = 3;
        }
        if (status != 0)
            return temd_set_error(-5, "basis_build: Y0 is numerically rank-deficient (Cholesky pivot %d of %d non-positive in pass %d); "
                                      "L = %d is too large for this grid", status - 1, p->Lp, pass + 1, p->L);
        // Y <- L^-1 Y (transposed storage), written to the other buffer pair
        double* dst = (pass == 0) ? p->qt : p->qt_alt;
        double* dstp = (pass == 0) ? p->qpt : p->qpt_alt;
        if ((rc = launch_synth(p->linv2, p->lpad, p->lpad, p->lpad, cur, p->N, p->ld_q, dst, p->ld_q, st))) return rc;
        if ((rc = launch_synth(p->linv2, p->lpad, p->lpad, p->lpad, curp, p->M, p->ld_p, dstp, p->ld_p, st))) return rc;
        if (pass > 0) { std::swap(p->qt, p->qt_alt); std::swap(p->qpt, p->qpt_alt); }
        // accumulate L^-1
        if (pass == 0) {
            TEMD_CUDA(cudaMemcpyAsync(p->linv, p->linv2, (size_t)p->lpad * p->lpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
        } else {
            if ((rc = launch_matmul_small(p->linv2, p->linv, p->linv1, p->lpad, p->lpad, st))) return temd_set_error(rc, "matmul launch failed");
            std::swap(p->linv, p->linv1);
        }
    }
    if ((rc = finish_build(p, sanity_host, p->Lp, st))) return rc;
    return 0;
}

extern "C" int temd_basis_build(temd_plan* p, const double* x, const double* x_out, double* sanity_host, void* stream) {
    return basis_build_impl(p, x, x_out, nullptr, sanity_host, stream);
}

extern "C" int temd_basis_build_dedup(temd_plan* p, const double* x_unique, const double* x_out, const double* mult,
                                      double* sanity_host, void* stream) {
    if (mult == nullptr) return temd_set_error(-1, "basis_build_dedup: null multiplicities");
    return basis_build_impl(p, x_unique, x_out, mult, sanity_host, stream);
}

// Minimum-norm build: the first whitening pass uses W^T = (V_r Sigma_r^-1)^T from the Jacobi SVD of the weighted
// unique-node basis Yw (temd_svd.cu) instead of L^-1; rows r..lpad-1 of every whitened basis are zero.  One Cholesky
// pass on the leading r x r block then removes the cond_r eps loss of orthogonality of the first.
extern "C" int temd_basis_build_min_norm(temd_plan* p, const double* x, const double* x_unique, const double* mult,
                                         int nunique, const double* x_out, int* rank_host, double* sanity_host,
                                         void* stream) {
    if (p == nullptr || x_unique == nullptr || mult == nullptr || x_out == nullptr || nunique < 1)
        return temd_set_error(-1, "basis_build_min_norm: null argument or nunique < 1");
    if (x == nullptr && nunique != p->N)
        return temd_set_error(-1, "basis_build_min_norm: x = NULL (plan on the unique nodes) needs nunique = ncol = %d, got %d",
                              p->N, nunique);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    p->built = false;
    int rc = raw_basis(p, x ? x : x_unique, x_out, x ? nullptr : mult, st);
    if (rc) return rc;
    // Yw^T [lpad][ld_u] on the unique nodes; the vectors the SVD rotates are its rows (tall) or its columns (wide)
    const int U = nunique, Lp = p->Lp, lpad = p->lpad;
    const bool tall = U >= Lp;
    const size_t ld_u = round_up(U, 16);
    struct Scratch {
        void* ptr = nullptr;
        ~Scratch() { if (ptr) cudaFree(ptr); }
    } scratch;
    const size_t ywt_d = (size_t)lpad * ld_u, a_d = tall ? 0 : (size_t)U * lpad, vt_d = tall ? (size_t)lpad * lpad : 0;
    const size_t total_d = ywt_d + a_d + vt_d + 2 * (size_t)lpad;
    TEMD_CUDA(cudaMalloc(&scratch.ptr, total_d * sizeof(double) + 2 * sizeof(unsigned long long)));
    double* ywt = static_cast<double*>(scratch.ptr);
    double* a = ywt + ywt_d;
    double* vt = a + a_d;
    double* sigma = vt + vt_d;
    double* sigma_sorted = sigma + lpad;
    unsigned long long* off = reinterpret_cast<unsigned long long*>(sigma_sorted + lpad);
    if ((rc = launch_basis(x_unique, U, p->L, p->rec_a, p->rec_b, ywt, ld_u, lpad, st))) return temd_set_error(rc, "basis kernel launch failed");
    {
        dim3 grid((unsigned)((ld_u + 255) / 256), lpad);
        k_scale_cols_sqrt<<<grid, 256, 0, st>>>(ywt, mult, lpad, U, ld_u);
        TEMD_CUDA(cudaGetLastError());
    }
    int sweeps = 0;
    if (tall) {
        if ((rc = launch_identity(vt, lpad, lpad, st))) return temd_set_error(rc, "identity launch failed");
        rc = jacobi_svd_whitening(ywt, ld_u, U, Lp, vt, lpad, Lp, mult, U, p->linv2, lpad, sigma, sigma_sorted, p->status,
                                  off, &sweeps, st);
    } else {
        dim3 tb(32, 8), grid((U + 31) / 32, (Lp + 31) / 32);
        k_transpose<<<grid, tb, 0, st>>>(ywt, Lp, U, ld_u, a, lpad);
        TEMD_CUDA(cudaGetLastError());
        rc = jacobi_svd_whitening(a, lpad, Lp, U, nullptr, 0, Lp, mult, U, p->linv2, lpad, sigma, sigma_sorted, p->status,
                                  off, &sweeps, st);
    }
    if (rc) return rc;
    int rank = 0;
    TEMD_CUDA(cudaMemcpyAsync(&rank, p->status, sizeof(int), cudaMemcpyDeviceToHost, st));
    TEMD_CUDA(cudaStreamSynchronize(st));
    if (rank < 1 || rank > Lp) return temd_set_error(-5, "basis_build_min_norm: rank %d outside [1, %d]", rank, Lp);
    // pass 1: Q^T = W^T Y^T on both grids, written to qt / qpt
    if ((rc = launch_synth(p->linv2, lpad, lpad, lpad, p->qt_alt, p->N, p->ld_q, p->qt, p->ld_q, st))) return rc;
    if ((rc = launch_synth(p->linv2, lpad, lpad, lpad, p->qpt_alt, p->M, p->ld_p, p->qpt, p->ld_p, st))) return rc;
    TEMD_CUDA(cudaMemcpyAsync(p->linv, p->linv2, (size_t)lpad * lpad * sizeof(double), cudaMemcpyDeviceToDevice, st));
    // pass 2: Cholesky of the leading r x r block of Q^T Q
    if ((rc = gram_of(p, p->qt, st))) return rc;
    if ((rc = launch_chol_inv(p->gram, lpad, rank, p->lt, p->linv2, lpad, lpad, p->status, st))) return temd_set_error(rc, "cholesky launch failed");
    int status = 0;
    TEMD_CUDA(cudaMemcpyAsync(&status, p->status, sizeof(int), cudaMemcpyDeviceToHost, st));
    TEMD_CUDA(cudaStreamSynchronize(st));
    if (status != 0)
        return temd_set_error(-5, "basis_build_min_norm: Cholesky pivot %d of the rank-%d whitened basis non-positive "
                                  "(L = %d)", status - 1, rank, p->L);
    if ((rc = launch_synth(p->linv2, lpad, lpad, lpad, p->qt, p->N, p->ld_q, p->qt_alt, p->ld_q, st))) return rc;
    if ((rc = launch_synth(p->linv2, lpad, lpad, lpad, p->qpt, p->M, p->ld_p, p->qpt_alt, p->ld_p, st))) return rc;
    std::swap(p->qt, p->qt_alt);
    std::swap(p->qpt, p->qpt_alt);
    if ((rc = launch_matmul_small(p->linv2, p->linv, p->linv1, lpad, lpad, st))) return temd_set_error(rc, "matmul launch failed");
    std::swap(p->linv, p->linv1);
    if ((rc = finish_build(p, sanity_host, rank, st))) return rc;
    if (rank_host != nullptr) *rank_host = rank;
    return 0;
}

extern "C" int temd_basis_build_weighted(temd_plan* p, const double* x, const double* x_out, const double* w, void* stream) {
    if (p == nullptr || x == nullptr || x_out == nullptr || w == nullptr) return temd_set_error(-1, "basis_build_weighted: null argument");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    std::vector<double> ra(p->lpad, 0.0), rb(p->lpad, 0.0);
    const double PI = 3.141592653589793238462643383279502884;
    ra[0] = std::sqrt(1.0 / (4.0 * PI));
    if (p->L >= 1) ra[1] = std::sqrt(3.0 / (4.0 * PI));
    for (int l = 2; l <= p->L; l++) {
        ra[l] = std::sqrt(4.0 * l * l - 1.0) / l;
        rb[l] = ((l - 1.0) / l) * std::sqrt((2.0 * l + 1.0) / (2.0 * l - 3.0));
    }
    TEMD_CUDA(cudaMemcpyAsync(p->rec_a, ra.data(), p->lpad * sizeof(double), cudaMemcpyHostToDevice, st));
    TEMD_CUDA(cudaMemcpyAsync(p->rec_b, rb.data(), p->lpad * sizeof(double), cudaMemcpyHostToDevice, st));
    TEMD_CUDA(cudaStreamSynchronize(st));
    TEMD_CUDA(cudaMemcpyAsync(p->x, x, p->N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    TEMD_CUDA(cudaMemcpyAsync(p->x_out, x_out, p->M * sizeof(double), cudaMemcpyDeviceToDevice, st));
    int rc;
    if ((rc = launch_basis(p->x, p->N, p->L, p->rec_a, p->rec_b, p->qt, p->ld_q, p->lpad, st))) return temd_set_error(rc, "basis kernel launch failed");
    if ((rc = launch_basis(p->x_out, p->M, p->L, p->rec_a, p->rec_b, p->qpt, p->ld_p, p->lpad, st))) return temd_set_error(rc, "basis kernel launch failed");
    dim3 grid((unsigned)((p->ld_q + 255) / 256), p->lpad);
    k_scale_cols<<<grid, 256, 0, st>>>(p->qt, w, p->qt_alt, p->lpad, p->N, p->ld_q);
    TEMD_CUDA(cudaGetLastError());
    TEMD_CUDA(cudaStreamSynchronize(st));
    p->built = true;
    p->weighted = true;
    p->dqpt_built = false;
    p->rank = p->Lp;
    return 0;
}

extern "C" int temd_basis_export(temd_plan* p, double* Y0, double* Y0inv, double* Y0p, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "basis_export: basis not built");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    int rc;
    dim3 tb(32, 8);
    if (p->weighted) {
        if (Y0 != nullptr) {
            dim3 grid((p->N + 31) / 32, (p->Lp + 31) / 32);
            k_transpose<<<grid, tb, 0, st>>>(p->qt, p->Lp, p->N, p->ld_q, Y0, p->Lp);
        }
        if (Y0p != nullptr) {
            dim3 grid((p->M + 31) / 32, (p->Lp + 31) / 32);
            k_transpose<<<grid, tb, 0, st>>>(p->qpt, p->Lp, p->M, p->ld_p, Y0p, p->Lp);
        }
        if (Y0inv != nullptr)
            TEMD_CUDA(cudaMemcpy2DAsync(Y0inv, (size_t)p->N * sizeof(double), p->qt_alt, p->ld_q * sizeof(double),
                                        (size_t)p->N * sizeof(double), p->Lp, cudaMemcpyDeviceToDevice, st));
        TEMD_CUDA(cudaGetLastError());
        return 0;
    }
    if (Y0 != nullptr) {
        if ((rc = launch_basis(p->x, p->N, p->L, p->rec_a, p->rec_b, p->qt_alt, p->ld_q, p->lpad, st))) return temd_set_error(rc, "basis kernel launch failed");
        dim3 grid((p->N + 31) / 32, (p->Lp + 31) / 32);
        k_transpose<<<grid, tb, 0, st>>>(p->qt_alt, p->Lp, p->N, p->ld_q, Y0, p->Lp);
    }
    if (Y0p != nullptr) {
        if ((rc = launch_basis(p->x_out, p->M, p->L, p->rec_a, p->rec_b, p->qpt_alt, p->ld_p, p->lpad, st))) return temd_set_error(rc, "basis kernel launch failed");
        dim3 grid((p->M + 31) / 32, (p->Lp + 31) / 32);
        k_transpose<<<grid, tb, 0, st>>>(p->qpt_alt, p->Lp, p->M, p->ld_p, Y0p, p->Lp);
    }
    if (Y0inv != nullptr) {
        // Y0inv = L^-T Q^T : rows l of (Linv^T)[l][l'] = Linv[l'][l]
        dim3 grid((p->lpad + 31) / 32, (p->lpad + 31) / 32);
        k_transpose<<<grid, tb, 0, st>>>(p->linv, p->lpad, p->lpad, p->lpad, p->lt, p->lpad);
        if ((rc = launch_synth(p->lt, p->Lp, p->lpad, p->lpad, p->qt, p->N, p->ld_q, p->qt_alt, p->ld_q, st))) return rc;
        TEMD_CUDA(cudaMemcpy2DAsync(Y0inv, (size_t)p->N * sizeof(double), p->qt_alt, p->ld_q * sizeof(double),
                                    (size_t)p->N * sizeof(double), p->Lp, cudaMemcpyDeviceToDevice, st));
    }
    TEMD_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int temd_project(temd_plan* p, const double* const* fields_host, int nfields, int rows, size_t ld,
                            const double* lev_scale, int scale_field, int nlev, double* coef, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "project: basis not built (call temd_basis_build)");
    if (fields_host == nullptr || coef == nullptr || rows < 1 || nfields < 1 || nfields > TEMD_MAX_FIELDS || ld < (size_t)p->N)
        return temd_set_error(-1, "project: bad arguments (nfields %d, rows %d, ld %zu, ncol %d)", nfields, rows, ld, p->N);
    if (lev_scale != nullptr && nlev < 1) return temd_set_error(-1, "project: nlev must be >= 1 with lev_scale");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    int ntb, lblocks;
    project_lblocks(p->lpad, &ntb, &lblocks);
    const int tiles = ((rows + 127) / 128) * nfields;
    const int nchunks = (p->N + 15) / 16;
    const int nsplit = project_pick_split(tiles * lblocks, nchunks, p->sms, 64);
    double* work = nullptr;
    int rc = ensure_work(p, st, project_workspace_doubles(nfields, rows, p->lpad, nsplit), &work);
    if (rc) return rc;
    return launch_project(fields_host, nfields, rows, p->N, ld, p->weighted ? p->qt_alt : p->qt, p->lpad, p->ld_q, coef, work, nsplit,
                          lev_scale, scale_field, nlev < 1 ? 1 : nlev, st);
}

extern "C" int temd_synth_out(temd_plan* p, const double* coef, int rows, double* out, size_t ld_out, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "synth_out: basis not built");
    if (coef == nullptr || out == nullptr || rows < 1 || ld_out < (size_t)p->M) return temd_set_error(-1, "synth_out: bad arguments");
    TEMD_ON_DEVICE(p->dev);
    return launch_synth(coef, rows, p->lpad, p->lpad, p->qpt, p->M, p->ld_p, out, ld_out, reinterpret_cast<cudaStream_t>(stream));
}

// whitened derivative basis on the output grid: dQp^T = Linv * dY0p^T (quadrature mode: the raw derivative basis)
static int ensure_dqpt(temd_plan* p, cudaStream_t st) {
    if (p->dqpt_built) return 0;
    if (p->dqpt == nullptr) TEMD_CUDA(cudaMalloc(&p->dqpt, (size_t)p->lpad * p->ld_p * sizeof(double)));
    int rc;
    double* raw = p->weighted ? p->dqpt : p->qpt_alt;
    if ((rc = launch_basis_dlat(p->x_out, p->M, p->L, p->rec_a, p->rec_b, raw, p->ld_p, p->lpad, st))) return temd_set_error(rc, "basis_dlat launch failed");
    if (!p->weighted && (rc = launch_synth(p->linv, p->lpad, p->lpad, p->lpad, raw, p->M, p->ld_p, p->dqpt, p->ld_p, st))) return rc;
    p->dqpt_built = true;
    return 0;
}

extern "C" int temd_synth_out_dlat(temd_plan* p, const double* coef, int rows, double* out, size_t ld_out, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "synth_out_dlat: basis not built");
    if (coef == nullptr || out == nullptr || rows < 1 || ld_out < (size_t)p->M) return temd_set_error(-1, "synth_out_dlat: bad arguments");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    int rc = ensure_dqpt(p, st);
    if (rc) return rc;
    return launch_synth(coef, rows, p->lpad, p->lpad, p->dqpt, p->M, p->ld_p, out, ld_out, st);
}

extern "C" int temd_basis_export_dlat(temd_plan* p, double* dY0p, void* stream) {
    if (p == nullptr || !p->built || dY0p == nullptr) return temd_set_error(-1, "basis_export_dlat: basis not built / null output");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    int rc;
    if ((rc = launch_basis_dlat(p->x_out, p->M, p->L, p->rec_a, p->rec_b, p->qpt_alt, p->ld_p, p->lpad, st))) return temd_set_error(rc, "basis_dlat launch failed");
    dim3 tb(32, 8), grid((p->M + 31) / 32, (p->Lp + 31) / 32);
    k_transpose<<<grid, tb, 0, st>>>(p->qpt_alt, p->Lp, p->M, p->ld_p, dY0p, p->Lp);
    TEMD_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int temd_synth_native(temd_plan* p, const double* coef, int rows, double* out, size_t ld_out, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "synth_native: basis not built");
    if (coef == nullptr || out == nullptr || rows < 1 || ld_out < (size_t)p->N) return temd_set_error(-1, "synth_native: bad arguments");
    TEMD_ON_DEVICE(p->dev);
    const bool use_res = [] { const char* e = getenv("TEMD_SYNTH_RESIDENT"); return !(e && atoi(e) == 0); }();   // read per call: A/B in one process
    if (use_res) {
        const int rc = launch_synth_resident(coef, rows, p->lpad, p->lpad, p->qt, p->N, p->ld_q, out, ld_out, p->sms,
                                             reinterpret_cast<cudaStream_t>(stream));
        if (rc == 1) return 0;
        if (rc != 0) return rc;
    }
    return launch_synth(coef, rows, p->lpad, p->lpad, p->qt, p->N, p->ld_q, out, ld_out, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int temd_check_finite(const double* data, size_t n, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (data == nullptr) return temd_set_error(-1, "check_finite: null argument");
    // run on the device that owns `data`, whatever the caller's current device is
    cudaPointerAttributes attr;
    TEMD_CUDA(cudaPointerGetAttributes(&attr, data));
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)
        return temd_set_error(-1, "check_finite: data must be a device pointer");
    const int dev = attr.device;
    if (dev < 0 || dev >= 64) return temd_set_error(-1, "check_finite: device index out of range");
    TEMD_ON_DEVICE(dev);
    // one persistent 4-byte flag per device (never freed: cudaFree would synchronise the whole device); calls on one
    // device are serialised by the mutex because the flag is shared
    static int* flags[64] = {nullptr};
    static std::mutex mu[64];
    std::lock_guard<std::mutex> lock(mu[dev]);
    if (flags[dev] == nullptr) TEMD_CUDA(cudaMalloc(&flags[dev], sizeof(int)));
    int* flag = flags[dev];
    TEMD_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    const unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, 1184);
    k_check_finite<<<blocks ? blocks : 1, 256, 0, st>>>(data, n, flag);
    int h = 0;
    cudaError_t e = cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return temd_set_error((int)e, "check_finite: %s", cudaGetErrorString(e));
    if (h & 1) return temd_set_error(-2, "NaN values found");
    if (h & 2) return temd_set_error(-6, "infinite values found (no NaN)");
    return 0;
}

namespace temd { struct EpilogueArgs { temd_epilogue_args a; }; }

// Shared by temd_eddy_flux_project (nprod = 3: fields u, v, T, omega -> u'v', u'omega', v'theta') and
// temd_tracer_flux_project (nprod = 4: fields q1, q2, v, omega -> q1'v', q1'omega', q2'v', q2'omega').
static int eddy_flux_impl(temd_plan* p, const double* const* x4, int rows, size_t ld, const double* coef4,
                          const double* lev_scale, int nlev, double* coef_flux, int nprod, cudaStream_t st) {
    const int nchunks = (p->N + 15) / 16;
    // Two implementations of the same contraction (results agree to rounding):
    //   fused  one kernel, eddies and products never leave the SM (k_eddy): best while the 4 x 32 x lpad coefficient
    //          tile fits in shared memory (L + 1 <= 104), 32 B of HBM traffic per point;
    //   split  k_synth with the eddy epilogue writes the four eddy fields of a row batch to a scratch buffer,
    //          k_project in product mode reads them back and projects the products (96 B per point, still far
    //          below the FP64 roofline for L >= 104): both are plain GEMM pipelines whose tile shapes do not shrink with L.
    const int mode = [] {          // read at every call: lets one process A/B both implementations
        const char* e = getenv("TEMD_EDDY_MODE");
        return (e && !strcmp(e, "fused")) ? 1 : (e && !strcmp(e, "split")) ? 2 : 0;
    }();
    const bool can_fuse = eddy_supported(p->lpad) && (nprod == 3 || p->lpad <= 104);
    const bool split = (mode == 2) || !can_fuse || (mode == 0 && p->lpad > 104);
    if (!split) {
        const int nsplit = eddy_pick_split(rows, p->lpad, nchunks, p->sms, nprod);
        double* work = nullptr;
        int rc = ensure_work(p, st, eddy_workspace_doubles(rows, p->lpad, nsplit, nprod), &work);
        if (rc) return rc;
        return launch_eddy_flux_project(x4, rows, p->N, ld, p->qt, p->lpad, p->ld_q, coef4, coef_flux, work, nsplit,
                                        lev_scale, nlev, nprod, st);
    }
    // ---- split path, in row batches bounded by the scratch budget
    const double scratch_gb = [] { const char* e = getenv("TEMD_EDDY_SCRATCH_GB"); return (e && atof(e) > 0) ? atof(e) : 16.0; }();
    const size_t ld_e = round_up(p->N, 2);
    size_t rb = (size_t)(scratch_gb * 1073741824.0 / (4.0 * ld_e * sizeof(double)));
    rb = rb / 128 * 128;
    if (rb < 128) rb = 128;
    if (rb > (size_t)rows) rb = rows;
    double* scratch = nullptr;
    int rc = ensure_work(p, st, 4 * rb * ld_e, &scratch, 1);
    if (rc) return rc;
    double* e4[4] = {scratch, scratch + rb * ld_e, scratch + 2 * rb * ld_e, scratch + 3 * rb * ld_e};
    int ntb, lblocks;
    project_lblocks(p->lpad, &ntb, &lblocks);
    for (size_t r0 = 0; r0 < (size_t)rows; r0 += rb) {
        const int nr = (int)std::min(rb, (size_t)rows - r0);
        const double* xb[4] = {x4[0] + r0 * ld, x4[1] + r0 * ld, x4[2] + r0 * ld, x4[3] + r0 * ld};
        if ((rc = launch_synth_eddy4(coef4, rows, (int)r0, nr, p->lpad, p->qt, p->N, p->ld_q, xb, ld, lev_scale, 2, nlev, e4, ld_e, st)))
            return rc;
        const int tiles = ((nr + 127) / 128) * nprod;
        const int nsplit = project_pick_split(tiles * lblocks, nchunks, p->sms, 64);
        const size_t part_d = project_workspace_doubles(nprod, nr, p->lpad, nsplit), tmp_d = (size_t)nprod * nr * p->lpad;
        double* work = nullptr;
        if ((rc = ensure_work(p, st, part_d + tmp_d, &work))) return rc;
        const double* pairs3[6] = {e4[0], e4[1], e4[0], e4[3], e4[1], e4[2]};                   // u'v', u'omega', v'theta'
        const double* pairs4[8] = {e4[0], e4[2], e4[0], e4[3], e4[1], e4[2], e4[1], e4[3]};     // q1'v', q1'w', q2'v', q2'w'
        double* tmp = (nr == rows) ? coef_flux : work + part_d;
        if ((rc = launch_project_products(nprod == 3 ? pairs3 : pairs4, nprod, nr, p->N, ld_e, p->qt, p->lpad, p->ld_q, tmp, work,
                                          nsplit, st)))
            return rc;
        if (nr != rows)
            TEMD_CUDA(cudaMemcpy2DAsync(coef_flux + r0 * p->lpad, (size_t)rows * p->lpad * sizeof(double), tmp,
                                        (size_t)nr * p->lpad * sizeof(double), (size_t)nr * p->lpad * sizeof(double), nprod,
                                        cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

extern "C" int temd_eddy_flux_project(temd_plan* p, const double* u, const double* v, const double* t, const double* w,
                                      int rows, size_t ld, const double* coef4, const double* lev_scale, int nlev,
                                      double* coef_flux, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "eddy_flux_project: basis not built");
    if (!u || !v || !t || !w || !coef4 || !coef_flux || rows < 1 || ld < (size_t)p->N)
        return temd_set_error(-1, "eddy_flux_project: bad arguments");
    if (p->weighted) return temd_set_error(-1, "eddy_flux_project: not available with the quadrature-weights inverse (TEMDiagnostics never uses it)");
    TEMD_ON_DEVICE(p->dev);
    const double* x4[4] = {u, v, t, w};
    return eddy_flux_impl(p, x4, rows, ld, coef4, lev_scale, nlev, coef_flux, 3, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int temd_tracer_flux_project(temd_plan* p, const double* q1, const double* q2, const double* v, const double* w,
                                        int rows, size_t ld, const double* coef4, double* coef_flux, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "tracer_flux_project: basis not built");
    if (!q1 || !q2 || !v || !w || !coef4 || !coef_flux || rows < 1 || ld < (size_t)p->N)
        return temd_set_error(-1, "tracer_flux_project: bad arguments");
    if (p->weighted) return temd_set_error(-1, "tracer_flux_project: not available with the quadrature-weights inverse");
    TEMD_ON_DEVICE(p->dev);
    const double* x4[4] = {q1, q2, v, w};
    return eddy_flux_impl(p, x4, rows, ld, coef4, nullptr, 1, coef_flux, 4, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int temd_tem_epilogue(temd_plan* p, const temd_epilogue_args* args, void* stream) {
    if (p == nullptr || args == nullptr) return temd_set_error(-1, "tem_epilogue: null argument");
    if (args->nlev < 2 || args->nlat < 2 || args->nt < 1 || args->ld < (size_t)args->nlat)
        return temd_set_error(-1, "tem_epilogue: need nlev >= 2, nlat >= 2, nt >= 1 (np.gradient needs two points)");
    TEMD_ON_DEVICE(p->dev);
    EpilogueArgs w;
    w.a = *args;
    int rc = launch_tem_epilogue(w, reinterpret_cast<cudaStream_t>(stream));
    if (rc) return temd_set_error(rc, "tem_epilogue: kernel launch failed");
    return 0;
}

extern "C" int temd_eddy_native(temd_plan* p, const double* x, size_t ld_x, const double* coef, int rows,
                                const double* lev_scale, int nlev, double* out, size_t ld_out, void* stream) {
    if (p == nullptr || !p->built) return temd_set_error(-1, "eddy_native: basis not built");
    if (!x || !coef || !out || rows < 1 || ld_x < (size_t)p->N || ld_out < (size_t)p->N) return temd_set_error(-1, "eddy_native: bad arguments");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TEMD_ON_DEVICE(p->dev);
    int rc = launch_synth(coef, rows, p->lpad, p->lpad, p->qt, p->N, p->ld_q, out, ld_out, st);
    if (rc) return rc;
    dim3 grid((p->N + 255) / 256, rows < 32768 ? rows : 32768);
    k_eddy_native<<<grid, 256, 0, st>>>(x, ld_x, lev_scale, nlev < 1 ? 1 : nlev, out, ld_out, rows, p->N);
    TEMD_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int temd_multiply(const double* a, size_t ld_a, const double* b, size_t ld_b, double* out, size_t ld_out,
                             int rows, int ncol, void* stream) {
    if (!a || !b || !out || rows < 1 || ncol < 1) return temd_set_error(-1, "multiply: bad arguments");
    dim3 grid((ncol + 255) / 256, rows < 32768 ? rows : 32768);
    k_mul<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a, ld_a, b, ld_b, out, ld_out, rows, ncol);
    TEMD_CUDA(cudaGetLastError());
    return 0;
}

namespace temd { int launch_tracer_epilogue(const temd_tracer_args& a, cudaStream_t stream); }

extern "C" int temd_tracer_epilogue(temd_plan* p, const temd_tracer_args* args, void* stream) {
    if (p == nullptr || args == nullptr) return temd_set_error(-1, "tracer_epilogue: null argument");
    if (args->nlev < 2 || args->nlat < 2 || args->nt < 1 || args->ld < (size_t)args->nlat)
        return temd_set_error(-1, "tracer_epilogue: need nlev >= 2, nlat >= 2, nt >= 1");
    TEMD_ON_DEVICE(p->dev);
    int rc = launch_tracer_epilogue(*args, reinterpret_cast<cudaStream_t>(stream));
    if (rc) return temd_set_error(rc, "tracer_epilogue: kernel launch failed");
    return 0;
}

namespace temd {
int launch_group_sums(const double* const* x, int nfields, int rows, size_t ld, const int* perm, const int* goff,
                      int ngroups, int max_count, int min_count, int even_groups, const double* rsq, const double* lev_scale,
                      int scale_field, int nlev, int with_products, double* out, size_t ld_out, cudaStream_t stream);
int launch_dedup_flux(const double* gs, size_t ld_gs, const double* mw, size_t ld_m, const int* goff, const double* rsq,
                      int rows, int ngroups, double* out, size_t ld_o, cudaStream_t stream);
int launch_dedup_expand(const double* x, size_t ld_x, const double* scale, int nlev, const double* mw, size_t ld_m,
                        const int* gid, const double* rsq, double alpha, double beta, double* out, size_t ld_out, int rows,
                        int n, cudaStream_t stream);
}

extern "C" int temd_group_sums(const double* const* fields_host, int nfields, int rows, size_t ld, const int* perm,
                               const int* goff, int ngroups, int max_count, int min_count, int even_groups, const double* rsq,
                               const double* lev_scale, int scale_field, int nlev, int with_products, double* out,
                               size_t ld_out, void* stream) {
    if (!fields_host || !goff || !rsq || !out || nfields < 1 || nfields > 4 || rows < 1 || ngroups < 1 ||
        ld_out < (size_t)ngroups || min_count < 1 || max_count < min_count)
        return temd_set_error(-1, "group_sums: bad arguments");
    if (with_products && nfields != 4) return temd_set_error(-1, "group_sums: the flux sums need the four fields u, v, T, omega");
    for (int f = 0; f < nfields; f++) if (!fields_host[f]) return temd_set_error(-1, "group_sums: null field");
    const int rc = launch_group_sums(fields_host, nfields, rows, ld, perm, goff, ngroups, max_count, min_count, even_groups, rsq, lev_scale,
                                     lev_scale ? scale_field : -1, nlev, with_products, out, ld_out,
                                     reinterpret_cast<cudaStream_t>(stream));
    if (rc) return temd_set_error(rc, "group_sums: kernel launch failed");
    return 0;
}

extern "C" int temd_dedup_flux(const double* gsums, size_t ld_gs, const double* means_w, size_t ld_m, const int* goff,
                               const double* rsq, int rows, int ngroups, double* out, size_t ld_out, void* stream) {
    if (!gsums || !means_w || !goff || !rsq || !out || rows < 1 || ngroups < 1 || ld_gs < (size_t)ngroups ||
        ld_m < (size_t)ngroups || ld_out < (size_t)ngroups)
        return temd_set_error(-1, "dedup_flux: bad arguments");
    const int rc = launch_dedup_flux(gsums, ld_gs, means_w, ld_m, goff, rsq, rows, ngroups, out, ld_out,
                                     reinterpret_cast<cudaStream_t>(stream));
    if (rc) return temd_set_error(rc, "dedup_flux: kernel launch failed");
    return 0;
}

extern "C" int temd_dedup_expand(const double* x, size_t ld_x, const double* lev_scale, int nlev, const double* means_w,
                                 size_t ld_m, const int* gid, const double* rsq, double alpha, double beta, double* out,
                                 size_t ld_out, int rows, int ncol, void* stream) {
    if (!means_w || !gid || !out || rows < 1 || ncol < 1 || ld_out < (size_t)ncol || (x && ld_x < (size_t)ncol))
        return temd_set_error(-1, "dedup_expand: bad arguments");
    const int rc = launch_dedup_expand(x, ld_x, lev_scale, nlev, means_w, ld_m, gid, rsq, alpha, beta, out, ld_out, rows, ncol,
                                       reinterpret_cast<cudaStream_t>(stream));
    if (rc) return temd_set_error(rc, "dedup_expand: kernel launch failed");
    return 0;
}

extern "C" int temd_synth_fields(double* out, int field, int seed, int t0, int nt, int nlev, int ncol, size_t ld,
                                 const double* lat_rad, const double* lon_rad, const double* plev_hpa, void* stream) {
    if (!out || !lat_rad || !lon_rad || !plev_hpa || field < 0 || field > 4 || nt < 1 || nlev < 1 || ncol < 1 || ld < (size_t)ncol)
        return temd_set_error(-1, "synth_fields: bad arguments");
    int rc = launch_synth_fields(out, field, seed, t0, nt, nlev, ncol, ld, lat_rad, lon_rad, plev_hpa,
                                 reinterpret_cast<cudaStream_t>(stream));
    if (rc) return temd_set_error(rc, "synth_fields: kernel launch failed");
    return 0;
}

// Host-side helper for ordinary (pageable) input arrays: a multi-threaded memcpy into a pinned staging buffer, so
// that the host->device copy that follows is a true asynchronous DMA (a single-threaded pageable cudaMemcpy reaches
// ~10 GB/s on the test box, the pinned DMA 55 GB/s).  Pure host code; no arithmetic.
extern "C" int temd_host_copy(void* dst, const void* src, size_t bytes, int nthreads) {
    if (dst == nullptr || src == nullptr) return temd_set_error(-1, "host_copy: null argument");
    if (nthreads < 1) nthreads = 1;
    const size_t min_chunk = (size_t)4 << 20;
    size_t nt = (bytes + min_chunk - 1) / min_chunk;
    if (nt > (size_t)nthreads) nt = (size_t)nthreads;
    if (nt <= 1) { memcpy(dst, src, bytes); return 0; }
    const size_t chunk = ((bytes + nt - 1) / nt + 63) & ~(size_t)63;
    std::vector<std::thread> th;
    th.reserve(nt);
    for (size_t i = 0; i < nt; i++) {
        const size_t off = i * chunk;
        if (off >= bytes) break;
        const size_t len = (off + chunk <= bytes) ? chunk : bytes - off;
        th.emplace_back([=] { memcpy(static_cast<char*>(dst) + off, static_cast<const char*>(src) + off, len); });
    }
    for (auto& t : th) t.join();
    return 0;
}
