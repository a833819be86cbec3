// K4 `project`: tall-K FP64 tensor-core GEMM   R[row][l] = sum_n X[row][n] * QT[l][n]
//
// Replaces the first GEMM of `np.matmul(np.matmul(Y, self.Y0inv), AA)` (reference
// PyTEMDiags/sph_zonal_mean.py:251) in the factored/whitened form of DESIGN.md: with the
// orthonormalised basis Q (QT = Q^T stored [Lpad][N], ncol contiguous) the spectral coefficients
// of a field are c = Q^T x.  rows = (time, lev) pairs of one field, n = native columns.
//
// Structure (B200): one CTA = 128 rows x (NTB*8) degrees x a contiguous range of 16-column
// chunks (split-K).  A producer warp streams [128 x 16] X boxes and [NTB*8 x 16] QT boxes through a
// STAGES-deep TMA/mbarrier ring (128-B swizzle); 8 consumer warps each own a 16-row strip and all
// NTB n8-tiles, issuing DMMA.8x8x4 from conflict-free LDS.64 fragments.  Split-K partials go to a
// workspace and are summed in a fixed order by `k_reduce_partials` (deterministic, no atomics).
#include <cstdlib>

#include "temd_common.cuh"
#include "temd_internal.h"

namespace temd {

constexpr int PROJ_BM = 128;

struct ProjMaps {
    CUtensorMap x[TEMD_MAX_FIELDS];   // per field: dims {N, rows}, box {16, 128}
    CUtensorMap q;                    // dims {N, Lpad}, box {16, NTB*8}
};

struct ProjParams {
    int rows;            // rows per field (DD)
    int tiles_per_field; // ceil(rows / 128)
    int nfields;
    int nchunks;         // ceil(N / 16)
    int chunks_per_split;
    int nsplit;
    int lpad;            // total padded degrees (multiple of 8)
    double* part;        // [nsplit][nfields][rows][lpad]
};

// PROD: "field" f is the element-wise product of the two arrays behind maps.x[2f] and maps.x[2f+1] (the eddy-flux
// products u'v', u'omega', v'theta' of tem_diagnostics.py:547-555 formed on the fly from eddy fields: the product
// arrays are never written).  A stage then holds two X tiles.
template <int NTB, bool PROD>
constexpr int proj_stage_bytes() { return ((PROD ? 2 : 1) * PROJ_BM + NTB * 8) * TILE_ROW_BYTES; }

template <int NTB, bool PROD>
constexpr int proj_stages() {
    int s = (200 * 1024) / proj_stage_bytes<NTB, PROD>();
    return s > 8 ? 8 : s;
}

template <int NTB, int WARPS, bool PROD>
__global__ void __launch_bounds__((WARPS + 1) * 32, 1)
k_project(const __grid_constant__ ProjMaps maps, const ProjParams p) {
    constexpr int MTW = PROJ_BM / 8 / WARPS;   // m8-tiles per consumer warp (2 with 8 warps, 1 with 16)
    constexpr int STAGES = proj_stages<NTB, PROD>();
    constexpr int STAGE_BYTES = proj_stage_bytes<NTB, PROD>();
    constexpr int XROWS = (PROD ? 2 : 1) * PROJ_BM;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-B alignment is required by the 128-B swizzle pattern
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ __align__(8) uint64_t bars[2 * STAGES];

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.tiles_per_field * p.nfields;
    const int tile = blockIdx.x % total_tiles;
    const int split = blockIdx.x / total_tiles;
    const int field = tile / p.tiles_per_field;
    const int row0 = (tile % p.tiles_per_field) * PROJ_BM;
    const int lblk = blockIdx.y;
    const int l0 = lblk * NTB * 8;
    const int c_begin = split * p.chunks_per_split;
    const int c_end = min(c_begin + p.chunks_per_split, p.nchunks);
    const int nloc = c_end - c_begin;

    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_base = smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), WARPS);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == WARPS) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            tma_prefetch_desc(&maps.x[PROD ? 2 * field : field]);
            tma_prefetch_desc(&maps.q);
            for (int i = 0; i < nloc; i++) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                mbar_wait(empty_bar(s), ph ^ 1);
                mbar_arrive_expect_tx(full_bar(s), STAGE_BYTES);
                const uint32_t dst = smem_base + s * STAGE_BYTES;
                const int col = (c_begin + i) * TILE_K;
                if constexpr (PROD) {
                    tma_load_2d(dst, &maps.x[2 * field], col, row0, full_bar(s));
                    tma_load_2d(dst + PROJ_BM * TILE_ROW_BYTES, &maps.x[2 * field + 1], col, row0, full_bar(s));
                } else {
                    tma_load_2d(dst, &maps.x[field], col, row0, full_bar(s));
                }
                tma_load_2d(dst + XROWS * TILE_ROW_BYTES, &maps.q, col, l0, full_bar(s));
            }
        }
        return;
    }

    // ------------------------------ DMMA consumers ------------------------------
    const int g = lane >> 2, t = lane & 3;
    double acc[MTW][NTB][2];
#pragma unroll
    for (int i = 0; i < MTW; i++)
#pragma unroll
        for (int j = 0; j < NTB; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    uint32_t coff[4];
#pragma unroll
    for (int kk = 0; kk < 4; kk++) coff[kk] = kmajor_col_off(g, t, kk);
    const uint32_t a_row_off = (warp * 8 * MTW + g) * TILE_ROW_BYTES;
    const uint32_t b_row_off = XROWS * TILE_ROW_BYTES + g * TILE_ROW_BYTES;

    for (int i = 0; i < nloc; i++) {
        const int s = i % STAGES;
        const uint32_t ph = (i / STAGES) & 1;
        mbar_wait(full_bar(s), ph);
        const uint32_t st = smem_base + s * STAGE_BYTES;
#pragma unroll
        for (int kk = 0; kk < 4; kk++) {
            double a[MTW], b[NTB];
#pragma unroll
            for (int i2 = 0; i2 < MTW; i2++) {
                a[i2] = lds64(st + a_row_off + i2 * 8 * TILE_ROW_BYTES + coff[kk]);
                if constexpr (PROD) a[i2] *= lds64(st + PROJ_BM * TILE_ROW_BYTES + a_row_off + i2 * 8 * TILE_ROW_BYTES + coff[kk]);
            }
#pragma unroll
            for (int j = 0; j < NTB; j++) b[j] = lds64(st + b_row_off + j * 8 * TILE_ROW_BYTES + coff[kk]);
#pragma unroll
            for (int j = 0; j < NTB; j++)
#pragma unroll
                for (int i2 = 0; i2 < MTW; i2++) dmma(acc[i2][j][0], acc[i2][j][1], a[i2], b[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty_bar(s));
    }

    // ------------------------------ epilogue: split-K partial ------------------------------
    double* out = p.part + ((size_t)split * p.nfields + field) * (size_t)p.rows * p.lpad;
#pragma unroll
    for (int i = 0; i < MTW; i++) {
        const int row = row0 + warp * 8 * MTW + i * 8 + g;
        if (row < p.rows) {
#pragma unroll
            for (int j = 0; j < NTB; j++) {
                const int l = l0 + j * 8 + 2 * t;
                if (l < p.lpad)
                    *reinterpret_cast<double2*>(out + (size_t)row * p.lpad + l) = make_double2(acc[i][j][0], acc[i][j][1]);
            }
        }
    }
}

// R[f][row][l] = rowscale * sum_s part[s][f][row][l]   (fixed summation order)
__global__ void k_reduce_partials(const double* __restrict__ part, double* __restrict__ out, int nsplit,
                                  size_t per_split, const double* __restrict__ lev_scale, int scale_field,
                                  int rows, int lpad, int nlev) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= per_split) return;
    double s = 0.0;
    for (int k = 0; k < nsplit; k++) s += part[(size_t)k * per_split + i];
    if (lev_scale != nullptr) {
        const size_t r = i / lpad;
        const int field = (int)(r / rows);
        if (field == scale_field) s *= lev_scale[(r % rows) % nlev];
    }
    out[i] = s;
}

int launch_reduce_partials(const double* part, double* out, int nsplit, int nfields, int rows, int lpad,
                           const double* lev_scale, int scale_field, int nlev, cudaStream_t stream) {
    const size_t per_split = (size_t)nfields * rows * lpad;
    k_reduce_partials<<<(unsigned)((per_split + 255) / 256), 256, 0, stream>>>(part, out, nsplit, per_split, lev_scale,
                                                                              scale_field, rows, lpad, nlev);
    const int rc = (int)cudaGetLastError();
    if (rc) return temd_set_error(rc, "reduce_partials: launch failed");
    return 0;
}

template <int NTB, int WARPS, bool PROD>
static int launch_project_w(const ProjMaps& maps, const ProjParams& p, int lblocks, cudaStream_t stream) {
    constexpr int smem = proj_stages<NTB, PROD>() * proj_stage_bytes<NTB, PROD>() + 1024;
    cudaError_t e = cudaFuncSetAttribute(k_project<NTB, WARPS, PROD>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    dim3 grid(p.tiles_per_field * p.nfields * p.nsplit, lblocks);
    k_project<NTB, WARPS, PROD><<<grid, (WARPS + 1) * 32, smem, stream>>>(maps, p);
    return (int)cudaGetLastError();
}

template <int NTB>
static int launch_project_t(const ProjMaps& maps, const ProjParams& p, int lblocks, bool prod, cudaStream_t stream) {
    // 8 measured faster (34.3 vs 33.9 TFLOP/s); read per call: A/B in one process
    const int warps = [] { const char* e = getenv("TEMD_PROJECT_WARPS"); return (e && atoi(e) == 16) ? 16 : 8; }();
    if (prod) return launch_project_w<NTB, 8, true>(maps, p, lblocks, stream);
    return warps == 8 ? launch_project_w<NTB, 8, false>(maps, p, lblocks, stream) : launch_project_w<NTB, 16, false>(maps, p, lblocks, stream);
}

// pick the l-block size: balanced blocks of at most 13 n8-tiles
void project_lblocks(int lpad, int* ntb, int* lblocks) {
    const int nt = lpad / 8;
    const int nb = (nt + 12) / 13;
    *lblocks = nb;
    *ntb = (nt + nb - 1) / nb;
}

// choose the split-K factor that minimises (waves x chunks per CTA) for `tiles` output tiles
int project_pick_split(int tiles, int nchunks, int sms, int max_split) {
    long best_cost = -1;
    int best = 1;
    for (int s = 1; s <= max_split && s <= nchunks; s++) {
        const long waves = ((long)tiles * s + sms - 1) / sms;
        const long cps = (nchunks + s - 1) / s;
        const long cost = waves * (cps + 24) + 2 * s;   // +24 chunks ~ prologue/epilogue per CTA
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = s; }
    }
    return best;
}

size_t project_workspace_doubles(int nfields, int rows, int lpad, int nsplit) {
    return (size_t)nsplit * nfields * rows * lpad;
}

// Host launcher.  x[f] are device pointers to [rows][ld_x] doubles (ld_x >= ncol, ld_x even);
// qt is [lpad][ld_q].  out: [nfields][rows][lpad].  prod: x holds 2 * nfields pointers and field f is x[2f] .* x[2f+1].
static int launch_project_impl(const double* const* x, int nfields, bool prod, int rows, int ncol, size_t ld_x, const double* qt,
                               int lpad, size_t ld_q, double* out, double* part, int nsplit, const double* lev_scale,
                               int scale_field, int nlev, cudaStream_t stream) {
    const int nmaps = prod ? 2 * nfields : nfields;
    if (nfields < 1 || nmaps > TEMD_MAX_FIELDS) return temd_set_error(-1, "project: nfields out of range");
    int ntb, lblocks;
    project_lblocks(lpad, &ntb, &lblocks);
    ProjMaps maps;
    for (int f = 0; f < nmaps; f++) {
        int rc = make_tma_2d(&maps.x[f], x[f], (uint64_t)ncol, (uint64_t)rows, ld_x * sizeof(double), TILE_K, PROJ_BM);
        if (rc) return rc;
    }
    for (int f = nmaps; f < TEMD_MAX_FIELDS; f++) maps.x[f] = maps.x[0];
    int rc = make_tma_2d(&maps.q, qt, (uint64_t)ncol, (uint64_t)lpad, ld_q * sizeof(double), TILE_K, ntb * 8);
    if (rc) return rc;
    ProjParams p;
    p.rows = rows;
    p.tiles_per_field = (rows + PROJ_BM - 1) / PROJ_BM;
    p.nfields = nfields;
    p.nchunks = (ncol + TILE_K - 1) / TILE_K;
    p.nsplit = nsplit;
    p.chunks_per_split = (p.nchunks + nsplit - 1) / nsplit;
    p.lpad = lpad;
    p.part = part;
    switch (ntb) {
#define CASE(N) case N: rc = launch_project_t<N>(maps, p, lblocks, prod, stream); break;
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13)
#undef CASE
        default: return temd_set_error(-1, "project: bad l-block size");
    }
    if (rc) return temd_set_error(rc, "project: kernel launch failed");
    return launch_reduce_partials(part, out, nsplit, nfields, rows, lpad, lev_scale, scale_field, nlev, stream);
}

int launch_project(const double* const* x, int nfields, int rows, int ncol, size_t ld_x, const double* qt,
                   int lpad, size_t ld_q, double* out, double* part, int nsplit, const double* lev_scale,
                   int scale_field, int nlev, cudaStream_t stream) {
    return launch_project_impl(x, nfields, false, rows, ncol, ld_x, qt, lpad, ld_q, out, part, nsplit, lev_scale, scale_field,
                               nlev, stream);
}

// out[f][row][l] = sum_n x[2f][row][n] x[2f+1][row][n] QT[l][n],  f < npairs (<= 4)
int launch_project_products(const double* const* xpairs, int npairs, int rows, int ncol, size_t ld_x, const double* qt,
                            int lpad, size_t ld_q, double* out, double* part, int nsplit, cudaStream_t stream) {
    return launch_project_impl(xpairs, npairs, true, rows, ncol, ld_x, qt, lpad, ld_q, out, part, nsplit, nullptr, -1, 1, stream);
}

}  // namespace temd
