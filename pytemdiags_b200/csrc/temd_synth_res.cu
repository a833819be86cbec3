// Native-grid synthesis with the coefficient tile resident in shared memory:  S[row][n] = sum_l C[row][l] * QT[l][n]
//
// Second GEMM of `np.matmul(np.matmul(Y, self.Y0inv), AA)` with Y = Y0 (reference
// PyTEMDiags/sph_zonal_mean.py:251 via sph_zonal_mean_native :285-290).  The contraction is short
// (lpad <= 208) and the output is N columns wide, so the generic tiled kernel (temd_synth.cu) restarts its
// pipeline every 64 columns; here a CTA keeps its BM x lpad coefficient tile in shared memory for its whole
// life and streams [lpad x 16] basis tiles through a TMA/mbarrier ring, writing a [BM x 16] output block per
// chunk.  Fragment scheme = GEMM1 of k_eddy (MN-major B operand, mnmajor_k permutation, Cs row stride = 4 or
// 12 mod 16 doubles).  HBM-write-bound for small L (8 B/pt), FP64-tensor-bound for L >~ 25.
#include <cstdlib>
#include <type_traits>

#include "temd_common.cuh"
#include "temd_internal.h"

namespace temd {

constexpr int SR_WARPS = 8;
constexpr int SR_THREADS = (SR_WARPS + 1) * 32;
constexpr int SR_MAX_STAGES = 8;

struct SynthResParams {
    int rows, ncol, nchunks, chunks_per_split, nsplit;
    int nt, ls, stages, qbox;
    const double* coef;   // [rows][lpad]
    double* out;          // [rows][ld_out]
    size_t ld_out;
};

static inline int sr_ls(int lpad) {
    int ls = lpad;
    while ((ls & 15) != 4 && (ls & 15) != 12) ls++;
    return ls;
}

template <int MTW, int NCHMAX>   // MTW: m8-tiles per warp (2 -> BM = 128, 1 -> BM = 64); NCHMAX: chunks per iteration (1, 2, 4)
__global__ void __launch_bounds__(SR_THREADS, MTW == 1 ? 2 : 1)      // BM = 64: two CTAs share an SM
k_synth_res(const __grid_constant__ CUtensorMap qmap, const SynthResParams p) {
    constexpr int BM = SR_WARPS * 8 * MTW;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ __align__(8) uint64_t bars[2 * SR_MAX_STAGES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lpad = p.nt * 8;
    const int stage_bytes = lpad * TILE_ROW_BYTES;
    const int ntiles = (p.rows + BM - 1) / BM;
    const int tile = blockIdx.x % ntiles, split = blockIdx.x / ntiles;
    const int row0 = tile * BM;
    const int c_begin = split * p.chunks_per_split;
    const int c_end = min(c_begin + p.chunks_per_split, p.nchunks);
    const int nloc = c_end - c_begin;
    const int STAGES = p.stages;
    const uint32_t smem_base = smem_u32(smem), bar_base = smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (SR_MAX_STAGES + s); };
    double* Cs = reinterpret_cast<double*>(smem + (size_t)STAGES * stage_bytes);
    const uint32_t cs_base = smem_base + STAGES * stage_bytes;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), SR_WARPS); }
        mbar_fence_init();
    }
    __syncthreads();
    if (warp == SR_WARPS) {
        if (lane == 0) {
            tma_prefetch_desc(&qmap);
            for (int i = 0; i < nloc; i++) {
                const int s = i % STAGES;
                mbar_wait(empty_bar(s), ((i / STAGES) & 1) ^ 1);
                mbar_arrive_expect_tx(full_bar(s), stage_bytes);
                const uint32_t dst = smem_base + s * stage_bytes;
                for (int r = 0; r < lpad; r += p.qbox) tma_load_2d(dst + r * TILE_ROW_BYTES, &qmap, (c_begin + i) * TILE_K, r, full_bar(s));
            }
        }
        return;
    }
    const int g = lane >> 2, t = lane & 3;
    for (int r = warp; r < BM; r += SR_WARPS) {
        const int row = row0 + r;
        const double* src = p.coef + (size_t)row * lpad;
        double* dst = Cs + (size_t)r * p.ls;
        for (int l = lane; l < lpad; l += 32) dst[l] = (row < p.rows) ? src[l] : 0.0;
    }
    named_bar_sync(1, SR_WARPS * 32);

    const int k1c0 = mnmajor_k(t, 0), k1c1 = mnmajor_k(t, 1);
    uint32_t a_off[MTW];
#pragma unroll
    for (int mi = 0; mi < MTW; mi++) a_off[mi] = cs_base + (uint32_t)((warp * 8 * MTW + mi * 8 + g) * p.ls) * 8u;

    // NCH chunks (pipeline stages) per iteration share the coefficient fragments
    auto round = [&](auto nch_tag, int i) {
        constexpr int NCH = decltype(nch_tag)::value;
        uint32_t qs[NCH];
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            const int s = (i + c) % STAGES;
            mbar_wait(full_bar(s), ((i + c) / STAGES) & 1);
            qs[c] = smem_base + s * stage_bytes;
        }
        double acc[NCH][MTW][2][2];
#pragma unroll
        for (int c = 0; c < NCH; c++)
#pragma unroll
            for (int mi = 0; mi < MTW; mi++)
#pragma unroll
                for (int jn = 0; jn < 2; jn++) acc[c][mi][jn][0] = acc[c][mi][jn][1] = 0.0;
#pragma unroll 2
        for (int l8 = 0; l8 < p.nt; l8++) {
#pragma unroll
            for (int cc = 0; cc < 2; cc++) {
                const int kin = cc ? k1c1 : k1c0;
                const int k = l8 * 8 + kin;
                double a[MTW], b[NCH][2];
#pragma unroll
                for (int mi = 0; mi < MTW; mi++) a[mi] = lds64(a_off[mi] + (uint32_t)k * 8u);
#pragma unroll
                for (int c = 0; c < NCH; c++)
#pragma unroll
                    for (int jn = 0; jn < 2; jn++)
                        b[c][jn] = lds64(qs[c] + (uint32_t)k * TILE_ROW_BYTES + (uint32_t)((((jn * 4 + (g >> 1)) ^ kin) & 7) << 4) + (uint32_t)((g & 1) << 3));
#pragma unroll
                for (int c = 0; c < NCH; c++)
#pragma unroll
                    for (int mi = 0; mi < MTW; mi++)
#pragma unroll
                        for (int jn = 0; jn < 2; jn++) dmma(acc[c][mi][jn][0], acc[c][mi][jn][1], a[mi], b[c][jn]);
            }
        }
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int c = 0; c < NCH; c++) mbar_arrive(empty_bar((i + c) % STAGES));
        }
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            const int col0 = (c_begin + i + c) * TILE_K;
#pragma unroll
            for (int mi = 0; mi < MTW; mi++) {
                const int row = row0 + warp * 8 * MTW + mi * 8 + g;
                if (row >= p.rows) continue;
#pragma unroll
                for (int jn = 0; jn < 2; jn++) {
                    const int col = col0 + jn * 8 + 2 * t;
                    double* dst = p.out + (size_t)row * p.ld_out + col;
                    if (col + 1 < p.ncol) *reinterpret_cast<double2*>(dst) = make_double2(acc[c][mi][jn][0], acc[c][mi][jn][1]);
                    else if (col < p.ncol) *dst = acc[c][mi][jn][0];
                }
            }
        }
    };
    int i = 0;
    if constexpr (NCHMAX >= 4) {
        for (; i + 4 <= nloc; i += 4) round(std::integral_constant<int, 4>{}, i);
    }
    if constexpr (NCHMAX >= 2) {
        for (; i + 2 <= nloc; i += 2) round(std::integral_constant<int, 2>{}, i);
    }
    for (; i < nloc; i++) round(std::integral_constant<int, 1>{}, i);
}

// returns 1 if this kernel handled the request, 0 if the caller should use the generic kernel, < 0 / > 0 on error
int launch_synth_resident(const double* c, int rows, int lpad, size_t ld_c, const double* b, int ncol, size_t ld_b,
                          double* out, size_t ld_out, int sms, cudaStream_t stream) {
    if (lpad > 104 || ld_c != (size_t)lpad || ncol < 1024) return 0;   // larger L: the generic kernel is faster (measured)
    if ((ld_out & 1) || (reinterpret_cast<uintptr_t>(out) & 15)) return 0;
    const int nt = lpad / 8;
    // 64-row tiles (MTW = 1) with few enough stages that TWO CTAs share an SM: measured on the config-5 sweep
    // 0.845 vs 0.822 of the FP64 peak at L = 100, 0.725 vs 0.718 at L = 50, 0.599 vs 0.605 at L = 25
    // (TEMD_SYNTH_RES_MTW=1|2 forces either; read per call, like TEMD_SYNTH_RES_NCH: A/B in one process).
    const int mtw_env = [] { const char* v = getenv("TEMD_SYNTH_RES_MTW"); return v ? atoi(v) : 0; }();
    const int mtw = (mtw_env == 1 || (mtw_env != 2 && nt > 4)) ? 1 : 2;
    const int bm = SR_WARPS * 8 * mtw;
    SynthResParams p;
    p.rows = rows; p.ncol = ncol;
    p.nchunks = (ncol + TILE_K - 1) / TILE_K;
    p.nt = nt; p.ls = sr_ls(lpad);
    int qd = 1;
    for (int d = 1; d <= 32 && d <= nt; d++) if (nt % d == 0) qd = d;
    p.qbox = qd * 8;
    const int cs_bytes = bm * p.ls * 8;
    const int stage_bytes = lpad * TILE_ROW_BYTES;
    p.stages = (232448 - 2048 - cs_bytes) / stage_bytes;
    if (p.stages > SR_MAX_STAGES) p.stages = SR_MAX_STAGES;
    if (mtw == 1) {       // keep the CTA under half an SM's shared memory
        while (p.stages > 2 && p.stages * stage_bytes + cs_bytes + 2048 > 113 * 1024) p.stages--;
    }
    if (p.stages < 2) return 0;
    const int smem = p.stages * stage_bytes + cs_bytes + 1024;
    const int ntiles = (rows + bm - 1) / bm;
    p.nsplit = project_pick_split(ntiles, p.nchunks, sms, 148);
    p.chunks_per_split = (p.nchunks + p.nsplit - 1) / p.nsplit;
    p.coef = c; p.out = out; p.ld_out = ld_out;
    CUtensorMap qmap;
    int rc = make_tma_2d(&qmap, b, (uint64_t)ncol, (uint64_t)lpad, ld_b * sizeof(double), TILE_K, p.qbox);
    if (rc) return rc;
    cudaError_t e = cudaSuccess;
    // two chunks per iteration pay off once the contraction is long enough (measured: L = 25 prefers one)
#define SR_LAUNCH(M_, T_)                                                                                         \
    do {                                                                                                          \
        e = cudaFuncSetAttribute(k_synth_res<M_, T_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);          \
        if (e != cudaSuccess) return temd_set_error((int)e, "synth_resident: cudaFuncSetAttribute failed");       \
        k_synth_res<M_, T_><<<ntiles * p.nsplit, SR_THREADS, smem, stream>>>(qmap, p);                             \
    } while (0)
    const int nch_env = [] { const char* v = getenv("TEMD_SYNTH_RES_NCH"); return v ? atoi(v) : 0; }();
    int nch = (nt > 4) ? 2 : 1;
    if (nch_env == 1 || nch_env == 2 || nch_env == 4) nch = nch_env;
    if (nch == 4 && p.stages < 8) nch = 2;
    if (mtw == 2 && nch == 4) SR_LAUNCH(2, 4);
    else if (mtw == 2 && nch == 2) SR_LAUNCH(2, 2);
    else if (mtw == 2) SR_LAUNCH(2, 1);
    else SR_LAUNCH(1, 2);
#undef SR_LAUNCH
    e = cudaGetLastError();
    if (e != cudaSuccess) return temd_set_error((int)e, "synth_resident: kernel launch failed");
    return 1;
}

}  // namespace temd
