// K5 `eddy_flux_project`: fused native-grid synthesis -> eddies -> flux products -> projection.
//
// Replaces, in one pass over the four input fields (reference PyTEMDiags/tem_diagnostics.py):
//   _decompose_zm_eddy  :517-529   X' = X - ZM.sph_zonal_mean_native(X)   (X = ua, va, theta, wap)
//   _compute_fluxes     :547-557   upvp = up*vp, upwapp = up*wapp, vptp = vp*thetap  and the first
//                                  GEMM of their zonal means (sph_zonal_mean.py:251)
// The reference materialises 4 native means, 4 eddies and 3 products (11 N x K x T arrays); here
// none of them reaches HBM.  Per CTA: BM (time,lev) rows, a split-K range of 16-column chunks.
//
//   per chunk:  GEMM1  E_f[BM x 16] = X_f - C_f[BM x lpad] * QT[lpad x 16]   f = u, v, theta, omega (theta: X = lev_scale * T;
//                      the accumulators start from the X tile and the resident coefficients are negated),
//               E_f written in place over the X tile
//               GEMM2  acc_g[BM x lpad] += (E_a .* E_b)[BM x 16] * QT^T[16 x lpad]   g = uv, uw, v.theta
//
// Both GEMMs are DMMA.8x8x4; the QT chunk tile ([lpad rows][16 cols], TMA, 128-B swizzle) is the
// B operand of both: "MN-major" (contraction over tile rows) in GEMM1, "K-major" in GEMM2.
// C_f lives in shared memory for the CTA's lifetime (row-major, row stride = 4 or 12 mod 16
// doubles so that the GEMM1 A fragments are bank-conflict-free under the mnmajor_k permutation).
//
// Warp organisation (measured choices, see DESIGN.md §6): 16 consumer warps + 1 TMA producer warp; the
// 4 (BM=32) / 8 (BM=16) warps that own one 8-row m-tile form a group that synchronises on its own named
// barrier for the GEMM1 -> GEMM2 hand-off; one barrier round covers two pipeline stages when four stages fit
// (GEMM1 of both chunks shares the coefficient fragments).  BM = 32 / 16 / 8 rows for L+1 <= 104 / 208 / 408 is
// dictated by the 4 x BM x lpad coefficient tile that must stay resident next to >= 2 pipeline stages.
// Tried and rejected (slower): predicated per-(tile, product) work splitting to balance GEMM2 across a group
// (27.0 vs 32.6 TFLOP/s: predicated DMMA + WARPSYNC), run-time selection between loop shapes inside one kernel
// (ptxas schedules both worse; loop shapes are template parameters instead), splitting GEMM2 over k-steps as
// well as degrees inside a group (21 accumulator tiles per warp spill under the 120-register cap of 17 warps:
// 27.9 TFLOP/s), explicit software pipelining of the GEMM1 fragment loads (two register sets: 80.1 vs 78.5 ms, ptxas'
// own schedule of the unrolled loop is better), and a look-ahead schedule (GEMM1 of chunk i+1 before GEMM2 of chunk i, group hand-off through an
// mbarrier waited one phase later so that no warp idles at a barrier: 30.2 TFLOP/s - the barrier is not the limiter).
#include <cstdlib>
#include <type_traits>

#include "temd_common.cuh"
#include "temd_internal.h"

namespace temd {

constexpr int ED_SMEM_LIMIT = 232448 - 2048;   // 227 KB minus alignment slack and static barriers
constexpr int ED_MAX_STAGES = 6;

struct EddyMaps {
    CUtensorMap x[4];   // dims {N, rows}, box {16, BM}
    CUtensorMap q;      // dims {N, lpad}, box {16, min(lpad, 256)}
};

struct EddyParams {
    int rows, nchunks, chunks_per_split, nsplit;
    int nt;            // lpad / 8
    int ls;            // Cs row stride (doubles)
    int stages;
    int nlev;
    int qbox;          // rows per QT TMA box (divides lpad, <= 256)
    int nch;           // chunks per barrier round (2 needs >= 4 pipeline stages)
    const double* coef4;      // [4][rows][lpad]
    const double* lev_scale;  // [nlev] or null
    double* part;             // [nsplit][3][rows][lpad]
};

__host__ __device__ inline int eddy_ls(int lpad) {
    int ls = lpad;
    while ((ls & 15) != 4 && (ls & 15) != 12) ls++;
    return ls;
}

// GEMM2 inner step for one 16-column chunk: CNT (<= NJ) n8-tiles of this warp.
//   NP = 3 (TEM): products u'v', u'omega', v'theta' of the fields (u, v, theta, omega).  PAIRED: the eddy phase already
//       left v'theta' in the theta tile and u'omega' in the omega tile (see below), so only u'v' is formed here.
//   NP = 4 (tracer pair): fields (q1, q2, v, omega), products q1'v', q1'omega', q2'v', q2'omega'
//       (tem_diagnostics.py:560-570 for two tracers at once: v' and omega' are synthesised once for both).
template <int CNT, int NJ, int XF_BYTES, bool PAIRED, int NP>
__device__ __forceinline__ void eddy_gemm2(double (&acc)[NP][NJ][2], uint32_t st, uint32_t qs, uint32_t e_row_off,
                                           const uint32_t (&coff2)[4], int g, int j_begin) {
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
        const uint32_t eo = st + e_row_off + coff2[kk];
        const double e0 = lds64(eo);
        const double e1 = lds64(eo + XF_BYTES);
        const double e2 = lds64(eo + 2 * XF_BYTES);
        const double e3 = lds64(eo + 3 * XF_BYTES);
        double a[NP];
        if constexpr (NP == 3) {
            a[0] = e0 * e1;
            a[1] = PAIRED ? e3 : e0 * e3;
            a[2] = PAIRED ? e2 : e1 * e2;
        } else {
            a[0] = e0 * e2; a[1] = e0 * e3; a[2] = e1 * e2; a[3] = e1 * e3;
        }
        const uint32_t bo = qs + (uint32_t)((j_begin * 8 + g) * TILE_ROW_BYTES) + coff2[kk];
        double b[CNT];
#pragma unroll
        for (int jj = 0; jj < CNT; jj++) b[jj] = lds64(bo + (uint32_t)jj * 8u * TILE_ROW_BYTES);
#pragma unroll
        for (int jj = 0; jj < CNT; jj++)
#pragma unroll
            for (int q = 0; q < NP; q++) dmma(acc[q][jj][0], acc[q][jj][1], a[q], b[jj]);
    }
}

// Producer warps: with 16 consumer warps a single extra warp would put 5 warps on one SM sub-partition and cap every
// thread at 96 registers (16384 / 5 / 32, rounded down to 8).  A full producer WARPGROUP instead lets the kernel
// re-balance with setmaxnreg: the 4 producer warps drop to 24 registers, the 16 consumers rise to 112.  The CTA's
// register pool is what it was launched with (640 threads x 96): 512 x 112 + 128 x 24 = 60416 <= 61440.  (A target
// the pool cannot satisfy makes setmaxnreg.inc spin forever.)
template <int WARPS> constexpr int eddy_producer_warps() { return WARPS == 16 ? 4 : 1; }

template <int BM, int NJ, int WARPS, bool TWO, int NP>
__global__ void __launch_bounds__((WARPS + eddy_producer_warps<WARPS>()) * 32, 1)
k_eddy(const __grid_constant__ EddyMaps maps, const EddyParams p) {
    constexpr int MT = BM / 8;          // m8-tiles per CTA
    constexpr int PW = eddy_producer_warps<WARPS>();
    constexpr int NW2 = WARPS / MT;     // warps per m-tile group (2, 4, 8 or 16)
    // GEMM1: a group owns 8 units (4 fields x 2 n8-tiles of the 16-column chunk) of its m-tile
    //   NW2 = 2: 2 fields x 2 n-tiles per warp;  NW2 = 4: 2 fields x 1 n-tile (fewest LDS per DMMA once two chunks
    //   share the coefficient fragments);  NW2 = 8: 1 field x 1 n-tile
    constexpr int NF1 = (NW2 <= 4) ? 2 : 1;   // fields per warp
    constexpr int NN1 = (NW2 == 2) ? 2 : 1;   // n8-tiles per warp
    constexpr int XF_BYTES = BM * TILE_ROW_BYTES;   // one field's X tile
    static_assert(NW2 == 2 || NW2 == 4 || NW2 == 8, "unsupported warp layout");
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ __align__(8) uint64_t bars[2 * ED_MAX_STAGES];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lpad = p.nt * 8;
    const int stage_bytes = 4 * XF_BYTES + p.nt * 8 * TILE_ROW_BYTES;
    const int ntiles = (p.rows + BM - 1) / BM;
    const int tile = blockIdx.x % ntiles;
    const int split = blockIdx.x / ntiles;
    const int row0 = tile * BM;
    const int c_begin = split * p.chunks_per_split;
    const int c_end = min(c_begin + p.chunks_per_split, p.nchunks);
    const int nloc = c_end - c_begin;
    const int STAGES = p.stages;

    const uint32_t smem_base = smem_u32(smem), bar_base = smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (ED_MAX_STAGES + s); };
    double* Cs = reinterpret_cast<double*>(smem + (size_t)STAGES * stage_bytes);
    const uint32_t cs_base = smem_base + STAGES * stage_bytes;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), WARPS); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp >= WARPS) {
        // ------------------------------ TMA producer ------------------------------
        if constexpr (PW == 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 24;\n");
        if (warp == WARPS && lane == 0) {
            for (int f = 0; f < 4; f++) tma_prefetch_desc(&maps.x[f]);
            tma_prefetch_desc(&maps.q);
            for (int i = 0; i < nloc; i++) {
                const int s = i % STAGES;
                mbar_wait(empty_bar(s), ((i / STAGES) & 1) ^ 1);
                mbar_arrive_expect_tx(full_bar(s), stage_bytes);
                const uint32_t dst = smem_base + s * stage_bytes;
                const int col = (c_begin + i) * TILE_K;
#pragma unroll
                for (int f = 0; f < 4; f++) tma_load_2d(dst + f * XF_BYTES, &maps.x[f], col, row0, full_bar(s));
                for (int r = 0; r < lpad; r += p.qbox)
                    tma_load_2d(dst + 4 * XF_BYTES + r * TILE_ROW_BYTES, &maps.q, col, r, full_bar(s));
            }
        }
        return;
    }

    // ------------------------------ consumers ------------------------------
    if constexpr (PW == 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 112;\n");
    const int g = lane >> 2, t = lane & 3;
    const int tid = threadIdx.x;   // 0 .. WARPS*32-1
    // spectral coefficients of the 4 fields for this CTA's rows -> Cs[f][r][LS]
    // GEMM1 maps DMMA row g of an m-tile to physical tile row rho(g) = (g >> 1) | ((g & 1) << 2): the eight lanes of
    // a quarter-warp (g = 2q, 2q+1) then touch rows q and q+4, whose 128-B-swizzled 16-byte chunks fall in opposite
    // halves of the row, so the LDS.128 / STS.128 of the eddy phase take the minimum 4 wavefronts (the natural
    // mapping pairs rows 2q, 2q+1 on the same four chunks: 8 wavefronts, ncu r01_prof_eddy3).  Cs slot s therefore
    // holds the coefficients of row (s & ~7) + rho(s & 7).  GEMM2 reads the E tiles with the natural row mapping.
    for (int fr = warp; fr < 4 * BM; fr += WARPS) {
        const int f = fr / BM, rs = fr % BM;
        const int r = (rs & ~7) | ((rs & 7) >> 1) | ((rs & 1) << 2);
        const int row = row0 + r;
        const double* src = p.coef4 + ((size_t)f * p.rows + row) * lpad;
        double* dst = Cs + (size_t)fr * p.ls;
        // NEGATED: GEMM1 then accumulates x - C*QT directly on top of the X tile values (see round())
        for (int l = lane; l < lpad; l += 32) dst[l] = (row < p.rows) ? -src[l] : 0.0;
    }
    (void)tid;
    named_bar_sync(15, WARPS * 32);

    // Warp roles.  The warps that produce the eddies of m-tile `mi` (GEMM1) are exactly the warps that
    // consume them (GEMM2), so the E hand-off needs only a barrier among that group, not the whole
    // CTA.  Groups are laid out so that the warps sharing an SM sub-partition (warp % 4) belong to
    // different groups and carry complementary GEMM2 loads.
    const int mi = warp / NW2, r_in = warp % NW2;
    // fields: 0 = u, 1 = v, 2 = theta, 3 = omega.  With two fields per warp the pairs are {u, omega} and {v, theta}:
    // each warp can then form one flux product (u'omega' resp. v'theta') from its own registers in the eddy phase
    // and store it over the second field's tile, which nobody needs any more; GEMM2 multiplies only u'v'.
    constexpr bool PAIRED = (NF1 == 2) && (NP == 3);   // the tracer-pair mode needs every eddy twice: nothing to overwrite
    int fid[NF1];
    if (NF1 == 2) {                  // field pairs {0, 3} and {1, 2}: {u, omega} / {v, theta}, or {q1, omega} / {q2, v}
        const int pr = (NW2 == 2) ? r_in : (r_in & 1);
        fid[0] = pr;                 // u or v
        fid[NF1 - 1] = 3 - pr;       // omega or theta
    } else {
        fid[0] = (r_in >> 1) & 3;
    }
    const int jn1 = (NW2 == 2) ? 0 : (NW2 == 4 ? (r_in >> 1) : (r_in & 1));
    const int wq = (r_in + ((NW2 == 2) ? (mi >> 1) : mi)) % NW2;
    const int grp_bar = 1 + mi, grp_threads = NW2 * 32;
    const int j_begin = (wq * p.nt) / NW2;
    const int j_cnt = ((wq + 1) * p.nt) / NW2 - j_begin;      // NJ or NJ-1 (NJ = ceil(nt / NW2))

    // theta scale for this thread's row (field 2 only)
    const int g1 = (g >> 1) | ((g & 1) << 2);   // rho(g): physical row of this thread's GEMM1 accumulators
    double tscale = 1.0;
    {
        const int row = row0 + mi * 8 + g1;
        if (p.lev_scale != nullptr && row < p.rows) tscale = p.lev_scale[row % p.nlev];
    }

    double acc[NP][NJ][2];
#pragma unroll
    for (int a = 0; a < NP; a++)
#pragma unroll
        for (int j = 0; j < NJ; j++) acc[a][j][0] = acc[a][j][1] = 0.0;

    // per-thread constant offsets
    const int k1c0 = mnmajor_k(t, 0), k1c1 = mnmajor_k(t, 1);
    uint32_t a1_off[NF1];   // GEMM1 A: Cs[(f*BM + mi*8 + g)][.]
#pragma unroll
    for (int ff = 0; ff < NF1; ff++) a1_off[ff] = cs_base + (uint32_t)((fid[ff] * BM + mi * 8 + g) * p.ls) * 8u;
    uint32_t coff2[4];
#pragma unroll
    for (int kk = 0; kk < 4; kk++) coff2[kk] = kmajor_col_off(g, t, kk);
    const uint32_t e_row_off = (uint32_t)((mi * 8 + g) * TILE_ROW_BYTES);
    const uint32_t q_off = 4 * XF_BYTES;

    // One barrier round handles NCH consecutive chunks (pipeline stages): GEMM1 of all of them (sharing the
    // coefficient fragments), their eddies, ONE group barrier, then GEMM2 of all of them.
    auto round = [&](auto nch_tag, int i) {
        constexpr int NCH = decltype(nch_tag)::value;
        uint32_t st[NCH], qs[NCH];
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            const int s = (i + c) % STAGES;
            mbar_wait(full_bar(s), ((i + c) / STAGES) & 1);
            st[c] = smem_base + s * stage_bytes;
            qs[c] = st[c] + q_off;
        }
        // ---------------- GEMM1: E = X - C * QT (contraction over l = QT tile rows) ----------------
        // The accumulators start from the X tile values (theta: lev_scale * T) and Cs holds -C, so the tensor pipe
        // delivers the eddies themselves: no FP64 subtract per element on the pipe DMMA shares with DADD/DFMA.
        double sacc[NCH][NF1][NN1][2];
#pragma unroll
        for (int c = 0; c < NCH; c++)
#pragma unroll
            for (int nn = 0; nn < NN1; nn++) {
                const uint32_t off = swz_off(mi * 8 + g1, (jn1 + nn) * 8 + 2 * t);
#pragma unroll
                for (int ff = 0; ff < NF1; ff++) {
                    double2 x = lds128(st[c] + fid[ff] * XF_BYTES + off);
                    if (fid[ff] == 2) { x.x *= tscale; x.y *= tscale; }
                    sacc[c][ff][nn][0] = x.x;
                    sacc[c][ff][nn][1] = x.y;
                }
            }
#pragma unroll 2
        for (int l8 = 0; l8 < p.nt; l8++) {
#pragma unroll
            for (int cc = 0; cc < 2; cc++) {
                const int kin = cc ? k1c1 : k1c0;           // row inside the 8-row group
                const int k = l8 * 8 + kin;
                double a[NF1], b[NCH][NN1];
#pragma unroll
                for (int ff = 0; ff < NF1; ff++) a[ff] = lds64(a1_off[ff] + (uint32_t)k * 8u);
#pragma unroll
                for (int c = 0; c < NCH; c++)
#pragma unroll
                    for (int nn = 0; nn < NN1; nn++) {
                        const int jn = jn1 + nn;
                        b[c][nn] = lds64(qs[c] + (uint32_t)k * TILE_ROW_BYTES + (uint32_t)((((jn * 4 + (g >> 1)) ^ kin) & 7) << 4) + (uint32_t)((g & 1) << 3));
                    }
#pragma unroll
                for (int c = 0; c < NCH; c++)
#pragma unroll
                    for (int ff = 0; ff < NF1; ff++)
#pragma unroll
                        for (int nn = 0; nn < NN1; nn++) dmma(sacc[c][ff][nn][0], sacc[c][ff][nn][1], a[ff], b[c][nn]);
            }
        }
        // ---------------- eddies (and, when paired, one flux product), in place over the X tiles ----------------
#pragma unroll
        for (int c = 0; c < NCH; c++)
#pragma unroll
            for (int nn = 0; nn < NN1; nn++) {
                const int row = mi * 8 + g1;
                const int col = (jn1 + nn) * 8 + 2 * t;
                const uint32_t off = swz_off(row, col);
                double e0[NF1], e1[NF1];
#pragma unroll
                for (int ff = 0; ff < NF1; ff++) {
                    e0[ff] = sacc[c][ff][nn][0];
                    e1[ff] = sacc[c][ff][nn][1];
                }
                sts128(st[c] + fid[0] * XF_BYTES + off, e0[0], e1[0]);
                if (PAIRED) sts128(st[c] + fid[NF1 - 1] * XF_BYTES + off, e0[0] * e0[NF1 - 1], e1[0] * e1[NF1 - 1]);
                else if (NF1 == 2) sts128(st[c] + fid[NF1 - 1] * XF_BYTES + off, e0[NF1 - 1], e1[NF1 - 1]);
            }
        named_bar_sync(grp_bar, grp_threads);

        // ---------------- GEMM2: acc += (E_a .* E_b) * QT^T (contraction over the 16 columns) ----------------
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            if (j_cnt == NJ) eddy_gemm2<NJ, NJ, XF_BYTES, PAIRED, NP>(acc, st[c], qs[c], e_row_off, coff2, g, j_begin);
            else eddy_gemm2<(NJ > 1 ? NJ - 1 : 1), NJ, XF_BYTES, PAIRED, NP>(acc, st[c], qs[c], e_row_off, coff2, g, j_begin);
        }
        // the E tiles were written through the generic proxy; order them before the next TMA refill
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int c = 0; c < NCH; c++) mbar_arrive(empty_bar((i + c) % STAGES));
        }
    };

    // TWO is a template parameter on purpose: with both loop shapes behind a run-time flag ptxas schedules
    // both of them worse (measured on the sibling kernel k_synth_res: 82 % -> 76 % of peak)
    int i = 0;
    if constexpr (TWO) {
        for (; i + 2 <= nloc; i += 2) round(std::integral_constant<int, 2>{}, i);
    }
    for (; i < nloc; i++) round(std::integral_constant<int, 1>{}, i);

    // ------------------------------ split-K partials ------------------------------
    const int row = row0 + mi * 8 + g;
    if (row < p.rows) {
#pragma unroll
        for (int a = 0; a < NP; a++) {
            double* out = p.part + (((size_t)split * NP + a) * p.rows + row) * lpad;
#pragma unroll
            for (int jj = 0; jj < NJ; jj++) {
                if (jj < j_cnt) *reinterpret_cast<double2*>(out + (j_begin + jj) * 8 + 2 * t) = make_double2(acc[a][jj][0], acc[a][jj][1]);
            }
        }
    }
}

// Row tile.  L + 1 <= 104: BM = 32 with 8 (default) / 16 warps and four stages.  TEMD_EDDY_BM=24 selects an
// experimental layout with 12 consumer warps (three 8-row groups of four warps: every SM sub-partition hosts three
// warps of three different groups, and the smaller X tiles leave room for FIVE pipeline stages, i.e. 1.5 barrier rounds
// of TMA look-ahead instead of one).  Measured on the config-2 slab: 80.4 ms against 78.5 ms for 8 fat warps - the
// four-warps-per-group role split costs more shared-memory traffic than the extra look-ahead returns.
// The tracer-pair kernel (nprod = 4) has only the BM = 32 layout: TEMD_EDDY_BM does not apply to it.
static int eddy_bm(int nt, int nprod) {
    if (nprod == 4) return 32;
    if (nt <= 13) {
        const char* e = getenv("TEMD_EDDY_BM");      // read per call: A/B in one process
        return (e && atoi(e) == 24) ? 24 : 32;
    }
    return nt <= 26 ? 16 : 8;
}

int eddy_supported(int lpad) { return lpad >= 8 && lpad / 8 <= 51; }

static int eddy_stages(int nt, int bm, int* smem_bytes) {
    const int lpad = nt * 8;
    const int cs_bytes = 4 * bm * eddy_ls(lpad) * 8;
    const int stage_bytes = 4 * bm * TILE_ROW_BYTES + lpad * TILE_ROW_BYTES;
    int stages = (ED_SMEM_LIMIT - cs_bytes) / stage_bytes;
    if (stages > ED_MAX_STAGES) stages = ED_MAX_STAGES;
    *smem_bytes = stages * stage_bytes + cs_bytes + 1024;
    return stages;
}

int eddy_pick_split(int rows, int lpad, int nchunks, int sms, int nprod) {
    const int bm = eddy_bm(lpad / 8, nprod);
    return project_pick_split((rows + bm - 1) / bm, nchunks, sms, 64);
}

size_t eddy_workspace_doubles(int rows, int lpad, int nsplit, int nprod) { return (size_t)nsplit * nprod * rows * lpad; }

template <int BM, int NJ, int WARPS, bool TWO, int NP>
static int launch_eddy_2(const EddyMaps& maps, const EddyParams& p, int smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(k_eddy<BM, NJ, WARPS, TWO, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    const int ntiles = (p.rows + BM - 1) / BM;
    k_eddy<BM, NJ, WARPS, TWO, NP><<<ntiles * p.nsplit, (WARPS + eddy_producer_warps<WARPS>()) * 32, smem, stream>>>(maps, p);
    return (int)cudaGetLastError();
}

template <int BM, int NJ, int WARPS>
static int launch_eddy_t(const EddyMaps& maps, const EddyParams& p, int smem, cudaStream_t stream) {
    return p.nch == 2 ? launch_eddy_2<BM, NJ, WARPS, true, 3>(maps, p, smem, stream)
                      : launch_eddy_2<BM, NJ, WARPS, false, 3>(maps, p, smem, stream);
}

// tracer-pair instantiation (4 products): BM = 32, 8 consumer warps, one chunk per round (the fourth accumulator set
// takes the registers the second chunk's GEMM1 accumulators would need)
template <int NJ>
static int launch_eddy_pair(const EddyMaps& maps, const EddyParams& p, int smem, cudaStream_t stream) {
    return launch_eddy_2<32, NJ, 8, false, 4>(maps, p, smem, stream);
}

int launch_eddy_flux_project(const double* const* x4, int rows, int ncol, size_t ld_x, const double* qt, int lpad,
                             size_t ld_q, const double* coef4, double* coef_flux, double* part, int nsplit,
                             const double* lev_scale, int nlev, int nprod, cudaStream_t stream) {
    if (nprod != 3 && nprod != 4) return temd_set_error(-1, "eddy_flux_project: nprod must be 3 (TEM) or 4 (tracer pair)");
    if (!eddy_supported(lpad)) return temd_set_error(-1, "eddy_flux_project: L+1 > 408 is not supported by the fused kernel");
    const int nt = lpad / 8;
    const int bm = eddy_bm(nt, nprod);
    EddyMaps maps;
    int rc;
    for (int f = 0; f < 4; f++)
        if ((rc = make_tma_2d(&maps.x[f], x4[f], (uint64_t)ncol, (uint64_t)rows, ld_x * sizeof(double), TILE_K, bm))) return rc;
    int qd = 1;   // largest divisor d of nt with 8 d <= 256
    for (int d = 1; d <= 32 && d <= nt; d++) if (nt % d == 0) qd = d;
    if ((rc = make_tma_2d(&maps.q, qt, (uint64_t)ncol, (uint64_t)lpad, ld_q * sizeof(double), TILE_K, qd * 8))) return rc;
    EddyParams p;
    p.qbox = qd * 8;
    p.rows = rows;
    p.nchunks = (ncol + TILE_K - 1) / TILE_K;
    p.nsplit = nsplit;
    p.chunks_per_split = (p.nchunks + nsplit - 1) / nsplit;
    p.nt = nt;
    p.ls = eddy_ls(lpad);
    p.nlev = nlev < 1 ? 1 : nlev;
    p.coef4 = coef4;
    p.lev_scale = lev_scale;
    p.part = part;
    int smem;
    p.stages = eddy_stages(nt, bm, &smem);
    if (p.stages < 2) return temd_set_error(-1, "eddy_flux_project: not enough shared memory for lpad = %d", lpad);
    p.nch = (p.stages >= 4) ? 2 : 1;
    { const char* e = getenv("TEMD_EDDY_NCH"); if (e && atoi(e) == 1) p.nch = 1; }
    // Consumer warps (measured, tools/kbench.py, config 2 slab): since GEMM1 accumulates on top of the X tile (no FP64
    // subtract in the eddy phase) 8 fat warps (2 fields x 2 n-tiles each, 0.75 LDS per DMMA) beat 16 thin ones at
    // BM = 32: 78.5 vs 82.9 ms (before that change: 80.7 vs 78.6).  BM = 16 keeps 16 warps (only reachable with
    // TEMD_EDDY_MODE=fused: L + 1 > 104 takes the split path); BM = 8 has only 8 GEMM1 units per chunk.
    int warps = (bm == 24) ? 12 : (bm == 16) ? 16 : 8;
    { const char* e = getenv("TEMD_EDDY_WARPS"); if (e && bm != 8 && bm != 24) warps = atoi(e) == 8 ? 8 : 16; }
    rc = -1;
    if (nprod == 4) {
        if (bm != 32) return temd_set_error(-1, "eddy_flux_project: the tracer-pair kernel needs BM = 32 (L + 1 <= 104)");
        p.nch = 1;
        const int nj = (nt + 1) / 2;
        switch (nj) {
#define PCASE(N) case N: rc = launch_eddy_pair<N>(maps, p, smem, stream); break;
            PCASE(1) PCASE(2) PCASE(3) PCASE(4) PCASE(5) PCASE(6) PCASE(7)
#undef PCASE
            default: break;
        }
        if (rc) return temd_set_error(rc, "eddy_flux_project: tracer-pair kernel launch failed (nj %d)", nj);
        return launch_reduce_partials(part, coef_flux, nsplit, 4, rows, lpad, nullptr, -1, 1, stream);
    }
    const int nw2 = warps / (bm / 8);
    const int nj = (nt + nw2 - 1) / nw2;
#define ED_CASE(BM_, NJ_, W_) if (bm == BM_ && nj == NJ_ && warps == W_) rc = launch_eddy_t<BM_, NJ_, W_>(maps, p, smem, stream);
#define ED_CASES7(BM_, W_) ED_CASE(BM_, 1, W_) ED_CASE(BM_, 2, W_) ED_CASE(BM_, 3, W_) ED_CASE(BM_, 4, W_) ED_CASE(BM_, 5, W_) ED_CASE(BM_, 6, W_) ED_CASE(BM_, 7, W_)
#define ED_CASES4(BM_, W_) ED_CASE(BM_, 1, W_) ED_CASE(BM_, 2, W_) ED_CASE(BM_, 3, W_) ED_CASE(BM_, 4, W_)
    ED_CASES7(32, 8) ED_CASES7(16, 8) ED_CASES7(8, 8) ED_CASES4(32, 16) ED_CASES4(16, 16) ED_CASES4(24, 12)
#undef ED_CASES7
#undef ED_CASES4
#undef ED_CASE
    if (rc) return temd_set_error(rc, "eddy_flux_project: kernel launch failed (bm %d, nj %d, warps %d)", bm, nj, warps);
    return launch_reduce_partials(part, coef_flux, nsplit, 3, rows, lpad, nullptr, -1, 1, stream);
}

}  // namespace temd
