"""Every kernel instantiation libtemd.so ships, launched on purpose and checked against a float64 reference.

The host dispatchers pick template instantiations of k_eddy, k_project and k_synth_res from L, the row count and
the TEMD_* knobs.  Each row of CASES names a problem (grid, K, T, L, tracers, knobs) and the instantiations it must
launch.  On the GPU a case proves which kernels ran (torch.profiler, CUDA activity only) and compares every output
plane with the float64 oracle at max|d| / max|ref| <= 1e-10.  On any machine, test_instantiation_ledger reads the
instantiations from the library's symbol table and requires each one to be named by a case or listed in
UNREACHABLE with the reason no input or knob selects it: a new instantiation cannot ship without a parity case.

Every case keeps the edges where tiles go wrong: rows = T*K is not a multiple of the row tile (15, 21, 25, 33, 150,
...; 5 rows is fewer than one BM = 8 tile), the column count is not a multiple of 16 (pg2 grids with odd ne), and
the native-synthesis cases run on 4,095 columns (91 x 45 lat-lon), so the single-element tail store of
k_synth_res executes.  Every case is also well conditioned (cond(Y0) <= 20, asserted): on an ill-conditioned basis two
float64 references (SVD pseudo-inverse, normal equations) already disagree by more than the 1e-10 bar - by 2e-8 in
etfy at L = 72 on ne9pg2, cond(Y0) = 537 - so that bar only measures the kernels on well-posed problems."""
import collections
import functools
import re
import subprocess

import numpy as np
import pytest

import oracle
from pytemdiags_b200 import synthetic as syn

TOL = 1e-10
MAX_COND = 20.0
ZM7 = ('ub', 'vb', 'thetab', 'wapb', 'upvpb', 'upwappb', 'vptpb')
TRACER_METHODS = ('etfy', 'etfz', 'etdiv', 'qtendetfd', 'qtendvtem', 'qtendwtem')
TRACER_PROPS = ('qb', 'qpvpb', 'qpwappb', 'dqb_dp')
KERNEL_RE = re.compile(r'temd::k_(?:eddy|project|synth_res)<[^>]*>')

Case = collections.namedtuple('Case', 'id kind grid K T L ntrac env kernels')
#   kind  'tem'     project + eddy_flux_project + synth_out: the seven ZM7 planes against oracle.tem_suite
#         'tracer'  TEMDiagnostics(q=[...]) against oracle.tem_suite(q=...) for every tracer, and the four planes of
#                   Engine.tracer_flux_project + synth_out against NumPy
#         'zonal'   Engine.project + synth_native / synth_out and sph_zonal_mean_native against Y0 Y0inv A, Y0p Y0inv A


def _ep(bm, nj, warps, two, nprod=3):
    return 'temd::k_eddy<%d, %d, %d, %s, %d>' % (bm, nj, warps, 'true' if two else 'false', nprod)


def _pj(ntb, warps=8, prod=False):
    return 'temd::k_project<%d, %d, %s>' % (ntb, warps, 'true' if prod else 'false')


def _sr(mtw, nch):
    return 'temd::k_synth_res<%d, %d>' % (mtw, nch)


def pg2(ne):
    return ('pg2', ne)


LATLON = ('latlon', 91, 45)       # 4,095 columns: odd, >= 1024 (the resident synthesis kernel's threshold)

# Dispatch, for nt = ceil((L + 1) / 8) n8-tiles of degrees:
#   k_eddy BM 32 (nt <= 13): 8 warps, NJ = ceil(nt / 2); 16 warps (TEMD_EDDY_WARPS=16), NJ = ceil(nt / 4);
#          BM 24 (TEMD_EDDY_BM=24): 12 warps, NJ = ceil(nt / 4);  tracer pair: <32, ceil(nt / 2), 8, false, 4>
#          BM 16 (nt 14-26, TEMD_EDDY_MODE=fused): 16 warps NJ = ceil(nt / 8); 8 warps NJ = ceil(nt / 4)
#          BM 8 (nt 27-51, fused): 8 warps, NJ = ceil(nt / 8)
#          TWO (two chunks per barrier round) whenever >= 4 pipeline stages fit, i.e. for nt <= 23 at BM 16 and
#          nt <= 34 at BM 8; TEMD_EDDY_NCH=1 turns it off
#   k_project NTB = ceil(nt / ceil(nt / 13)) n8-tiles per l-block; 8 warps, 16 with TEMD_PROJECT_WARPS=16; the
#          product mode (split eddy path: L + 1 > 104, or TEMD_EDDY_MODE=split) always has 8 warps
#   k_synth_res (lpad <= 104, ncol >= 1024): <2, 1> for nt <= 4, <1, 2> above; TEMD_SYNTH_RES_MTW=2 -> <2, NCH>
#          with NCH = TEMD_SYNTH_RES_NCH (default 2 for nt > 4); TEMD_SYNTH_RESIDENT=0 -> the generic k_synth
SPLIT = {'TEMD_EDDY_MODE': 'split'}
FUSED = {'TEMD_EDDY_MODE': 'fused'}
NCH1 = {'TEMD_EDDY_NCH': '1'}
BM24 = {'TEMD_EDDY_BM': '24'}
W16 = {'TEMD_EDDY_WARPS': '16'}
W8 = {'TEMD_EDDY_WARPS': '8'}
PW16 = {'TEMD_PROJECT_WARPS': '16'}


def _env(*ds, **kw):
    out = {}
    for d in ds:
        out.update(d)
    out.update(kw)
    return out


CASES = [
    # ---- tracer pair k_eddy<32, NJ, 8, false, 4>, NJ 1..7; three tracers: the odd one out takes the TEM kernel
    Case('pair_L6', 'tracer', pg2(5), 5, 3, 6, 3, {}, [_pj(1), _ep(32, 1, 8, True), _ep(32, 1, 8, False, 4)]),
    Case('pair_L20', 'tracer', pg2(5), 7, 5, 20, 3, {}, [_pj(3), _ep(32, 2, 8, True), _ep(32, 2, 8, False, 4)]),
    Case('pair_L40', 'tracer', pg2(7), 11, 3, 40, 3, {}, [_pj(6), _ep(32, 3, 8, True), _ep(32, 3, 8, False, 4)]),
    Case('pair_L60', 'tracer', pg2(11), 6, 5, 60, 3, {}, [_pj(8), _ep(32, 4, 8, True), _ep(32, 4, 8, False, 4)]),
    Case('pair_L72', 'tracer', pg2(13), 13, 3, 72, 3, {}, [_pj(10), _ep(32, 5, 8, True), _ep(32, 5, 8, False, 4)]),
    Case('pair_L88', 'tracer', pg2(15), 9, 4, 88, 3, {}, [_pj(12), _ep(32, 6, 8, True), _ep(32, 6, 8, False, 4)]),
    Case('pair_L103', 'tracer', pg2(17), 6, 5, 103, 3, {}, [_pj(13), _ep(32, 7, 8, True), _ep(32, 7, 8, False, 4)]),
    # four pairs and an odd tracer; the tracer projection is split 8 + 1
    Case('pair_9tracers', 'tracer', pg2(7), 7, 3, 40, 9, {}, [_pj(6), _ep(32, 3, 8, True), _ep(32, 3, 8, False, 4)]),
    # split path in pair mode, row batches of 128 + 22
    Case('pair_split_L180', 'tracer', pg2(33), 50, 3, 180, 3, {'TEMD_EDDY_SCRATCH_GB': '1e-6'},
         [_pj(12), _pj(12, prod=True)]),
    # TEMD_EDDY_BM=24 applies to the TEM kernel only; the pair kernel keeps BM = 32
    Case('pair_bm24', 'tracer', pg2(7), 11, 3, 40, 2, BM24, [_pj(6), _ep(24, 2, 12, True), _ep(32, 3, 8, False, 4)]),
    # ---- TEM flux, default paths
    Case('tem_L72', 'tem', pg2(13), 11, 3, 72, 0, {}, [_pj(10), _ep(32, 5, 8, True)]),
    Case('tem_L180', 'tem', pg2(33), 50, 3, 180, 0, {}, [_pj(12), _pj(12, prod=True)]),
    # ---- split path forced: product-mode k_project NTB 1..13
    Case('split_L6', 'tem', pg2(5), 7, 3, 6, 0, SPLIT, [_pj(1), _pj(1, prod=True)]),
    Case('split_L12', 'tem', pg2(5), 7, 3, 12, 0, SPLIT, [_pj(2), _pj(2, prod=True)]),
    Case('split_L20', 'tem', pg2(5), 7, 3, 20, 0, SPLIT, [_pj(3), _pj(3, prod=True)]),
    Case('split_L30', 'tem', pg2(7), 7, 3, 30, 0, SPLIT, [_pj(4), _pj(4, prod=True)]),
    Case('split_L36', 'tem', pg2(7), 7, 3, 36, 0, SPLIT, [_pj(5), _pj(5, prod=True)]),
    Case('split_L44', 'tem', pg2(7), 7, 3, 44, 0, SPLIT, [_pj(6), _pj(6, prod=True)]),
    Case('split_L54', 'tem', pg2(11), 7, 3, 54, 0, SPLIT, [_pj(7), _pj(7, prod=True)]),
    Case('split_L60', 'tem', pg2(11), 7, 3, 60, 0, SPLIT, [_pj(8), _pj(8, prod=True)]),
    Case('split_L70', 'tem', pg2(13), 7, 3, 70, 0, SPLIT, [_pj(9), _pj(9, prod=True)]),
    Case('split_L75', 'tem', pg2(13), 7, 3, 75, 0, SPLIT, [_pj(10), _pj(10, prod=True)]),
    Case('split_L84', 'tem', pg2(15), 7, 3, 84, 0, SPLIT, [_pj(11), _pj(11, prod=True)]),
    Case('split_L90', 'tem', pg2(15), 7, 3, 90, 0, SPLIT, [_pj(12), _pj(12, prod=True)]),
    Case('split_L100', 'tem', pg2(17), 7, 3, 100, 0, SPLIT, [_pj(13), _pj(13, prod=True)]),
    # ---- BM 32, 8 warps, one chunk per round (TEMD_EDDY_NCH=1), NJ 1..7
    Case('nch1_L6', 'tem', pg2(5), 9, 5, 6, 0, NCH1, [_pj(1), _ep(32, 1, 8, False)]),
    Case('nch1_L20', 'tem', pg2(5), 9, 5, 20, 0, NCH1, [_pj(3), _ep(32, 2, 8, False)]),
    Case('nch1_L36', 'tem', pg2(7), 9, 5, 36, 0, NCH1, [_pj(5), _ep(32, 3, 8, False)]),
    Case('nch1_L54', 'tem', pg2(11), 9, 5, 54, 0, NCH1, [_pj(7), _ep(32, 4, 8, False)]),
    Case('nch1_L70', 'tem', pg2(13), 9, 5, 70, 0, NCH1, [_pj(9), _ep(32, 5, 8, False)]),
    Case('nch1_L84', 'tem', pg2(15), 9, 5, 84, 0, NCH1, [_pj(11), _ep(32, 6, 8, False)]),
    Case('nch1_L100', 'tem', pg2(17), 9, 5, 100, 0, NCH1, [_pj(13), _ep(32, 7, 8, False)]),
    # ---- BM 24 / 12 warps (TEMD_EDDY_BM=24), NJ 1..4, both loop shapes; 25 rows = one 24-row tile + 1
    Case('bm24_L20', 'tem', pg2(5), 5, 5, 20, 0, BM24, [_pj(3), _ep(24, 1, 12, True)]),
    Case('bm24_L36', 'tem', pg2(7), 5, 5, 36, 0, BM24, [_pj(5), _ep(24, 2, 12, True)]),
    Case('bm24_L70', 'tem', pg2(13), 5, 5, 70, 0, BM24, [_pj(9), _ep(24, 3, 12, True)]),
    Case('bm24_L100', 'tem', pg2(17), 5, 5, 100, 0, BM24, [_pj(13), _ep(24, 4, 12, True)]),
    Case('bm24_nch1_L20', 'tem', pg2(5), 5, 5, 20, 0, _env(BM24, NCH1), [_pj(3), _ep(24, 1, 12, False)]),
    Case('bm24_nch1_L36', 'tem', pg2(7), 5, 5, 36, 0, _env(BM24, NCH1), [_pj(5), _ep(24, 2, 12, False)]),
    Case('bm24_nch1_L70', 'tem', pg2(13), 5, 5, 70, 0, _env(BM24, NCH1), [_pj(9), _ep(24, 3, 12, False)]),
    Case('bm24_nch1_L100', 'tem', pg2(17), 5, 5, 100, 0, _env(BM24, NCH1), [_pj(13), _ep(24, 4, 12, False)]),
    # ---- BM 32 with 16 consumer warps (TEMD_EDDY_WARPS=16), NJ 1..4, both loop shapes
    Case('w16_L7', 'tem', pg2(5), 6, 3, 7, 0, W16, [_pj(1), _ep(32, 1, 16, True)]),
    Case('w16_L40', 'tem', pg2(7), 6, 3, 40, 0, W16, [_pj(6), _ep(32, 2, 16, True)]),
    Case('w16_L72', 'tem', pg2(13), 6, 3, 72, 0, W16, [_pj(10), _ep(32, 3, 16, True)]),
    Case('w16_L103', 'tem', pg2(17), 6, 3, 103, 0, W16, [_pj(13), _ep(32, 4, 16, True)]),
    Case('w16_nch1_L7', 'tem', pg2(5), 6, 3, 7, 0, _env(W16, NCH1), [_pj(1), _ep(32, 1, 16, False)]),
    Case('w16_nch1_L40', 'tem', pg2(7), 6, 3, 40, 0, _env(W16, NCH1), [_pj(6), _ep(32, 2, 16, False)]),
    Case('w16_nch1_L72', 'tem', pg2(13), 6, 3, 72, 0, _env(W16, NCH1), [_pj(10), _ep(32, 3, 16, False)]),
    Case('w16_nch1_L103', 'tem', pg2(17), 6, 3, 103, 0, _env(W16, NCH1), [_pj(13), _ep(32, 4, 16, False)]),
    # ---- fused BM 16 (TEMD_EDDY_MODE=fused; the default takes the split path above L + 1 = 104)
    Case('fused16_w16_L110', 'tem', pg2(21), 5, 3, 110, 0, FUSED, [_pj(7), _ep(16, 2, 16, True)]),
    Case('fused16_w16_L155', 'tem', pg2(27), 5, 3, 155, 0, FUSED, [_pj(10), _ep(16, 3, 16, True)]),
    Case('fused16_w16_L190', 'tem', pg2(33), 5, 3, 190, 0, FUSED, [_pj(12), _ep(16, 3, 16, False)]),
    Case('fused16_w16_L207', 'tem', pg2(35), 5, 3, 207, 0, FUSED, [_pj(13), _ep(16, 4, 16, False)]),
    Case('fused16_w8_L110', 'tem', pg2(21), 5, 3, 110, 0, _env(FUSED, W8), [_pj(7), _ep(16, 4, 8, True)]),
    Case('fused16_w8_L155', 'tem', pg2(27), 5, 3, 155, 0, _env(FUSED, W8), [_pj(10), _ep(16, 5, 8, True)]),
    Case('fused16_w8_L170', 'tem', pg2(27), 5, 3, 170, 0, _env(FUSED, W8), [_pj(11), _ep(16, 6, 8, True)]),
    Case('fused16_w8_L190', 'tem', pg2(33), 5, 3, 190, 0, _env(FUSED, W8), [_pj(12), _ep(16, 6, 8, False)]),
    Case('fused16_w8_L207', 'tem', pg2(35), 5, 3, 207, 0, _env(FUSED, W8), [_pj(13), _ep(16, 7, 8, False)]),
    Case('fused16_w16_nch1_L110', 'tem', pg2(21), 5, 3, 110, 0, _env(FUSED, NCH1), [_pj(7), _ep(16, 2, 16, False)]),
    Case('fused16_w8_nch1_L110', 'tem', pg2(21), 5, 3, 110, 0, _env(FUSED, W8, NCH1), [_pj(7), _ep(16, 4, 8, False)]),
    Case('fused16_w8_nch1_L155', 'tem', pg2(27), 5, 3, 155, 0, _env(FUSED, W8, NCH1), [_pj(10), _ep(16, 5, 8, False)]),
    # ---- fused BM 8: 5 rows, fewer than one tile
    Case('fused8_L215', 'tem', pg2(37), 5, 1, 215, 0, FUSED, [_pj(9), _ep(8, 4, 8, True)]),
    Case('fused8_L260', 'tem', pg2(45), 5, 1, 260, 0, FUSED, [_pj(11), _ep(8, 5, 8, True)]),
    Case('fused8_L285', 'tem', pg2(49), 5, 1, 285, 0, FUSED, [_pj(12), _ep(8, 5, 8, False)]),
    Case('fused8_L350', 'tem', pg2(61), 5, 1, 350, 0, FUSED, [_pj(11), _ep(8, 6, 8, False)]),
    Case('fused8_L395', 'tem', pg2(69), 5, 1, 395, 0, FUSED, [_pj(13), _ep(8, 7, 8, False)]),
    Case('fused8_nch1_L215', 'tem', pg2(37), 5, 1, 215, 0, _env(FUSED, NCH1), [_pj(9), _ep(8, 4, 8, False)]),
    # ---- native synthesis on an odd column count >= 1024
    Case('native_L20', 'zonal', LATLON, 5, 3, 20, 0, {}, [_pj(3), _sr(2, 1)]),
    Case('native_L40', 'zonal', LATLON, 5, 3, 40, 0, {}, [_pj(6), _sr(1, 2)]),
    Case('native_mtw2_nch2_L20', 'zonal', LATLON, 5, 3, 20, 0, {'TEMD_SYNTH_RES_MTW': '2', 'TEMD_SYNTH_RES_NCH': '2'},
         [_pj(3), _sr(2, 2)]),
    Case('native_mtw2_nch4_L20', 'zonal', LATLON, 5, 3, 20, 0, {'TEMD_SYNTH_RES_MTW': '2', 'TEMD_SYNTH_RES_NCH': '4'},
         [_pj(3), _sr(2, 4)]),
    Case('native_mtw2_L40', 'zonal', LATLON, 5, 3, 40, 0, {'TEMD_SYNTH_RES_MTW': '2'}, [_pj(6), _sr(2, 2)]),
    Case('native_generic_L40', 'zonal', LATLON, 5, 3, 40, 0, {'TEMD_SYNTH_RESIDENT': '0'}, [_pj(6)]),
    # ---- projection with 16 consumer warps (TEMD_PROJECT_WARPS=16), NTB 1..13
    Case('project_w16_L6', 'zonal', pg2(7), 7, 3, 6, 0, PW16, [_pj(1, 16), _sr(2, 1)]),
    Case('project_w16_L12', 'zonal', pg2(7), 7, 3, 12, 0, PW16, [_pj(2, 16), _sr(2, 1)]),
    Case('project_w16_L20', 'zonal', pg2(7), 7, 3, 20, 0, PW16, [_pj(3, 16), _sr(2, 1)]),
    Case('project_w16_L30', 'zonal', pg2(7), 7, 3, 30, 0, PW16, [_pj(4, 16), _sr(2, 1)]),
    Case('project_w16_L36', 'zonal', pg2(7), 7, 3, 36, 0, PW16, [_pj(5, 16), _sr(1, 2)]),
    Case('project_w16_L44', 'zonal', pg2(7), 7, 3, 44, 0, PW16, [_pj(6, 16), _sr(1, 2)]),
    Case('project_w16_L54', 'zonal', pg2(11), 7, 3, 54, 0, PW16, [_pj(7, 16), _sr(1, 2)]),
    Case('project_w16_L60', 'zonal', pg2(11), 7, 3, 60, 0, PW16, [_pj(8, 16), _sr(1, 2)]),
    Case('project_w16_L70', 'zonal', pg2(13), 7, 3, 70, 0, PW16, [_pj(9, 16), _sr(1, 2)]),
    Case('project_w16_L75', 'zonal', pg2(13), 7, 3, 75, 0, PW16, [_pj(10, 16), _sr(1, 2)]),
    Case('project_w16_L84', 'zonal', pg2(15), 7, 3, 84, 0, PW16, [_pj(11, 16), _sr(1, 2)]),
    Case('project_w16_L90', 'zonal', pg2(15), 7, 3, 90, 0, PW16, [_pj(12, 16), _sr(1, 2)]),
    Case('project_w16_L100', 'zonal', pg2(17), 7, 3, 100, 0, PW16, [_pj(13, 16), _sr(1, 2)]),
]

_NS = 'no input or knob selects it: '
UNREACHABLE = {
    _ep(16, 1, 16, True): _NS + 'BM 16 starts at nt = 14, so 16 warps (8 per m-tile) give NJ = ceil(nt / 8) >= 2',
    _ep(16, 1, 16, False): _NS + 'BM 16 starts at nt = 14, so 16 warps give NJ >= 2',
    **{_ep(16, nj, 8, two): _NS + 'BM 16 starts at nt = 14, so 8 warps (4 per m-tile) give NJ = ceil(nt / 4) >= 4'
       for nj in (1, 2, 3) for two in (True, False)},
    **{_ep(8, nj, 8, two): _NS + 'BM 8 starts at nt = 27, so NJ = ceil(nt / 8) >= 4'
       for nj in (1, 2, 3) for two in (True, False)},
    _ep(16, 4, 16, True): _NS + 'NJ 4 with 16 warps means nt 25-26, where only 3 pipeline stages fit (one chunk per round)',
    _ep(16, 7, 8, True): _NS + 'NJ 7 with 8 warps at BM 16 means nt 25-26, where only 3 pipeline stages fit',
    _ep(8, 6, 8, True): _NS + 'NJ 6 at BM 8 means nt 41-48; fewer than 4 pipeline stages fit from nt = 35 on',
    _ep(8, 7, 8, True): _NS + 'NJ 7 at BM 8 means nt 49-51; fewer than 4 pipeline stages fit from nt = 35 on',
}


def nerr(x, ref):
    return float(np.abs(np.asarray(x) - ref).max() / max(np.abs(ref).max(), 1e-300))


# ------------------------------------------------------------------ ledger (no GPU needed)

def shipped_instantiations(lib_path):
    out = subprocess.run(['nm', '-C', lib_path], check=True, capture_output=True, text=True).stdout
    return set(KERNEL_RE.findall(out))


def test_instantiation_ledger(temd_lib):
    """The kernel instantiations in libtemd.so are exactly those the cases launch plus the listed unreachable ones."""
    from pytemdiags_b200 import _lib
    shipped = shipped_instantiations(_lib.LIB_PATH)
    assert len(shipped) > 100, 'symbol table of %s lists only %d kernel instantiations' % (_lib.LIB_PATH, len(shipped))
    covered = {k for c in CASES for k in c.kernels}
    assert not covered & set(UNREACHABLE), sorted(covered & set(UNREACHABLE))
    missing = shipped - covered - set(UNREACHABLE)
    assert not missing, 'instantiations without a parity case in CASES (or a reason in UNREACHABLE): %s' % sorted(missing)
    stale = (covered | set(UNREACHABLE)) - shipped
    assert not stale, 'names in CASES / UNREACHABLE that libtemd.so does not ship: %s' % sorted(stale)


def test_case_ids_unique():
    ids = [c.id for c in CASES]
    assert len(ids) == len(set(ids))


# ------------------------------------------------------------------ GPU parity per case

def _ncol(grid):
    return 24 * grid[1] ** 2 if grid[0] == 'pg2' else grid[1] * grid[2]


@functools.lru_cache(maxsize=2)
def _problem(grid, K, T, L, ntrac):
    """Inputs and float64 reference of one problem (shared by the cases that only change knobs)."""
    lat, lon = syn.make_grid(grid)
    N = lat.shape[0]
    plev = syn.default_plev(K)
    f = syn.synth_fields(lat, lon, plev, T, seed=1000 + L, fields=('ua', 'va', 'ta', 'wap', 'q'))
    rng = np.random.default_rng(L)
    qs = [f['q'] * (1.0 + 0.25 * i) + 1e-4 * rng.standard_normal(f['q'].shape) for i in range(ntrac - 1)]
    qs = (qs + [3e-4 * np.abs(f['va']) + 1e-5]) if ntrac else []
    lat_out = oracle.zm_latitudes(1)
    big = N > 6000
    mats = oracle.sph_matrices(lat, lat_out, L, method='normal' if big else 'pinv', basis='recurrence' if big else 'scipy')
    ev = np.linalg.eigvalsh(mats[0].T @ mats[0])
    assert np.sqrt(ev[-1] / ev[0]) <= MAX_COND, 'cond(Y0) = %.3g: pick a finer grid for L = %d' % (np.sqrt(ev[-1] / ev[0]), L)
    tr = lambda x: np.ascontiguousarray(x.transpose(2, 1, 0))
    ref = oracle.tem_suite(tr(f['ua']), tr(f['va']), tr(f['ta']), tr(f['wap']), plev, lat, L=L, literal=False,
                           matrices=mats, q=[tr(q) for q in qs] or None)
    return lat, plev, f, qs, lat_out, mats, ref


def _rows(a):
    """(T, K, N) host array -> [T*K][N] device view of an even-strided buffer (the TMA operands need it)."""
    import torch
    r = a.reshape(-1, a.shape[-1])
    n = r.shape[1]
    buf = torch.zeros((r.shape[0], n + (n & 1)), dtype=torch.float64, device='cuda')
    buf[:, :n] = torch.as_tensor(r).cuda()
    return buf[:, :n]


def _profiled(fn):
    """Run fn under torch.profiler (CUDA activity only); returns (fn(), every kernel name seen)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _zm_np(mats, A):
    """Y0p Y0inv A and the eddy A - Y0 Y0inv A for A = (N, rows)."""
    Y0, Y0inv, Y0p = mats
    c = Y0inv @ A
    return Y0p @ c, A - Y0 @ c


def _run_tem(case, prob):
    import torch
    from pytemdiags_b200.engine import Engine
    lat, plev, f, _, lat_out, _, ref = prob
    K, T = case.K, case.T
    C = oracle.CONSTANTS
    eng = Engine(lat, lat_out, case.L).build_basis()
    sc = torch.as_tensor((C['P0'] / (plev * 100)) ** C['k']).cuda()
    xs = [_rows(f[n]) for n in ('ua', 'va', 'ta', 'wap')]

    def run():
        c4 = eng.project(xs, lev_scale=sc, scale_field=2, nlev=K)
        cf = eng.eddy_flux_project(xs[0], xs[1], xs[2], xs[3], c4, sc, K)
        return eng.synth_out(torch.cat([c4, cf], 0)).cpu().numpy().reshape(7, T, K, -1)

    zm, seen = _profiled(run)
    errs = {n: nerr(zm[i].transpose(2, 1, 0), ref[n]) for i, n in enumerate(ZM7)}
    return errs, seen


def _run_tracer(case, prob):
    from pytemdiags_b200 import TEMDiagnostics
    from pytemdiags_b200.engine import Engine
    lat, plev, f, qs, lat_out, mats, ref = prob
    N, rows = lat.shape[0], case.K * case.T
    eng = Engine(lat, lat_out, case.L).build_basis()
    q1, q2, v, w = (_rows(x) for x in (qs[0], qs[1], f['va'], f['wap']))

    def run():
        tem = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, q=qs, L=case.L,
                             dims=('time', 'lev', 'ncol'), debug_level=0)
        got = {}
        for i in range(len(qs)):
            for m in TRACER_METHODS:
                got['%s%d' % (m, i)] = np.asarray(getattr(tem, m)(i))
            for p_ in TRACER_PROPS:
                got['%s%d' % (p_, i)] = np.asarray(getattr(tem, p_)[i])
        c4 = eng.project([q1, q2, v, w])
        fl = eng.tracer_flux_project(q1, q2, v, w, c4)
        return got, eng.synth_out(fl).cpu().numpy()

    (got, planes), seen = _profiled(run)
    errs = {}
    for n, x in got.items():
        assert x.shape == ref[n].shape, (n, x.shape, ref[n].shape)
        errs[n] = nerr(x, ref[n])
    # Y0p Y0inv (q' .* v'), (q' .* omega') of the first pair, q' = q - Y0 Y0inv q
    eddy = {n: _zm_np(mats, x.reshape(rows, N).T)[1] for n, x in (('q1', qs[0]), ('q2', qs[1]), ('v', f['va']),
                                                                   ('w', f['wap']))}
    for k, (a_, b_) in enumerate((('q1', 'v'), ('q1', 'w'), ('q2', 'v'), ('q2', 'w'))):
        errs["pair %s'%s'" % (a_, b_)] = nerr(planes[k].T, _zm_np(mats, eddy[a_] * eddy[b_])[0])
    return errs, seen


def _run_zonal(case, prob):
    from pytemdiags_b200 import sph_zonal_averager
    from pytemdiags_b200.engine import Engine
    lat, _, f, _, lat_out, mats, _ = prob
    N, rows = lat.shape[0], case.K * case.T
    A = np.ascontiguousarray(f['ua'].reshape(rows, N).T)            # (N, rows)
    ref_out = _zm_np(mats, A)[0]
    ref_nat = A - _zm_np(mats, A)[1]
    eng = Engine(lat, lat_out, case.L).build_basis()
    x = _rows(f['ua'])

    def run():
        c = eng.project([x])[0]
        ZM = sph_zonal_averager(lat, lat_out, case.L)
        ZM.sph_compute_matrices()
        return eng.synth_native(c).cpu().numpy(), eng.synth_out(c).cpu().numpy(), ZM.sph_zonal_mean_native(A)

    (nat, out, pub), seen = _profiled(run)
    assert nat.shape == (rows, N) and pub.shape == (N, rows)
    errs = {'synth_native': nerr(nat.T, ref_nat), 'synth_out': nerr(out.T, ref_out),
            'sph_zonal_mean_native': nerr(pub, ref_nat)}
    return errs, seen


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=[c.id for c in CASES])
def test_instantiation_parity(monkeypatch, case):
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    prob = _problem(case.grid, case.K, case.T, case.L, case.ntrac)
    assert prob[0].shape[0] == _ncol(case.grid)
    errs, seen = {'tem': _run_tem, 'tracer': _run_tracer, 'zonal': _run_zonal}[case.kind](case, prob)
    ran = {k for n in seen for k in KERNEL_RE.findall(n)}
    missing = [k for k in case.kernels if k not in ran]
    assert not missing, 'expected %s to run; the profiler saw: %s' % (missing, sorted(seen))
    if case.env.get('TEMD_SYNTH_RESIDENT') == '0':
        assert not any('k_synth_res' in n for n in ran), sorted(ran)
        assert any('temd::k_synth(' in n for n in seen), sorted(seen)
    bad = {n: e for n, e in errs.items() if not e <= TOL}
    assert not bad, bad
    print('%s: worst %.2e (%s)' % (case.id, max(errs.values()), max(errs, key=errs.get)))
