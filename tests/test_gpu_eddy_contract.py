"""Every eddy-flux kernel body against a direct float64 contraction on the plan's own basis.

`eddy_flux_project` (and `tracer_flux_project`) take caller-supplied coefficients C and compute, with Q the plan's
whitened basis ([N][lpad], read back exactly as Q^T = synth_native(I): every output is one product with 1):

    E_f[r][n]  = s_f(r) X_f[r][n] - sum_l C_f[r][l] Q[n][l]      s = lev_scale[r % nlev] for theta, else 1
    cf_g[r][l] = sum_n Q[n][l] E_a[r][n] E_b[r][n]               g = (u,v), (u,w), (v,theta)  |  pair: (q1,v), (q1,w), (q2,v), (q2,w)

With white-noise X and random C of the same size at every degree, the eddies are O(1), every degree tile and every
column contributes O(1) and the float64 reference has no cancellation, so the coefficient planes are compared directly
(a degree permutation shows up as itself) at max|d| / max|ref| <= 1e-12 per plane; the expected error is about
eps * sqrt(N) of the plane's maximum.  The project's 1e-10 oracle bar also carries basis-conditioning error.

Each case states the instantiation it must launch (torch.profiler, CUDA activity).  For k_eddy it also reads the launch
grid from the exported trace and checks grid.x / ceil(rows / BM) against a mirror of project_pick_split, and it checks
the inlined consumer body through the plan's lpad (NT = lpad / 8).  Every case also checks the two paddings that must
not matter: NaN in the X padding columns [N, ld) and random values in C's padding degrees [L + 1, lpad) leave the result
bit-identical, and cf[..., L + 1:] is exactly 0 (products with the zero basis rows are exact).

On any machine, test_warp_tile_body_ledger derives the 26 (NT, TWO) bodies the default k_eddy<32, NJ, 8, TWO, 3> inlines
and requires a case for each, and test_case_table_reaches_edges checks that the table reaches the column tails, tiny
column counts, row counts and split-K chunk counts the kernels branch on, at small and at large NT."""
import collections
import json
import math
import re

import numpy as np
import pytest

from pytemdiags_b200 import synthetic as syn

TOL = 1e-12
# dedup: the reference's Q is the expanded basis rsq[u] * Qw[u] (one rounding), the kernels scale the group flux sums
# by rsq instead, and the group sums recombine p - d_a s_b - d_b s_a + n d_a d_b, whose terms are up to ~sqrt(n) times
# the result for n ~ 100 members of white noise: about 10x the dense estimate, still 1e-14, so the dense bar holds
# (measured worst on a B200: 2.7e-15 dedup, 2.3e-15 dense)
TOL_DEDUP = 1e-12
SMS_B200 = 148
KERNEL_RE = re.compile(r'temd::k_(?:eddy|project|gsum_warp|gsum_thread)<[^>]*>')
TEM_PAIRS = ((0, 1), (0, 3), (1, 2))               # u'v', u'omega', v'theta'  (fields u, v, theta, omega)
TRACER_PAIRS = ((0, 2), (0, 3), (1, 2), (1, 3))    # q1'v', q1'omega', q2'v', q2'omega'  (fields q1, q2, v, omega)

Case = collections.namedtuple('Case', 'id kind grid rows nlev L env kernel min_norm')
#   kind  'tem'    Engine.eddy_flux_project      'pair'  Engine.tracer_flux_project
#         'dedup'  DedupEngine.eddy_flux_project, Q expanded to the full grid
#   grid  ('pg2', ne, drop): ne pg2 with the last `drop` columns removed (N mod 16 = 8 - drop for odd ne, -drop for
#         even ne); ('gauss', n): one column per Gauss-Legendre latitude; ('latlon', nlat, nlon, 'lat' | 'lon'):
#         raveled lat-major (groups are contiguous column ranges) or lon-major (groups are scattered)


def _ep(bm, nj, warps, two, nprod=3):
    return 'temd::k_eddy<%d, %d, %d, %s, %d>' % (bm, nj, warps, 'true' if two else 'false', nprod)


def _wt(nt, two):
    """the default k_eddy instantiation whose warp-tile body runs at nt degree tiles"""
    return _ep(32, (nt + 1) // 2, 8, two)


def _pjp(ntb):
    return 'temd::k_project<%d, 8, true>' % ntb


def _gs(mode):
    return 'temd::k_gsum_warp<true, %d>' % mode


NCH1 = {'TEMD_EDDY_NCH': '1'}
SPLIT = {'TEMD_EDDY_MODE': 'split', 'TEMD_EDDY_SCRATCH_GB': '1e-6'}     # 128-row batches, the last one ragged


def pg2(ne, drop=0):
    return ('pg2', ne, drop)


def gauss(n):
    return ('gauss', n)


CASES = [
    # ---- warp-tile body, two chunks per round (the default): (NT, true) for NT = 1..13
    Case('wt1_two', 'tem', gauss(13), 5, 7, 7, {}, _wt(1, True), False),             # N = 13: one chunk, nloc 1
    Case('wt2_two', 'tem', pg2(3, 7), 33, 13, 12, {}, _wt(2, True), False),          # tail 1
    Case('wt3_two', 'tem', gauss(30), 31, 7, 23, {}, _wt(3, True), False),           # nloc 2
    Case('wt4_two', 'tem', pg2(4, 1), 97, 13, 29, {}, _wt(4, True), False),          # tail 15; 3 splits of 8 chunks
    Case('wt5_two', 'tem', gauss(40), 1, 7, 39, {}, _wt(5, True), False),            # nloc 3
    Case('wt6_two', 'tem', pg2(7, 7), 5, 7, 44, {}, _wt(6, True), False),            # tail 1; splits of 14 and 15
    Case('wt7_two', 'tem', pg2(8, 7), 33, 13, 55, {}, _wt(7, True), False),          # tail 9
    Case('wt8_two', 'tem', pg2(11, 1), 97, 7, 60, {}, _wt(8, True), False),          # tail 7; splits of 21 and 23
    Case('wt9_two', 'tem', pg2(13), 500, 13, 71, {}, _wt(9, True), False),           # tail 8; splits of 22 and 29
    Case('wt10_two', 'tem', pg2(12, 7), 31, 7, 76, {}, _wt(10, True), False),        # tail 9
    Case('wt11_two', 'tem', pg2(15, 7), 1, 13, 87, {}, _wt(11, True), False),        # tail 1
    Case('wt12_two', 'tem', pg2(16), 5, 7, 92, {}, _wt(12, True), False),            # tail 0
    Case('wt13_two', 'tem', pg2(17, 1), 500, 7, 103, {}, _wt(13, True), False),      # tail 7; splits of 42 and 49
    # ---- warp-tile body, one chunk per round (TEMD_EDDY_NCH=1): (NT, false) for NT = 1..13
    Case('wt1_one', 'tem', pg2(3, 1), 97, 7, 4, NCH1, _wt(1, False), False),         # tail 7
    Case('wt2_one', 'tem', gauss(40), 33, 13, 15, NCH1, _wt(2, False), False),       # nloc 3
    Case('wt3_one', 'tem', pg2(4, 7), 5, 7, 20, NCH1, _wt(3, False), False),         # tail 9
    Case('wt4_one', 'tem', pg2(4), 3000, 13, 31, NCH1, _wt(4, False), False),        # tail 0; one split of 24 chunks
    Case('wt5_one', 'tem', pg2(5), 31, 7, 36, NCH1, _wt(5, False), False),           # tail 8
    Case('wt6_one', 'tem', pg2(7, 1), 1000, 13, 47, NCH1, _wt(6, False), False),     # tail 7; splits of 17 and 19
    Case('wt7_one', 'tem', pg2(11, 7), 5, 7, 52, NCH1, _wt(7, False), False),        # tail 1
    Case('wt8_one', 'tem', pg2(11), 33, 13, 63, NCH1, _wt(8, False), False),         # tail 8
    Case('wt9_one', 'tem', pg2(13, 7), 97, 7, 68, NCH1, _wt(9, False), False),       # tail 1
    Case('wt10_one', 'tem', pg2(14, 1), 1, 7, 79, NCH1, _wt(10, False), False),      # tail 15
    Case('wt11_one', 'tem', pg2(15), 500, 13, 84, NCH1, _wt(11, False), False),      # tail 8
    Case('wt12_one', 'tem', pg2(16, 7), 33, 7, 95, NCH1, _wt(12, False), False),     # tail 9
    Case('wt13_one', 'tem', pg2(18, 1), 97, 13, 100, NCH1, _wt(13, False), False),   # tail 15
    # ---- large NT on 13 / 24 / 40 columns: rank-deficient bases (min_norm=True), the degrees beyond the rank have
    #      zero basis rows; nloc 1, 2, 3
    Case('wt13_two_n13', 'tem', gauss(13), 33, 7, 103, {}, _wt(13, True), True),
    Case('wt9_two_n24', 'tem', gauss(24), 97, 13, 71, {}, _wt(9, True), True),
    Case('wt12_one_n40', 'tem', gauss(40), 5, 13, 95, NCH1, _wt(12, False), True),
    # ---- group bodies: BM 24 / 12 warps, BM 32 / 16 warps, fused BM 16 and BM 8
    Case('bm24', 'tem', pg2(7, 7), 33, 7, 40, {'TEMD_EDDY_BM': '24'}, _ep(24, 2, 12, True), False),
    Case('w16', 'tem', pg2(13, 1), 31, 13, 72, {'TEMD_EDDY_WARPS': '16'}, _ep(32, 3, 16, True), False),
    Case('fused16', 'tem', pg2(27, 7), 33, 7, 155, {'TEMD_EDDY_MODE': 'fused'}, _ep(16, 3, 16, True), False),
    Case('fused8', 'tem', pg2(37, 1), 13, 13, 215, {'TEMD_EDDY_MODE': 'fused'}, _ep(8, 4, 8, True), False),
    # ---- tracer pair k_eddy<32, NJ, 8, false, 4>, NJ 1..7
    Case('pair1', 'pair', pg2(3, 7), 33, 1, 7, {}, _ep(32, 1, 8, False, 4), False),
    Case('pair2', 'pair', pg2(5, 1), 5, 1, 28, {}, _ep(32, 2, 8, False, 4), False),
    Case('pair3', 'pair', pg2(7, 7), 97, 1, 40, {}, _ep(32, 3, 8, False, 4), False),
    Case('pair4', 'pair', pg2(11, 1), 1, 1, 55, {}, _ep(32, 4, 8, False, 4), False),
    Case('pair5', 'pair', pg2(13, 7), 31, 1, 79, {}, _ep(32, 5, 8, False, 4), False),
    Case('pair6', 'pair', pg2(15, 1), 500, 1, 84, {}, _ep(32, 6, 8, False, 4), False),
    Case('pair7', 'pair', pg2(17, 7), 33, 1, 103, {}, _ep(32, 7, 8, False, 4), False),
    # ---- split path (synth-eddy epilogue + product-mode projection), ragged 128-row batches
    Case('split_L60', 'tem', pg2(11, 7), 200, 13, 60, SPLIT, _pjp(8), False),
    Case('split_L110', 'tem', pg2(21, 1), 300, 7, 110, {'TEMD_EDDY_SCRATCH_GB': '1e-6'}, _pjp(7), False),
    Case('split_pair_L110', 'pair', pg2(21, 7), 150, 1, 110, {'TEMD_EDDY_SCRATCH_GB': '1e-6'}, _pjp(7), False),
    # ---- dedup: group-sum loop modes 0 (scattered), 1 (contiguous, odd counts), 2 (contiguous, even counts)
    Case('dedup_mode0', 'dedup', ('latlon', 24, 100, 'lon'), 33, 7, 19, {}, _gs(0), False),
    Case('dedup_mode1', 'dedup', ('latlon', 24, 99, 'lat'), 5, 13, 20, {}, _gs(1), False),
    Case('dedup_mode2', 'dedup', ('latlon', 24, 70, 'lat'), 97, 7, 17, {}, _gs(2), False),
]


def make_lat(grid):
    if grid[0] == 'pg2':
        lat = syn.pg2_grid(grid[1])[0]
        return lat[:lat.shape[0] - grid[2]]
    if grid[0] == 'gauss':
        return np.rad2deg(np.arcsin(np.polynomial.legendre.leggauss(grid[1])[0]))
    lat = syn.latlon_grid(grid[1], grid[2])[0]
    return lat if grid[3] == 'lat' else np.ascontiguousarray(lat.reshape(grid[1], grid[2]).T).ravel()


def ncol(grid):
    if grid[0] == 'pg2':
        return 24 * grid[1] ** 2 - grid[2]
    return grid[1] if grid[0] == 'gauss' else grid[1] * grid[2]


def nt_of(L):
    return (L + 8) // 8


def eddy_shape(kernel):
    """(BM, NJ, WARPS, TWO, NP) of a k_eddy instantiation name, or None"""
    m = re.fullmatch(r'temd::k_eddy<(\d+), (\d+), (\d+), (true|false), (\d+)>', kernel)
    return m and (int(m[1]), int(m[2]), int(m[3]), m[4] == 'true', int(m[5]))


def body(case):
    """(NT, TWO) of the warp-tile body the case runs, or None for the other layouts"""
    s = eddy_shape(case.kernel)
    if s is None or s[:3] != (32, s[1], 8) or s[4] != 3:
        return None
    return nt_of(case.L), s[3]


def pick_split(tiles, nchunks, sms, max_split=64):
    """mirror of project_pick_split (csrc/temd_project.cu)"""
    best, best_cost = 1, None
    for s in range(1, min(max_split, nchunks) + 1):
        cost = -(-tiles * s // sms) * (-(-nchunks // s) + 24) + 2 * s
        if best_cost is None or cost < best_cost:
            best, best_cost = s, cost
    return best


def chunk_counts(nchunks, nsplit):
    """chunks of each split-K range, as the kernel computes nloc"""
    cps = -(-nchunks // nsplit)
    return [min(cps, nchunks - i * cps) for i in range(nsplit)]


def split_of(case, sms):
    bm = eddy_shape(case.kernel)[0]
    nch = -(-ncol(case.grid) // 16)
    s = pick_split(-(-case.rows // bm), nch, sms)
    return s, chunk_counts(nch, s)


# ------------------------------------------------------------------ ledgers (no GPU needed)

def test_warp_tile_body_ledger():
    """k_eddy<32, NJ, 8, TWO, 3> serves nt <= 13 with NJ = ceil(nt / 2) and inlines the bodies NT = 2 NJ - 1 and 2 NJ
    (capped at 13), for both loop shapes: each of these 26 bodies has a case."""
    bodies = {(b, two) for nt in range(1, 14) for b in (2 * ((nt + 1) // 2) - 1, 2 * ((nt + 1) // 2)) if b <= 13
              for two in (True, False)}
    assert len(bodies) == 26
    covered = {body(c) for c in CASES} - {None}
    assert covered <= bodies, sorted(covered - bodies)
    assert not bodies - covered, 'warp-tile bodies without a case: %s' % sorted(bodies - covered)
    for c in CASES:
        s = eddy_shape(c.kernel)
        if s is not None and s[0] == 32 and s[2] == 8:
            assert s[1] == (nt_of(c.L) + 1) // 2, (c.id, 'NJ = ceil(nt / 2) at BM 32 with 8 warps')


def test_case_ids_unique():
    ids = [c.id for c in CASES]
    assert len(ids) == len(set(ids))


def test_case_table_reaches_edges():
    """Column tails, one / two / three chunks, row counts and split-K chunk counts, each at NT <= 6 and at NT >= 7 of
    the warp-tile body (split counts at the B200's SM count: on the GPU each case checks its launch grid)."""
    small, large = collections.defaultdict(set), collections.defaultdict(set)
    for c in CASES:
        b = body(c)
        if b is None:
            continue
        n = ncol(c.grid)
        s, locs = split_of(c, SMS_B200)
        edges = {('tail', n % 16), ('rows', c.rows), ('nchunks', min(-(-n // 16), 4))}
        if b[1]:
            edges |= {('nloc', 'odd' if x % 2 else 'even', s > 1) for x in locs}
        (small if b[0] <= 6 else large)[c.id] = edges
    want = {('tail', t) for t in (0, 1, 7, 8, 9, 15)} | {('rows', r) for r in (1, 5, 31, 33, 97)} \
        | {('nchunks', k) for k in (1, 2, 3)} | {('nloc', p, True) for p in ('odd', 'even')}
    for name, side in (('NT <= 6', small), ('NT >= 7', large)):
        seen = set().union(*side.values())
        assert not want - seen, '%s never reaches %s' % (name, sorted(want - seen))
    for c in CASES:
        if c.kind != 'pair':
            assert c.nlev > 1 and math.gcd(c.nlev, 8) == 1, (c.id, 'nlev must be coprime to 8')
        assert ncol(c.grid) == make_lat(c.grid).shape[0]


# ------------------------------------------------------------------ float64 reference

def contract_ref(Q, X, C, lev_scale, nlev, pairs, scale_field):
    """[nprod][rows][lpad] from Q [N][lpad], X [4][rows][N] (padding columns removed), C [4][rows][lpad]"""
    rows = X.shape[1]
    s = np.ones((4, rows))
    if lev_scale is not None:
        s[scale_field] = lev_scale[np.arange(rows) % nlev]
    E = s[:, :, None] * X - C @ Q.T
    return np.stack([(E[a] * E[b]) @ Q for a, b in pairs])


# ------------------------------------------------------------------ GPU

def _launches(fn, tmp_path):
    """fn() under torch.profiler (CUDA activity); returns (fn(), [(kernel name, launch grid)])."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / 'trace.json'
    prof.export_chrome_trace(str(path))
    with open(path) as fh:
        events = json.load(fh)['traceEvents']
    return out, [(e['name'], e.get('args', {}).get('grid')) for e in events if e.get('cat') == 'kernel']


def _engine(case, lat):
    from pytemdiags_b200.engine import DedupEngine, Engine
    cls = DedupEngine if case.kind == 'dedup' else Engine
    return cls(lat, np.linspace(-90.0, 90.0, 7), case.L, min_norm=case.min_norm).build_basis()


def _padded(X, ld, pad):
    """[rows][N] host array -> [rows][N] device view of a [rows][ld] buffer whose padding columns hold `pad`"""
    import torch
    buf = torch.full((X.shape[0], ld), pad, dtype=torch.float64, device='cuda')
    buf[:, :X.shape[1]] = torch.as_tensor(X).cuda()
    return buf[:, :X.shape[1]]


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=[c.id for c in CASES])
def test_eddy_contract(monkeypatch, tmp_path, case):
    import torch
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    lat = make_lat(case.grid)
    N, rows, L = lat.shape[0], case.rows, case.L
    eng = _engine(case, lat)
    lpad = eng.lpad
    assert lpad == 8 * nt_of(L)
    if body(case) is not None:
        assert lpad // 8 == body(case)[0]
    Q = np.ascontiguousarray(eng.synth_native(torch.eye(lpad, dtype=torch.float64, device='cuda')).cpu().numpy().T)
    assert Q.shape == (N, lpad) and not Q[:, L + 1:].any()

    rng = np.random.default_rng(sum(map(ord, case.id)))
    X = rng.standard_normal((4, rows, N))
    C = rng.standard_normal((4, rows, lpad)) * math.sqrt(N / (L + 1))   # C Q^T about as large as X
    C[:, :, L + 1:] = 0.0
    C_pad = C.copy()
    C_pad[:, :, L + 1:] = rng.standard_normal((4, rows, lpad - L - 1))
    lev_scale = None if case.kind == 'pair' else 0.5 + rng.permutation(case.nlev) / case.nlev
    pairs = TRACER_PAIRS if case.kind == 'pair' else TEM_PAIRS
    ref = contract_ref(Q, X, C, lev_scale, case.nlev, pairs, 2)

    ld = N + (N & 1) + 6
    sc = None if lev_scale is None else torch.as_tensor(lev_scale).cuda()

    def run(pad, coef):
        xs = [_padded(x, ld, pad) for x in X]
        c4 = torch.as_tensor(coef).cuda()
        if case.kind == 'pair':
            return eng.tracer_flux_project(xs[0], xs[1], xs[2], xs[3], c4).cpu().numpy()
        return eng.eddy_flux_project(xs[0], xs[1], xs[2], xs[3], c4, sc, case.nlev).cpu().numpy()

    got, launched = _launches(lambda: run(0.0, C), tmp_path)
    names = {k for n, _ in launched for k in KERNEL_RE.findall(n)}
    assert case.kernel in names, 'expected %s to run; the profiler saw: %s' % (case.kernel, sorted(n for n, _ in launched))
    assert not {n for n in names if 'k_eddy' in n} - {case.kernel}, sorted(names)
    note = ''
    if eddy_shape(case.kernel) is not None:
        grids = [g for n, g in launched if case.kernel in n]
        assert len(grids) == 1 and grids[0] is not None, ('no launch grid in the trace', grids)
        bm = eddy_shape(case.kernel)[0]
        nsplit, locs = split_of(case, torch.cuda.get_device_properties(0).multi_processor_count)
        assert grids[0][0] == -(-rows // bm) * nsplit, (grids[0], rows, bm, nsplit)
        note = ', nsplit %d, chunks per split %s' % (nsplit, sorted(set(locs)))
    if case.kind == 'dedup':
        assert not any('k_gsum_thread' in n for n in names), sorted(names)

    assert got.shape == ref.shape
    errs = [float(np.abs(got[q] - ref[q]).max() / np.abs(ref[q]).max()) for q in range(len(pairs))]
    print('%s: worst %.2e over %d planes (N %d, rows %d, lpad %d%s)' % (case.id, max(errs), len(errs), N, rows, lpad, note))
    bar = TOL_DEDUP if case.kind == 'dedup' else TOL
    assert max(errs) <= bar, errs

    assert not got[:, :, L + 1:].any(), 'padding degrees of the flux coefficients are not 0'
    nan_pad = run(float('nan'), C)
    assert np.isfinite(nan_pad).all(), 'NaN in the X padding columns reached the result'
    assert np.array_equal(nan_pad, got), 'X padding columns changed the result'
    assert np.array_equal(run(0.0, C_pad), got), "C's padding degrees changed the result"
