"""GPU: `min_norm=True` - minimum-norm zonal means on rank-deficient bases, from the on-GPU Jacobi SVD.

The yardstick is NumPy's minimum-norm least-squares solution, np.linalg.lstsq(Y0, I, rcond=None) (tests/
min_norm_reference.py).  Parity with it is only meaningful where the rank decision has a gap and the kept part is
well-conditioned: each parity case asserts sigma_r / sigma_1 >= 1e-4 and sigma_{r+1} / sigma_1 <= cutoff / 10 first.
Where the spectrum runs down to the cutoff (ill-posed cases) any two correct implementations may differ completely,
so only invariants are checked there."""
import os
import sys

import numpy as np
import pytest

import oracle
from pytemdiags_b200 import synthetic as syn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import min_norm_reference as R  # noqa: E402

pytestmark = pytest.mark.gpu

LAT_OUT = oracle.zm_latitudes(1)


def _grid(name):
    if name == 'll72x144+row':
        return R.latlon_plus_row()[0]
    if name.startswith('ll'):                       # 'll24x48' (cell-centre rows) or 'll91x182p' (rows at both poles)
        nlat, nlon = (int(v) for v in name[2:].rstrip('p').split('x'))
        return syn.latlon_grid(nlat, nlon, poles=name.endswith('p'))[0]
    if name.startswith('ne'):                       # 'ne4' = ne4pg2
        return syn.pg2_grid(int(name[2:]))[0]
    raise ValueError(name)


# grid, L, NumPy's rank (DESIGN.md §2; the issue's table, recomputed by weighted_spectrum in every case)
PARITY = [('ll24x48', 50, 24), ('ll24x48', 1000, 24), ('ll36x72', 50, 36), ('ll18x36', 300, 18), ('ll91x182p', 200, 91),
          ('ne2', 20, 14), ('ne4', 70, 52), ('ne4', 80, 52), ('ne5', 120, 80), ('ll72x144+row', 72, 72),
          ('ll72x144+row', 100, 72)]
ILL_POSED = [('ne4', 50), ('ne4', 100), ('ne8', 140)]


def nerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / np.abs(b).max())


def _averager(lat, L, dedup, **kw):
    from pytemdiags_b200 import sph_zonal_averager
    av = sph_zonal_averager(lat, LAT_OUT, L, min_norm=True, dedup=dedup, device='cuda:0', **kw)
    av.sph_compute_matrices()
    return av


def _field(lat, rows=37, seed=0):
    """(N, rows): smooth zonal structure, zonal waves and noise; rows is not a multiple of any tile size."""
    rng = np.random.default_rng(seed)
    N = lat.shape[0]
    phi = np.deg2rad(lat)
    base = np.cos(phi)[:, None] * np.linspace(1, 3, rows)[None, :] + np.sin(3 * phi)[:, None]
    return base + 0.3 * rng.standard_normal((N, rows))


@pytest.mark.parametrize('dedup', [False, True], ids=['dense', 'dedup'])
@pytest.mark.parametrize('grid,L,rank', PARITY, ids=['%s-L%d' % (g, L) for g, L, _ in PARITY])
def test_parity_with_numpy_lstsq(grid, L, rank, dedup):
    lat = _grid(grid)
    s, cutoff, r = R.weighted_spectrum(lat, L)
    assert r == rank
    assert s[r - 1] / s[0] >= 1e-4, 'kept part ill-conditioned: sigma_r / sigma_1 = %.2g' % (s[r - 1] / s[0])
    assert r == s.shape[0] or s[r] <= cutoff / 10, 'no gap at the cutoff: sigma_r+1 / cutoff = %.2g' % (s[r] / cutoff)
    Y0, Y0inv, Y0p, r_np = R.sph_matrices_lstsq_numpy(lat, LAT_OUT, L)
    assert r_np == rank
    av = _averager(lat, L, dedup)
    assert av.rank == rank
    A = _field(lat)
    c = Y0inv @ A
    errs = {'zonal_mean': nerr(av.sph_zonal_mean(A), Y0p @ c),
            'native': nerr(av.sph_zonal_mean_native(A), Y0 @ c),
            'dlat': nerr(av.sph_zonal_mean_dlat(A), oracle.sph_basis_dlat(LAT_OUT, L) @ c),
            'Y0inv': nerr(av.Y0inv, Y0inv)}
    assert max(errs.values()) <= 1e-10, errs
    eng = av._engine
    eng.build_basis(sanity=True)
    assert eng.rank == rank
    assert abs(eng.sanity[0] - rank) <= 1e-9 * rank and abs(eng.sanity[1]) <= 1e-9 * rank, eng.sanity


def test_tall_case_default_build_refuses():
    """U = L+1 = 73 distinct nodes, numerical rank 72: the early distinct-latitude check passes, the Cholesky
    factorisation of the default build breaks down."""
    from pytemdiags_b200 import sph_zonal_averager
    av = sph_zonal_averager(_grid('ll72x144+row'), LAT_OUT, 72, device='cuda:0')
    with pytest.raises(RuntimeError, match='rank-deficient'):
        av.sph_compute_matrices()


def _basis_rows(av):
    """Rows of the whitened basis Q^T on the native columns, (lpad, N), by native synthesis of unit coefficients.
    (Q^T Q is checked directly: Y0inv Y0 formed on the host carries eps * sigma_1 / sigma_r ~ 1e-4 of rounding here.)"""
    import torch
    eng = av._engine
    eye = torch.eye(eng.lpad, dtype=torch.float64, device=eng.device)
    return eng.synth_native(eye).cpu().numpy()


@pytest.mark.parametrize('dedup', [False, True], ids=['dense', 'dedup'])
@pytest.mark.parametrize('grid,L', ILL_POSED, ids=['%s-L%d' % c for c in ILL_POSED])
def test_ill_posed_invariants(grid, L, dedup):
    lat = _grid(grid)
    s, cutoff, r_np = R.weighted_spectrum(lat, L)
    near = int(np.sum((s >= cutoff / 10) & (s <= 10 * cutoff)))
    av = _averager(lat, L, dedup)
    r = av.rank
    assert abs(r - r_np) <= near, (r, r_np, near)
    q = _basis_rows(av)
    G = q @ q.T
    I_r = np.zeros_like(G)
    I_r[np.arange(r), np.arange(r)] = 1.0
    assert np.abs(G - I_r).max() <= 1e-12, np.abs(G - I_r).max()
    A = _field(lat, rows=5)
    zn = av.sph_zonal_mean_native(A)
    assert nerr(av.sph_zonal_mean_native(zn), zn) <= 1e-12


@pytest.mark.parametrize('dedup', [False, True], ids=['dense', 'dedup'])
@pytest.mark.parametrize('grid,L', [('ll24x48', 50), ('ll18x36', 300), ('ll91x182p', 200)])
def test_latlon_known_answers(grid, L, dedup):
    """Every distinct latitude kept: the native mean is the per-latitude mean, the output mean the minimum-norm
    Legendre interpolant of those means, and a field whose Legendre coefficients lie in the row space of Y_U
    (the part of coefficient space the grid can see) is reproduced exactly on the output grid."""
    lat = _grid(grid)
    av = _averager(lat, L, dedup)
    A = _field(lat, rows=6, seed=3)
    assert nerr(av.sph_zonal_mean_native(A), R.latitude_means(lat, A)) <= 1e-12
    assert nerr(av.sph_zonal_mean(A), R.legendre_interpolant(lat, LAT_OUT, L, A)) <= 1e-10
    _, xu, _, _ = R.unique_nodes(lat)
    Yu = oracle.sph_basis_recurrence(xu, L)
    coef = Yu.T @ np.random.default_rng(5).standard_normal((xu.shape[0], 2))
    x = np.cos(np.deg2rad(90 - lat))
    F = oracle.sph_basis_recurrence(x, L) @ coef
    Fp = oracle.sph_basis_recurrence(np.cos(np.deg2rad(90 - LAT_OUT)), L) @ coef
    assert nerr(av.sph_zonal_mean(F), Fp) <= 1e-10


@pytest.mark.parametrize('dedup', [False, True], ids=['dense', 'dedup'])
def test_full_tem_and_tracers(dedup):
    from pytemdiags_b200 import TEMDiagnostics
    lat, lon = syn.latlon_grid(24, 48, poles=False)
    L, K, T = 50, 7, 3
    plev = syn.default_plev(K)
    f = syn.synth_fields(lat, lon, plev, T, seed=11, fields=('ua', 'va', 'ta', 'wap', 'q'))
    rng = np.random.default_rng(2)
    qs = [f['q'], f['q'] * 1.5 + 1e-4 * rng.standard_normal(f['q'].shape), 3e-4 * np.abs(f['va']) + 1e-5]
    Y0, Y0inv, Y0p, r = R.sph_matrices_lstsq_numpy(lat, LAT_OUT, L)
    tr = lambda x: np.ascontiguousarray(x.transpose(2, 1, 0))
    ref = oracle.tem_suite(tr(f['ua']), tr(f['va']), tr(f['ta']), tr(f['wap']), plev, lat, L=L, literal=False,
                           matrices=(Y0, Y0inv, Y0p), q=[tr(q) for q in qs])
    tem = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, q=qs, L=L, dims=('time', 'lev', 'ncol'),
                         debug_level=0, device='cuda:0', min_norm=True, dedup=dedup)
    assert tem.rank == r == 24
    errs = {n: nerr(getattr(tem, n)(), ref[n]) for n in oracle.TEM_OUTPUTS}
    for i in range(len(qs)):
        for m in ('etfy', 'etfz', 'etdiv', 'qtendetfd', 'qtendvtem', 'qtendwtem'):
            errs['%s%d' % (m, i)] = nerr(getattr(tem, m)(i), ref['%s%d' % (m, i)])
        for p_ in ('qb', 'qpvpb', 'qpwappb', 'dqb_dp'):
            errs['%s%d' % (p_, i)] = nerr(getattr(tem, p_)[i], ref['%s%d' % (p_, i)])
    assert max(errs.values()) <= 1e-10, {k: v for k, v in errs.items() if v > 1e-10}


@pytest.mark.parametrize('dedup', [False, True], ids=['dense', 'dedup'])
@pytest.mark.parametrize('L', [50, 200])
def test_full_rank_grid_matches_default_path(L, dedup):
    """ne30pg2 (cond(Y0) 1.2 at L = 50, 19 at L = 200): L = 50 runs the fused eddy kernel, L = 200 the split path."""
    from pytemdiags_b200 import TEMDiagnostics
    lat, lon = syn.pg2_grid(30)
    K, T = 5, 2
    plev = syn.default_plev(K)
    f = syn.synth_fields(lat, lon, plev, T, seed=7)
    kw = dict(L=L, dims=('time', 'lev', 'ncol'), debug_level=0, device='cuda:0', dedup=dedup)
    mn = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, min_norm=True, **kw)
    base = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, **kw)
    assert mn.rank == L + 1 and base.rank == L + 1
    errs = {n: nerr(getattr(mn, n)(), getattr(base, n)()) for n in oracle.TEM_OUTPUTS}
    A = _field(lat, rows=9)
    errs['native'] = nerr(mn.ZM.sph_zonal_mean_native(A), base.ZM.sph_zonal_mean_native(A))
    assert max(errs.values()) <= 1e-12, errs


@pytest.mark.parametrize('dedup', [False, True], ids=['dense', 'dedup'])
def test_config4_grid_at_L1000(dedup):
    """0.25-degree lat-lon grid, 1,038,240 columns, 721 distinct latitudes, L = 1000: rank 721 and the native mean is
    the per-latitude mean."""
    lat = syn.latlon_grid(721, 1440)[0]
    av = _averager(lat, 1000, dedup)
    assert av.rank == 721
    A = _field(lat, rows=3, seed=9)
    assert nerr(av.sph_zonal_mean_native(A), R.latitude_means(lat, A)) <= 1e-12
