"""GPU: parity at BASELINE.json's full grid sizes (SURVEY.md §8d).

Config 1 is checked on the whole array against the oracle run on the spot.  For configs 2-4 one time
step (time steps are independent) and for the config-5 L sweep the expected outputs were computed by the
CPU oracle in the build container (tests/golden/make_scale_golden.py, factored form: the reference's
literal N x N operator needs 1-20 TB there); inputs are regenerated bit-identically from the seed.
Size-independent properties (projector idempotence, linearity) are checked as well."""
import os

import numpy as np
import pytest

import oracle
from pytemdiags_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
TOL = 1e-10
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def nerr(x, ref):
    return float(np.abs(np.asarray(x) - ref).max() / max(np.abs(ref).max(), 1e-300))


def test_config1_full():
    """E3SM ne30pg2 (21,600 cols) x 72 levels x 24 steps, L=50: the whole array, every output."""
    from pytemdiags_b200 import TEMDiagnostics
    lat, lon = syn.pg2_grid(30)
    K, T, L = 72, 24, 50
    plev = syn.default_plev(K)
    f = syn.synth_fields(lat, lon, plev, T, seed=1)
    tem = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, L=L, dims=('time', 'lev', 'ncol'), debug_level=0)
    mats = oracle.sph_matrices(lat, oracle.zm_latitudes(1), L, method='pinv')
    tr = lambda x: np.ascontiguousarray(x.transpose(2, 1, 0))
    ref = oracle.tem_suite(tr(f['ua']), tr(f['va']), tr(f['ta']), tr(f['wap']), plev, lat, L=L, literal=False, matrices=mats)
    bad = {}
    for n in oracle.TEM_OUTPUTS + oracle.TEM_INTERMEDIATES:
        got = getattr(tem, n)
        e = nerr(got() if callable(got) else got, ref[n])
        if not e < TOL:
            bad[n] = e
    assert not bad, bad


@pytest.mark.parametrize('name', ['scale_config2_t1', 'scale_config3_t1', 'scale_config4_t1'])
def test_big_config_one_step(name):
    """configs 2 (ne120pg2, L=100: fused k_eddy BM=32), 3 (ne256pg2 x 128 lev, L=200) and 4 (721x1440 lat-lon, L=300)
    at full column count, one time step of the record.  Configs 3 and 4 have L + 1 > 104 and take the split eddy path
    (k_synth eddy epilogue + product-mode k_project); the fused BM = 16 / 8 kernels are covered by
    tests/test_gpu_instantiations.py."""
    from pytemdiags_b200 import TEMDiagnostics
    path = os.path.join(GOLD, name + '.npz')
    if not os.path.exists(path):
        pytest.skip('fixture %s not generated' % name)
    g = np.load(path)
    grid = tuple(g['grid'].tolist())
    grid = (grid[0],) + tuple(int(x) for x in grid[1:])
    K, L, seed, t0 = int(g['K']), int(g['L']), int(g['seed']), int(g['t0'])
    lat, lon = syn.make_grid(grid)
    plev = syn.default_plev(K)
    f = syn.synth_fields(lat, lon, plev, 1, seed=seed, t0=t0)
    tem = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, L=L, dims=('time', 'lev', 'ncol'), debug_level=0)
    bad = {}
    for n in oracle.TEM_OUTPUTS + ('ub', 'vb', 'thetab', 'wapb', 'upvpb', 'upwappb', 'vptpb'):
        got = getattr(tem, n)
        e = nerr(got() if callable(got) else got, g[n])
        if not e < TOL:
            bad[n] = e
    assert not bad, bad


@pytest.mark.parametrize('L', [25, 50, 100, 200, 400, 800])
def test_config5_zonal_mean_sweep(L):
    """zonal-mean-only sweep on ne120pg2 x 72 levels: sph_zonal_mean and sph_zonal_mean_native."""
    from pytemdiags_b200 import sph_zonal_averager
    path = os.path.join(GOLD, 'scale_config5_sweep.npz')
    if not os.path.exists(path):
        pytest.skip('fixture not generated')
    g = np.load(path)
    lat, lon = syn.pg2_grid(120)
    lat_out = oracle.zm_latitudes(1)
    f = syn.synth_fields(lat, lon, syn.default_plev(72), 1, seed=4, fields=('ua',))['ua'][0]    # [K][N]
    ZM = sph_zonal_averager(lat, lat_out, L)
    ZM.sph_compute_matrices()
    zm = ZM.sph_zonal_mean(f, ncol_last=True)             # [K][M]
    zn = ZM.sph_zonal_mean_native(f, ncol_last=True)      # [K][N]
    assert nerr(zm, g['zm_L%d' % L]) < TOL
    assert nerr(zn[:, :512], g['zn_L%d' % L]) < TOL
    # size-independent properties: idempotence of the projector and linearity
    assert nerr(ZM.sph_zonal_mean_native(zn, ncol_last=True), zn) < 1e-11
    h = np.roll(f, 7, axis=1) * 0.37
    assert nerr(ZM.sph_zonal_mean(f + h, ncol_last=True), zm + ZM.sph_zonal_mean(h, ncol_last=True)) < 1e-11


def test_config4_y0inv_against_svd_pinv():
    """config 4 (1,038,240 columns, L=300, cond(Y0) ~ 19): 64 sampled columns of the exported Y0inv against
    numpy's SVD pseudo-inverse of the full Y0.  The one-step fixtures above were computed with the normal-equations
    inverse, i.e. the same algebra as the GPU's whitened basis; this check decouples the expectation from it
    (measured agreement ~1e-13, as bounded by cond(Y0)^2 eps)."""
    from pytemdiags_b200 import sph_zonal_averager
    lat, lon = syn.latlon_grid(721, 1440)
    L = 300
    lat1 = np.linspace(-90, 90, 721)
    Y0 = np.repeat(oracle.sph_basis(lat1, L), 1440, axis=0)             # rows depend on latitude only
    assert np.array_equal(np.repeat(lat1, 1440), lat)
    Y0inv_ref = np.linalg.pinv(Y0)                                      # SVD (gesdd), default rcond
    ZM = sph_zonal_averager(lat, oracle.zm_latitudes(1), L)
    ZM.sph_compute_matrices()
    cols = np.random.default_rng(0).choice(lat.shape[0], 64, replace=False)
    got = ZM.Y0inv[:, cols]
    assert nerr(got, Y0inv_ref[:, cols]) < TOL, nerr(got, Y0inv_ref[:, cols])
    ZD = sph_zonal_averager(lat, oracle.zm_latitudes(1), L, dedup=True)
    ZD.sph_compute_matrices()
    assert nerr(ZD.Y0inv[:, cols], Y0inv_ref[:, cols]) < TOL
