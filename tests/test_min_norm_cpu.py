"""CPU: the NumPy reference of `min_norm=True` against its closed form, and the keyword plumbing of the feature."""
import os
import sys

import numpy as np
import pytest

import oracle
from pytemdiags_b200 import synthetic as syn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import min_norm_reference as R  # noqa: E402

LAT_OUT = oracle.zm_latitudes(1)


def nerr(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max())


@pytest.mark.parametrize('nlat,nlon,poles,L', [(24, 48, False, 50), (24, 48, False, 1000), (36, 72, False, 50),
                                               (18, 36, False, 300), (19, 36, True, 23), (91, 182, True, 200)])
def test_lstsq_numpy_matches_closed_form_on_latlon(nlat, nlon, poles, L):
    """On a lat-lon grid with fewer latitudes than degrees, NumPy's minimum-norm answer is the per-latitude mean on
    the native grid and the minimum-norm Legendre interpolant of those means on the output grid."""
    lat = syn.latlon_grid(nlat, nlon, poles=poles)[0]
    Y0, Y0inv, Y0p, r = R.sph_matrices_lstsq_numpy(lat, LAT_OUT, L)
    assert r == min(nlat, L + 1)
    A = np.random.default_rng(nlat + L).standard_normal((lat.shape[0], 4))
    c = Y0inv @ A
    assert nerr(Y0 @ c, R.latitude_means(lat, A)) <= 1e-13
    assert nerr(Y0p @ c, R.legendre_interpolant(lat, LAT_OUT, L, A)) <= 1e-13


@pytest.mark.parametrize('ne,L', [(2, 20), (4, 70), (5, 120)])
def test_svd_form_equals_literal_lstsq(ne, L):
    lat = syn.pg2_grid(ne)[0]
    lit = R.sph_matrices_lstsq_numpy(lat, LAT_OUT, L, method='lstsq')
    svd = R.sph_matrices_lstsq_numpy(lat, LAT_OUT, L, method='svd')
    assert lit[3] == svd[3] == R.weighted_spectrum(lat, L)[2]
    assert nerr(svd[1], lit[1]) <= 1e-9


def test_min_norm_with_weights_raises():
    from pytemdiags_b200 import sph_zonal_averager
    lat = syn.latlon_grid(24, 48)[0]
    with pytest.raises(RuntimeError, match='min_norm=True is not available together with weights='):
        sph_zonal_averager(lat, LAT_OUT, 50, weights=np.full(lat.shape[0], 1.0 / lat.shape[0]), min_norm=True)


def test_min_norm_reaches_the_engine_and_its_cache_key(monkeypatch):
    import pytemdiags_b200.zonal as zonal

    made = []

    class _Stub:
        def __init__(self, lat, lat_out, L, device=None, min_norm=False):
            self.min_norm = min_norm
            made.append(self)

    monkeypatch.setattr(zonal, 'Engine', _Stub)
    monkeypatch.setattr(zonal, 'DedupEngine', _Stub)
    monkeypatch.setattr(zonal, '_ENGINE_CACHE', {})
    lat = syn.latlon_grid(24, 48)[0]
    a = zonal._cached_engine(lat, LAT_OUT, 50, 'cuda:0')
    b = zonal._cached_engine(lat, LAT_OUT, 50, 'cuda:0', min_norm=True)
    c = zonal._cached_engine(lat, LAT_OUT, 50, 'cuda:0', dedup=True, min_norm=True)
    assert [e.min_norm for e in made] == [False, True, True] and len({id(a), id(b), id(c)}) == 3
    assert zonal._cached_engine(lat, LAT_OUT, 50, 'cuda:0', min_norm=True) is b


def test_tem_passes_min_norm_to_the_averager(monkeypatch):
    import pytemdiags_b200.tem as tem_mod

    class _Stub:
        def __init__(self, lat, lat_out, L, **kw):
            self.kw, self.rank = kw, 24

        def sph_compute_matrices(self, **kw):
            pass

        def sph_zonal_mean(self, A):
            raise NotImplementedError

    monkeypatch.setattr(tem_mod, 'sph_zonal_averager', _Stub)
    monkeypatch.setattr(tem_mod.TEMDiagnostics, '_compute_all', lambda self: None)
    lat, lon = syn.pg2_grid(2)
    plev = syn.default_plev(4)
    f = syn.synth_fields(lat, lon, plev, 2, seed=0)
    args = (f['ua'], f['va'], f['ta'], f['wap'], plev, lat)
    t = tem_mod.TEMDiagnostics(*args, dims=('time', 'lev', 'ncol'), debug_level=0, min_norm=True)
    assert t.ZM.kw['min_norm'] is True and t.rank == 24
    t = tem_mod.TEMDiagnostics(*args, dims=('time', 'lev', 'ncol'), debug_level=0)
    assert t.ZM.kw['min_norm'] is False
