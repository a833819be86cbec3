"""`sph_zonal_averager` — host-side mirror of reference PyTEMDiags/sph_zonal_mean.py:35-422.

Same constructor arguments, methods, attributes and error behaviour; the matrices are never read
from / written to `maps/*.nc` (the basis is regenerated on the GPU in milliseconds), so the
cache-related arguments are accepted and ignored.
"""
import os

import numpy as np
import torch

from . import arrays as ar
from .engine import DedupEngine, Engine

# Engines (plan + orthonormalised basis in HBM) are kept per (grid, output grid, L, device), the device-memory
# analogue of the reference's on-disk `maps/Y0_*.nc` cache (sph_zonal_mean.py:165-177,330-345).
_ENGINE_CACHE = {}
_ENGINE_CACHE_MAX = int(os.environ.get('TEMD_ENGINE_CACHE', '4'))   # plans kept (2.6 GB of basis each at config 3)


def _cached_engine(lat, lat_out, L, device, overwrite=False, weights=None, dedup=False, min_norm=False):
    import hashlib
    dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    wkey = None if weights is None else hashlib.sha1(np.ascontiguousarray(weights, dtype=np.float64).tobytes()).hexdigest()
    key = (hashlib.sha1(lat.tobytes()).hexdigest(), hashlib.sha1(lat_out.tobytes()).hexdigest(), int(L), str(dev), wkey,
           bool(dedup), bool(min_norm))
    if overwrite:
        _ENGINE_CACHE.pop(key, None)
    eng = _ENGINE_CACHE.get(key)
    if eng is None:
        while len(_ENGINE_CACHE) >= _ENGINE_CACHE_MAX:
            _ENGINE_CACHE.pop(next(iter(_ENGINE_CACHE)))
        eng = (DedupEngine if dedup else Engine)(lat, lat_out, L, device=dev, min_norm=min_norm)
        _ENGINE_CACHE[key] = eng
    return eng


DEFAULT_LAT_ATTRS = {'long_name': 'Latitude of Grid Cell Centers', 'standard_name': 'latitude',
                     'units': 'degrees_north', 'axis': 'Y'}   # sph_zonal_mean.py:27-28


class sph_zonal_averager:
    def __init__(self, lat, lat_out, L, weights=None, grid_name=None, grid_out_name=None,
                 ncoldim='ncol', overwrite=False, save_dest=None, debug=False, logfile=None, device=None, dedup=False,
                 min_norm=False):
        '''
        Zonal averages of fields on unstructured grids by spherical-harmonic (m=0) least squares.

        Parameters follow the reference (sph_zonal_mean.py:36-37): `lat` native latitudes [deg] (N),
        `lat_out` output latitudes [deg] (M), `L` maximum degree.  `weights` (grid-cell area weights summing
        to 1) selects the reference's deprecated quadrature inverse Y0inv = Y0^T diag(4 pi w)
        (sph_zonal_mean.py:72,180-181,383-386); unlike the reference the caller's array is not scaled in
        place.  `grid_name`, `grid_out_name`, `overwrite`,
        `save_dest` only name cache files in the reference and are ignored.  `device`: CUDA device.
        `dedup=True` (this build only) turns on the structure-exploiting fast path: columns sharing a latitude share a
        basis row (sph_zonal_mean.py:361-363), so fields are first reduced to per-latitude sums and every GEMM runs on
        the unique latitudes (721 instead of 1,038,240 columns on a 0.25-degree lat-lon grid).  Same results to rounding.
        `min_norm=True` (this build only) accepts a rank-deficient basis, e.g. L+1 above the number of distinct
        latitudes: the result is NumPy's minimum-norm least-squares solution, np.linalg.lstsq(Y0, ., rcond=None), whose
        cutoff drops singular values <= eps * max(N, L+1) * sigma_1.  On a lat-lon grid the native mean is then the
        per-latitude mean and the output mean the minimum-norm Legendre interpolant of those means.  `rank` is the
        number of directions kept (L+1 on a full-rank grid).  Not available together with `weights`.
        '''
        self.L = L
        self.lat = lat.values if ar.is_dataarray(lat) else lat
        self.lat_out = lat_out.values if ar.is_dataarray(lat_out) else lat_out
        self.lat = np.asarray(self.lat.cpu() if isinstance(self.lat, torch.Tensor) else self.lat, dtype=np.float64)
        self.lat_out = np.asarray(self.lat_out.cpu() if isinstance(self.lat_out, torch.Tensor) else self.lat_out,
                                  dtype=np.float64)
        self.weights = weights
        self.grid_name = grid_name
        self.grid_out_name = grid_out_name
        self.save_dest = save_dest
        self.ncoldim = ncoldim
        self.debug = debug
        self.logfile = logfile
        if weights is not None:
            self.weights = np.asarray(weights.values if ar.is_dataarray(weights) else weights, dtype=np.float64)
            if len(self.weights) != len(self.lat):
                raise RuntimeError('number of weights must equal number of native grid latitudes!')
        self.N = len(self.lat)
        self.M = len(self.lat_out)
        self.l = np.arange(self.L + 1)
        # file names the reference would use (sph_zonal_mean.py:165-174); never touched here
        gname = self.grid_name if self.grid_name is not None else 'ncol{}'.format(self.N)
        goname = self.grid_out_name
        if goname is None:
            goname = '{}deg'.format(np.diff(self.lat_out)[0]) if self.M > 1 else 'point'
        self.grid_name, self.grid_out_name = gname, goname
        self.Y0_file_out = None
        self.Y0p_file_out = None
        if min_norm and weights is not None:
            raise RuntimeError('min_norm=True is not available together with weights=')
        if not torch.cuda.is_available():
            raise RuntimeError('pytemdiags_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        if dedup and weights is not None:
            raise RuntimeError('dedup=True is not available together with weights=')
        self.dedup = bool(dedup)
        self.min_norm = bool(min_norm)
        self._engine = _cached_engine(self.lat, self.lat_out, self.L, device, overwrite=overwrite, weights=self.weights,
                                      dedup=self.dedup, min_norm=self.min_norm)
        self._mats = None

    # ------------------------------------------------------------------
    def sph_compute_matrices(self, overwrite=False, read_only=False, no_write=False):
        '''Builds the basis on the GPU (sph_zonal_mean.py:302-422).  `read_only=True` means "load
        from the cache only" in the reference; there is no cache, so it returns without computing.'''
        if read_only:
            return
        if self._engine.built and not overwrite:
            return                                   # "read from the cache" (sph_zonal_mean.py:330-345)
        self._engine.build_basis(sanity=bool(self.debug) and self.weights is None, weights=self.weights)
        self._mats = None
        if self.debug and self.weights is None:
            print('(sph_zonal_mean debug) Sanity check: sum(diag(Q^T Q)) = {} (should be {}); '
                  'sum(offdiag) = {} (should be zero)'.format(self._engine.sanity[0], self._engine.rank,
                                                              self._engine.sanity[1]))

    @property
    def rank(self):
        '''Number of basis directions the zonal mean uses: L+1, or the numerical rank of Y0 with min_norm=True
        (None before sph_compute_matrices).'''
        return self._engine.rank if self._engine.built else None

    def _export(self):
        if not self._engine.built:
            return None
        if self._mats is None:
            self._mats = tuple(t.cpu().numpy() for t in self._engine.export_matrices())
        return self._mats

    @property
    def Y0(self):
        m = self._export()
        return None if m is None else m[0]

    @property
    def Y0inv(self):
        m = self._export()
        return None if m is None else m[1]

    @property
    def Y0p(self):
        m = self._export()
        return None if m is None else m[2]

    # ------------------------------------------------------------------
    def _sph_zonal_mean_generic(self, A, native, ncol_last=False, dlat=False):
        eng = self._engine
        if not eng.built:
            raise RuntimeError('Matrices Y0, Y0inv, and/or Y0p are undefined; either verify grid_name,'
                               'grid_name_out, and save_dest, or call sph_compute_matrices()'
                               'before sph_zonal_mean() or sph_zonal_mean_native()!')
        kind = ar.kind_of(A)
        name = getattr(A, 'name', None) if kind == 'dataarray' else None
        if name is None:
            name = '{unnamed variable}'
        r = ar.raw(A)
        dtype = ar.dtype_of(A)
        shape = tuple(r.shape)
        if kind == 'dataarray':
            dims = tuple(A.dims)
            if dims[0] != self.ncoldim or shape[0] != self.N:
                raise RuntimeError('(sph_zonal_mean_generic() Expected the first (leftmost) '
                                   'dimension of variable {} to be {} of length {}'.format(name, self.ncoldim, self.N))
        elif (shape[-1] if ncol_last else shape[0]) != self.N:
            raise RuntimeError('(sph_zonal_mean_generic() Expected the {} dimension of variable {} to be of '
                               'length {}'.format('last' if ncol_last else 'first (leftmost)', name, self.N))
        in_dev = r.device if isinstance(r, torch.Tensor) else None
        x = ar.to_device_f64(r, eng.device)
        if ncol_last and kind != 'dataarray':
            x2 = x.reshape(-1, self.N)
            rest = shape[:-1]
        else:
            x2 = x.reshape(self.N, -1).t()       # (DD, N) view of the reference's (N, DD)
            rest = shape[1:]
        if not (x2.stride(1) == 1 and x2.stride(0) >= self.N and x2.stride(0) % 2 == 0 and x2.data_ptr() % 16 == 0):
            ld = self.N + (self.N & 1)
            buf = torch.zeros((x2.shape[0], ld), dtype=torch.float64, device=eng.device)
            buf[:, :self.N] = x2
            x2 = buf[:, :self.N]
        with eng.lock:
            coef = eng.project([x2])
            eng.check_finite(coef, name, lambda: eng.scan_nonfinite(x2))
            if native:
                res = eng.synth_native(coef[0])                # (DD, N)
            elif dlat:
                res = eng.synth_out_dlat(coef)[0]              # (DD, M)
            else:
                res = eng.synth_out(coef)[0]                   # (DD, M)
        NN = res.shape[1]
        if ncol_last and kind != 'dataarray':
            res = res.reshape(tuple(rest) + (NN,))
        else:
            res = res.t().reshape((NN,) + tuple(rest))
        out = ar.from_device(res.contiguous(), 'numpy' if kind == 'dataarray' else kind, dtype, in_dev)
        if kind != 'dataarray':
            return out
        attrs = dict(getattr(A, 'attrs', {}) or {})
        if native:
            coords = {d: ar.coord_values(A, d) for d in dims if ar.coord_values(A, d) is not None}
            odims = dims
        else:
            # sph_zonal_mean.py:267-273: ncol -> lat, coordinate lat_out, latitude attrs
            odims = ('lat',) + dims[1:]
            coords = {d: ar.coord_values(A, d) for d in dims[1:] if ar.coord_values(A, d) is not None}
            coords['lat'] = self.lat_out
            attrs = dict(DEFAULT_LAT_ATTRS)
        attrs['long_name'] = ('latitude derivative (per radian) of the zonal mean of {}' if dlat else 'zonal mean of {}').format(name)
        return ar.make_dataarray(A, out, odims, coords=coords, name=name, attrs=attrs)

    def sph_zonal_mean_native(self, A, ncol_last=False):
        '''Zonal mean evaluated at every native column (sph_zonal_mean.py:285-290).'''
        return self._sph_zonal_mean_generic(A, True, ncol_last)

    def sph_zonal_mean(self, A, ncol_last=False):
        '''Zonal mean on the output latitudes (sph_zonal_mean.py:291-296).'''
        return self._sph_zonal_mean_generic(A, False, ncol_last)

    def sph_zonal_mean_dlat(self, A, ncol_last=False):
        '''Extra of this build (BASELINE.json north_star, "latitude derivatives in Legendre space"): d/dphi, per radian,
        of `sph_zonal_mean(A)` on the output latitudes, obtained by differentiating the Legendre basis instead of
        finite-differencing the result.  The reference has no counterpart (its lat_gradient is np.gradient,
        tem_util.py:154) and nothing on the default TEM path uses it.'''
        return self._sph_zonal_mean_generic(A, False, ncol_last, dlat=True)

    @property
    def dY0p(self):
        '''(M, L+1) latitude derivative of the basis at the output latitudes.'''
        return self._engine.export_dY0p().cpu().numpy() if self._engine.built else None
