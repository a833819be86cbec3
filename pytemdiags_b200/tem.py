"""`TEMDiagnostics` — host-side mirror of reference PyTEMDiags/tem_diagnostics.py:31-797.

Same constructor (both call shapes, SURVEY.md §8b), the same public methods, properties and error
behaviour.  The heavy lifting (zonal means, eddy fluxes, stencils) happens once in the constructor,
as in the reference (`__init__` :239-259), but on the GPU through libtemd; the methods return the
cached results of the fused epilogue instead of recomputing them.
"""
import warnings

import numpy as np
import torch

from . import arrays as ar
from . import constants as const
from .constants import P0
from .zonal import sph_zonal_averager

DEFAULT_DIMS = {'horz': 'ncol', 'vert': 'plev', 'time': 'time'}   # tem_diagnostics.py:25

_ARG_ORDER = ('lat_native', 'q', 'p0', 'zm_dlat', 'L', 'dim_names', 'grid_name', 'zm_grid_name',
              'map_save_dest', 'overwrite_map', 'zm_pole_points', 'debug_level', 'logfile')
_DEFAULTS = dict(lat_native=None, q=None, p0=P0, zm_dlat=1, L=50, dim_names=DEFAULT_DIMS, grid_name=None,
                 zm_grid_name=None, map_save_dest=None, overwrite_map=False, zm_pole_points=False,
                 debug_level=1, logfile=None)
_ZM_NAMES = ('ub', 'vb', 'thetab', 'wapb', 'upvpb', 'upwappb', 'vptpb')
_METHODS = ('vtem', 'omegatem', 'wtem', 'psitem', 'epfy', 'epfz', 'epdiv', 'utendepfd', 'utendvtem', 'utendwtem')
_DERIVED = ('dub_dp', 'dthetab_dp', 'ubcoslat', 'dubcoslat_dlat', 'psi', 'psicoslat', 'dpsicoslat_dlat',
            'dpsi_dp', 'int_vbdp')


# pinned host staging buffers for pageable inputs: (device, slot) -> [pinned uint8 tensor, last-DMA event]
_HOST_STAGING = {}


def release_host_staging():
    """Free the page-locked staging buffers kept for pageable host inputs (they are re-created on demand)."""
    for ent in _HOST_STAGING.values():
        if ent[1] is not None:
            ent[1].synchronize()
    _HOST_STAGING.clear()


def _slab_schedule(T, ts):
    """[(t0, t1)] covering [0, T) in slabs of `ts` time steps whose LAST slab is halved down to single steps
    (streaming from host memory is copy-bound: the work left after the final copy should be one step, not a slab)."""
    slabs = [(t0, min(T, t0 + ts)) for t0 in range(0, T, ts)]
    if len(slabs) > 1:
        t0, t1 = slabs.pop()
        while t1 - t0 > 1:
            mid = t0 + (t1 - t0 + 1) // 2
            slabs.append((t0, mid))
            t0 = mid
        slabs.append((t0, t1))
    return slabs


def _is_1d_of_len(x, n):
    try:
        r = ar.raw(x)
        return r.ndim == 1 and r.shape[0] == n
    except Exception:
        return False


class TEMDiagnostics:
    def __init__(self, ua, va, ta, wap, *args, **kwargs):
        '''
        TEM diagnostics on a pressure vertical coordinate (Gerber & Manzini 2016, Table A1).

        Call shapes (both accepted):
          TEMDiagnostics(ua, va, ta, wap, lat_native, q=None, p0=P0, zm_dlat=1, L=50, dim_names=...,
                         grid_name=None, zm_grid_name=None, map_save_dest=None, overwrite_map=False,
                         zm_pole_points=False, debug_level=1, logfile=None)   # tem_diagnostics.py:32-36
          TEMDiagnostics(ua, va, ta, wap, p, lat, ...)                        # README.md:40

        ua, va, ta, wap : DataArray-like (dims in any order, vertical coordinate = pressure in hPa),
            or numpy arrays / torch tensors together with `dims=` (default: the reference's internal
            order ('ncol', 'plev', 'time')) and `p=`.
        p : 1-D pressure levels (hPa unless p_units='Pa') or a gridpoint pressure field in Pa that is
            constant on each level (pressure-level data).  Mandatory for raw arrays.
        Extra keywords of this build: dims, p, p_units, time, device, slab_bytes, dedup (structure-exploiting fast
        path for grids with repeated latitudes, see sph_zonal_averager; default False), min_norm (minimum-norm
        least squares on a rank-deficient basis, see sph_zonal_averager; default False; `rank` then tells how many
        directions were kept).
        '''
        opts = dict(_DEFAULTS)
        extra = {k: kwargs.pop(k) for k in ('dims', 'p', 'p_units', 'time', 'device', 'slab_bytes', 'lat', 'dedup',
                                            'min_norm') if k in kwargs}
        pos = list(args)
        ncol_guess = None
        # README shape: (p, lat, ...) -- the 6th positional is a 1-D latitude vector
        if len(pos) >= 2 and not isinstance(pos[1], (list, tuple)) and pos[1] is not None \
                and hasattr(ar.raw(pos[1]), 'ndim') and ar.raw(pos[1]).ndim == 1 and ar.raw(pos[0]).ndim >= 1 \
                and 'lat' not in extra and 'lat_native' not in kwargs:
            ncol_guess = ar.raw(pos[1]).shape[0]
            if not _is_1d_of_len(pos[0], ncol_guess) or ar.raw(pos[0]).ndim > 1:
                extra['p'] = pos.pop(0)
        elif 'lat' in extra and len(pos) >= 1 and 'lat_native' not in kwargs:
            extra['p'] = pos.pop(0)
        if len(pos) > len(_ARG_ORDER):
            raise TypeError('too many positional arguments')
        for name, val in zip(_ARG_ORDER, pos):
            opts[name] = val
        for k_, v_ in kwargs.items():
            if k_ not in opts:
                raise TypeError("__init__() got an unexpected keyword argument '{}'".format(k_))
            opts[k_] = v_
        if 'lat' in extra:
            opts['lat_native'] = extra['lat']
        if opts['lat_native'] is None:
            raise TypeError("missing required argument 'lat_native' (latitudes of the native columns)")

        # ---- get input args (tem_diagnostics.py:217-236)
        self.ua, self.va, self.ta, self.wap = ua, va, ta, wap
        self.p0 = opts['p0']
        self.q = opts['q']
        self.ntrac = None
        self.lat_native = opts['lat_native']
        self.L = opts['L']
        self.zm_dlat = opts['zm_dlat']
        self.dim_names = opts['dim_names']
        self.zm_pole_points = opts['zm_pole_points']
        self.grid_name = opts['grid_name']
        self.zm_grid_name = opts['zm_grid_name']
        self.map_save_dest = opts['map_save_dest']
        self.overwrite_map = opts['overwrite_map']
        self.debug_level = opts['debug_level']
        self.logfile = opts['logfile']
        self._dims_in = extra.get('dims')
        self._p_in = extra.get('p')
        self._p_units = extra.get('p_units')
        self._time_in = extra.get('time')
        self._device = extra.get('device')
        self._slab_bytes = extra.get('slab_bytes')
        self._dedup = bool(extra.get('dedup', False))
        self._min_norm = bool(extra.get('min_norm', False))

        self._config_dims()

        # ---- zonal averaging object (tem_diagnostics.py:243-249)
        self.ZM = sph_zonal_averager(self._lat_native_np, self._lat_zm, self.L, grid_name=self.grid_name,
                                     grid_out_name=self.zm_grid_name, save_dest=self.map_save_dest,
                                     debug=self.debug_level > 1, overwrite=self.overwrite_map,
                                     ncoldim=self.ncolname, device=self._device, dedup=self._dedup,
                                     min_norm=self._min_norm)
        self.ZM.sph_compute_matrices(overwrite=self.overwrite_map)
        self._zonal_mean = self.ZM.sph_zonal_mean

        self._compute_all()
        self._out_file = None

    @property
    def rank(self):
        '''Number of basis directions of the zonal averager: L+1, or the numerical rank of Y0 with min_norm=True.'''
        return self.ZM.rank

    # ------------------------------------------------------------------
    def _log(self, s):
        if self.debug_level > 0:
            if self.logfile is not None:
                with open(self.logfile, 'a') as f:
                    f.write('(PyTEMDiags debug) {}\n'.format(s))
            else:
                print('(PyTEMDiags debug) {}'.format(s))

    def _config_dims(self):
        '''Input validation and layout bookkeeping (tem_diagnostics.py:266-405).'''
        self.ncolname = self.dim_names['horz']
        self.plevname = self.dim_names['vert']
        self.timename = self.dim_names.get('time', DEFAULT_DIMS['time'])
        self.data_dims = (self.ncolname, self.plevname, self.timename)

        # ---- tracers: a single array or a list of arrays (tem_diagnostics.py:282-301)
        if self.q is not None:
            if not isinstance(self.q, (list, tuple)):
                self.q = [self.q]
            else:
                self.q = list(self.q)
            for qi in self.q:
                if ar.kind_of(qi) != ar.kind_of(self.ua):
                    raise RuntimeError('tracers q must be passed as an xarray DataArray, or'
                                       'a list of xarray DataArrays')
            self.ntrac = len(self.q)
        else:
            self.ntrac = 0
        self._q_out_file = [None] * self.ntrac

        lat = self.lat_native
        lat_np = ar.raw(lat)
        lat_np = np.asarray(lat_np.cpu() if isinstance(lat_np, torch.Tensor) else lat_np, dtype=np.float64).ravel()
        self._lat_native_np = lat_np
        ncol = lat_np.shape[0]

        allvars = {'ua': self.ua, 'va': self.va, 'ta': self.ta, 'wap': self.wap}
        for i in range(self.ntrac):
            allvars['q{}'.format(i)] = self.q[i]
        self._vars = allvars
        self._kind = ar.kind_of(self.ua)
        self._in_dims = {}
        for var, dat in allvars.items():
            if ar.kind_of(dat) != self._kind:
                raise RuntimeError('Input data for arg \'{}\' must be of the same kind as ua ({})'.format(var, self._kind))
            r = ar.raw(dat)
            if self._kind == 'dataarray':
                dims = tuple(dat.dims)
            else:
                dims = self._dims_in
                if dims is None:
                    dims = self.data_dims[:r.ndim]
                dims = tuple({'horz': self.ncolname, 'vert': self.plevname, 'time': self.timename,
                              'lev': self.plevname}.get(d, d) for d in dims)
                if len(dims) != r.ndim:
                    raise RuntimeError('dims={} does not match the {} dimensions of {}'.format(dims, r.ndim, var))
            if self.ncolname not in dims:
                raise RuntimeError('Input data {} does not contain dim {}'.format(var, self.ncolname))
            if r.shape[dims.index(self.ncolname)] != ncol:
                raise RuntimeError('Dimension {} in variable {} is length {}, but input parameter lat is length {}; '
                                   'these must match!'.format(self.ncolname, var, r.shape[dims.index(self.ncolname)], ncol))
            if len(dims) < 2 or len(dims) > 3:
                raise RuntimeError('Input data has {0} dims, expected either 2 ({1}, {2}) or 3 ({1}, {2}, {3})'.format(
                    len(dims), self.ncolname, self.plevname, self.timename))
            if self.plevname not in dims:
                raise RuntimeError('Input data {} does not contain dim {}'.format(var, self.plevname))
            for d in dims:
                if d not in self.data_dims:
                    raise RuntimeError('Input data {} has unexpected dim {}'.format(var, d))
            self._in_dims[var] = dims
        shp = {v: {d: ar.raw(allvars[v]).shape[i] for i, d in enumerate(self._in_dims[v])} for v in allvars}
        for v in allvars:
            if shp[v] != shp['ua'] and {d: n for d, n in shp[v].items()} != {d: n for d, n in shp['ua'].items()}:
                raise RuntimeError('Input variables ua and {} have different shapes'.format(v))
        self.NCOL = ncol
        self.NLEV = shp['ua'][self.plevname]
        self.NT = shp['ua'].get(self.timename, 1)
        self._log('DATA DIMENSIONS: {} x {} x {} = {} x {} x {}'.format(self.ncolname, self.plevname, self.timename,
                                                                         self.NCOL, self.NLEV, self.NT))

        # ---- vertical coordinate (hPa) and time coordinate
        plev = None
        if self._p_in is not None:
            pr = ar.raw(self._p_in)
            pr = np.asarray(pr.cpu() if isinstance(pr, torch.Tensor) else pr, dtype=np.float64)
            units = self._p_units
            if pr.ndim == 1:
                if pr.shape[0] != self.NLEV:
                    raise RuntimeError('p has length {} but the vertical dimension has length {}'.format(pr.shape[0], self.NLEV))
                plev = pr / 100.0 if units == 'Pa' else pr
            else:
                pdims = tuple(self._p_in.dims) if ar.is_dataarray(self._p_in) else self._in_dims['ua']
                if pr.ndim != len(pdims):
                    raise RuntimeError('gridpoint pressure p must have the same dims as ua')
                ax = pdims.index(self.plevname)
                prm = np.moveaxis(pr, ax, 0).reshape(pr.shape[ax], -1)
                if not np.allclose(prm, prm[:, :1], rtol=1e-12, atol=0):
                    raise RuntimeError('gridpoint pressure p varies on a level: TEMDiagnostics needs data on a '
                                       'pressure vertical coordinate (tem_diagnostics.py:37-40)')
                plev = prm[:, 0] if units == 'hPa' else prm[:, 0] / 100.0
        elif self._kind == 'dataarray':
            plev = ar.coord_values(self.ua, self.plevname)
            if plev is not None:
                plev = np.asarray(plev, dtype=np.float64)
        if plev is None:
            raise RuntimeError('pressure levels are required: pass p= (1-D, hPa) or DataArrays with a {} '
                               'coordinate'.format(self.plevname))
        time = None
        if self._time_in is not None:
            time = np.asarray(self._time_in)
        elif self._kind == 'dataarray' and self.timename in self._in_dims['ua']:
            time = ar.coord_values(self.ua, self.timename)
        if time is None:
            time = np.arange(self.NT)
        self.time = time

        # ---- pressure must increase to the right (tem_diagnostics.py:372-382)
        self._flip_lev = bool(plev[0] > plev[-1])
        self._plev_input_order = plev
        if self._flip_lev:
            plev = plev[::-1].copy()
            self._log('Reversed direction of vertical dimension for all data')
        self.plev = plev
        self.p = self.plev * 100                                   # :385

        # ---- zonal-mean latitudes (:388-396)
        tol = 1e-6
        assert float(180 / self.zm_dlat).is_integer(), '180 must be divisible by dlat_out'
        self._lat_zm = np.arange(-90, 90 + self.zm_dlat, self.zm_dlat)
        if self._lat_zm[-1] > 90 + tol:
            self._lat_zm = self._lat_zm[:-1]
        if not self.zm_pole_points:
            self._lat_zm = (self._lat_zm[1:] + self._lat_zm[:-1]) / 2
        self.ZM_N = len(self._lat_zm)
        # ---- latitude-based quantities (:401-405)
        self._f_zm = 2 * const.Om * np.sin(self._lat_zm * np.pi / 180)
        self._coslat_zm = np.cos(self._lat_zm * np.pi / 180)
        self.lat, self.coslat = self._lat_zm, self._coslat_zm
        self.f = self._f_zm[:, np.newaxis, np.newaxis]

    # ------------------------------------------------------------------
    def _slab(self, var, t0, t1, device):
        '''Time steps [t0, t1) of one input as a float64 device tensor [(t1-t0)*K][N] (lev in input order).
        Host arrays are copied with non_blocking=True (a true async DMA when the array is pinned).'''
        dat = self._vars[var]
        r = ar.raw(dat)
        dims = self._in_dims[var]
        if self.timename in dims:
            sl = [slice(None)] * r.ndim
            sl[dims.index(self.timename)] = slice(t0, t1)
            r = r[tuple(sl)]
        else:
            r = r[..., None] if isinstance(r, np.ndarray) else r.unsqueeze(-1)
            dims = dims + (self.timename,)
        perm = [dims.index(self.timename), dims.index(self.plevname), dims.index(self.ncolname)]
        if isinstance(r, np.ndarray) and not r.flags.c_contiguous and not r.flags.f_contiguous:
            r = np.ascontiguousarray(r)     # strided host slice (time is not the leading dim): pack on the host
        x = ar.to_device_f64(r, device, non_blocking=True)
        if perm != [0, 1, 2]:
            x = x.permute(*perm)            # layout change happens on the device
        N = self.NCOL
        x = x.reshape(-1, N) if x.is_contiguous() else x.contiguous().reshape(-1, N)
        if N % 2 or x.data_ptr() % 16:
            buf = torch.zeros((x.shape[0], N + (N & 1)), dtype=torch.float64, device=device)
            buf[:, :N] = x
            x = buf[:, :N]
        return x

    def _is_native_device_layout(self, var, device):
        '''True if the input is a float64 CUDA tensor on `device`, C-contiguous in (time, lev, ncol) order with an even,
        16-byte aligned row pitch: the kernels can then read it in place.'''
        r = ar.raw(self._vars[var])
        dims = self._in_dims[var]
        return (isinstance(r, torch.Tensor) and r.is_cuda and r.device == device and r.dtype == torch.float64
                and dims == (self.timename, self.plevname, self.ncolname) and r.is_contiguous()
                and self.NCOL % 2 == 0 and r.data_ptr() % 16 == 0)

    def _fill(self, dst, var, t0, t1, device, slot=None):
        '''Copy time steps [t0, t1) of one input into the staging buffer dst [(t1-t0)*K][ld] (float64, (time, lev,
        ncol) order).  Host arrays in that order go straight into place with one asynchronous copy (a true DMA when
        pinned); other layouts / dtypes / devices are uploaded as they are and permuted on the device.'''
        r = getattr(self, '_whole', {}).get(var)
        if r is None:
            r = ar.raw(self._vars[var])
        dims = self._in_dims[var]
        if self.timename in dims:
            sl = [slice(None)] * r.ndim
            sl[dims.index(self.timename)] = slice(t0, t1)
            r = r[tuple(sl)]
        else:
            r = r[..., None] if isinstance(r, np.ndarray) else r.unsqueeze(-1)
            dims = dims + (self.timename,)
        perm = [dims.index(self.timename), dims.index(self.plevname), dims.index(self.ncolname)]
        K, N = self.NLEV, self.NCOL
        view = dst[:(t1 - t0) * K].view(t1 - t0, K, dst.shape[1])[:, :, :N]
        if isinstance(r, np.ndarray):
            if r.dtype.byteorder not in ('=', '|') or not r.flags.writeable:
                r = np.array(r, dtype=r.dtype.newbyteorder('='))
            if not (r.flags.c_contiguous or r.flags.f_contiguous):
                r = np.ascontiguousarray(r)     # strided host slice (time is not the leading dim): pack on the host
            r = torch.from_numpy(r)
        if perm == [0, 1, 2] and not r.is_cuda and r.is_contiguous():
            if not r.is_pinned() and r.numel() * r.element_size() >= (8 << 20):
                r = self._stage_pinned(r, slot)
            view.copy_(r, non_blocking=True)
        else:
            view.copy_(r.to(device, non_blocking=True).permute(*perm))

    def _upload_whole(self, names, device):
        '''Host arrays whose time axis is not the leading one cannot be cut into contiguous time slabs.  If the whole
        record fits comfortably in HBM it is uploaded once in its own layout (flat copies, pinned staging for pageable
        memory) and the slabs are permuted on the device; otherwise _fill packs each slab on the host.'''
        self._whole = {}
        todo = []
        for v in names:
            r = ar.raw(self._vars[v])
            dims = self._in_dims[v]
            host = isinstance(r, np.ndarray) or not r.is_cuda
            if host and self.timename in dims and dims[0] != self.timename:
                todo.append(v)
        if not todo:
            return
        total = sum(int(np.prod(ar.raw(self._vars[v]).shape)) * ar.raw(self._vars[v]).dtype.itemsize
                    if isinstance(ar.raw(self._vars[v]), np.ndarray)
                    else ar.raw(self._vars[v]).numel() * ar.raw(self._vars[v]).element_size() for v in todo)
        free, _ = torch.cuda.mem_get_info(device)
        if total > 0.4 * free:
            return
        for v in todo:
            r = ar.raw(self._vars[v])
            if isinstance(r, np.ndarray):
                if r.dtype.byteorder not in ('=', '|') or not r.flags.writeable or not r.flags.c_contiguous:
                    r = np.ascontiguousarray(r, dtype=r.dtype.newbyteorder('='))
                r = torch.from_numpy(r)
            r = r.contiguous()
            d = torch.empty(r.shape, dtype=r.dtype, device=device)
            flat_s, flat_d = r.view(-1), d.view(-1)
            step = (256 << 20) // r.element_size()
            for k0, o in enumerate(range(0, flat_s.numel(), step)):
                piece = flat_s[o:o + step]
                if not piece.is_pinned():
                    self._pending_stage_events = []
                    piece = self._stage_pinned(piece, ('whole', k0 % 2))
                    flat_d[o:o + step].copy_(piece, non_blocking=True)
                    for pe in self._pending_stage_events:
                        pe.record(torch.cuda.current_stream(device))
                else:
                    flat_d[o:o + step].copy_(piece, non_blocking=True)
            self._whole[v] = d

    def _stage_pinned(self, r, slot):
        '''Pageable host tensor -> pinned staging tensor (process-wide cache, one per (device, buffer set, field),
        capped by TEMD_STAGING_MAX_BYTES and freed by `release_host_staging()`) by a multi-threaded memcpy in libtemd,
        so the following H2D copy is an asynchronous DMA.'''
        import ctypes as C
        import os
        eng = self.ZM._engine
        nbytes = r.numel() * r.element_size()
        key = (str(eng.device), slot)
        ent = _HOST_STAGING.get(key)
        if ent is None or ent[0].numel() < nbytes:
            _HOST_STAGING.pop(key, None)
            cap = int(os.environ.get('TEMD_STAGING_MAX_BYTES', 8 << 30))
            if sum(e[0].numel() for e in _HOST_STAGING.values()) + nbytes > cap:
                release_host_staging()
            ent = [torch.empty(nbytes, dtype=torch.uint8).pin_memory(), None]
            _HOST_STAGING[key] = ent
        if ent[1] is not None:
            ent[1].synchronize()          # the previous DMA out of this staging buffer must have finished
        rc = eng.lib.temd_host_copy(C.c_void_p(ent[0].data_ptr()), C.c_void_p(r.data_ptr()), nbytes,
                                    max(1, min(8, (os.cpu_count() or 2) // 2)))
        if rc:
            raise RuntimeError('temd_host_copy failed')
        ev_ = torch.cuda.Event()
        out = ent[0][:nbytes].view(r.dtype).view(r.shape)
        ent[1] = ev_
        self._pending_stage_events.append(ev_)
        return out

    def _compute_all(self):
        '''_compute_potential_temperature, _decompose_zm_eddy, _compute_fluxes, _compute_derivatives
        (tem_diagnostics.py:491-611) and every diagnostics method (:615-797), on the GPU.

        The record is processed in time slabs (time steps are independent): while slab i is in the
        project / eddy-flux kernels on the compute stream, slab i+1 is copied host->device (or
        re-laid-out) on a second stream.'''
        eng = self.ZM._engine
        with eng.lock:      # cached engines are shared: per-call state (epilogue planes, staging) is not re-entrant
            self._compute_all_locked(eng)

    def _compute_all_locked(self, eng):
        dev = eng.device
        K, T, N = self.NLEV, self.NT, self.NCOL
        # theta = T (p0/p)^k per level (tem_diagnostics.py:498), in the input's level order
        p_in = self._plev_input_order * 100
        lev_scale = eng._dev((self.p0 / p_in) ** const.k)
        ntr = self.ntrac
        names = ('ua', 'va', 'ta', 'wap') + tuple('q{}'.format(i) for i in range(ntr))
        nf = len(names)
        ld = N + (N & 1)
        zero_copy = all(self._is_native_device_layout(v, dev) for v in names)
        # slab size: in-place device inputs need no staging, so the whole record goes in one launch (best wave
        # quantisation); host inputs stream through two ~2 GB staging sets
        budget = self._slab_bytes if self._slab_bytes is not None else ((1 << 42) if zero_copy else (2 << 30))
        ts = max(1, min(T, int(budget // (nf * 8 * K * N))))
        coef = torch.empty((7, T * K, eng.lpad), dtype=torch.float64, device=dev)
        coefq = torch.empty((3 * ntr, T * K, eng.lpad), dtype=torch.float64, device=dev) if ntr else None

        def compute(xs, t0, t1):
            c4, cf = eng.tem_coefficients(xs[:4], lev_scale, K)
            coef[:4, t0 * K:t1 * K] = c4
            coef[4:, t0 * K:t1 * K] = cf
            if ntr:
                # tracers (tem_diagnostics.py:532-538, 560-570): qb, q'v', q'omega' per tracer
                coefq[:, t0 * K:t1 * K] = eng.tracer_coefficients(xs[4:], xs[:4], c4, lev_scale, K)

        with torch.cuda.device(dev):
            if zero_copy:
                # float64 CUDA tensors already laid out (time, lev, ncol): the kernels read them in place
                for t0 in range(0, T, ts):
                    t1 = min(T, t0 + ts)
                    compute([ar.raw(self._vars[v])[t0:t1].reshape(-1, N) for v in names], t0, t1)
            else:
                # two fixed staging sets: slab i+1 is copied / re-laid-out on a side stream into one set while
                # slab i is computed from the other (no per-slab allocation, no cross-stream allocator traffic)
                main = torch.cuda.current_stream(dev)
                side = torch.cuda.Stream(dev)
                self._upload_whole(names, dev)
                bufs = [[torch.empty((ts * K, ld), dtype=torch.float64, device=dev) for _ in names] for _ in range(2)]
                if ld != N:
                    for set_ in bufs:
                        for b_ in set_:
                            b_[:, N:].zero_()
                filled = [None, None]
                consumed = [None, None]
                side.wait_stream(main)

                def fill(i, t0, t1):
                    with torch.cuda.stream(side):
                        if consumed[i % 2] is not None:
                            side.wait_event(consumed[i % 2])
                        self._pending_stage_events = []
                        for fi_, (v, dst) in enumerate(zip(names, bufs[i % 2])):
                            self._fill(dst, v, t0, t1, dev, slot=(i % 2, fi_))
                        ev_ = torch.cuda.Event()
                        ev_.record(side)
                        for pe in self._pending_stage_events:
                            pe.record(side)       # marks the end of the DMAs that read the pinned staging buffers
                    filled[i % 2] = ev_

                # slabs of ts steps, except that the LAST one is halved down to single steps: what is left to do after the
                # final host->device copy (the path is copy-bound) is then the compute of one step, not of a whole slab
                slabs = _slab_schedule(T, ts)
                fill(0, *slabs[0])
                for i, (t0, t1) in enumerate(slabs):
                    if i + 1 < len(slabs):
                        fill(i + 1, *slabs[i + 1])
                    main.wait_event(filled[i % 2])
                    compute([b_[:(t1 - t0) * K, :N] for b_ in bufs[i % 2]], t0, t1)
                    ev_ = torch.cuda.Event()
                    ev_.record(main)
                    consumed[i % 2] = ev_
                main.wait_stream(side)
                self._whole = {}
        def classify(vs):
            # failure path only: look at the inputs themselves (a time step at a time) to tell NaN from infinity
            def run():
                found = None
                for v in vs:
                    for t0 in range(T):
                        k_ = eng.scan_nonfinite(self._slab(v, t0, t0 + 1, dev))
                        if k_ == 'nan':
                            return 'nan'
                        found = found or k_
                return found
            return run
        eng.check_finite(coef, 'ua/va/ta/wap', classify(names[:4]))       # sph_zonal_mean.py:219-221
        if ntr:
            eng.check_finite(coefq, 'q', classify(names[4:]))
        self._coef_in = coef           # coefficient rows in the INPUT's level order (for the native-grid properties)
        self._coefq_in = coefq
        self._lev_scale = lev_scale
        if self._flip_lev:
            coef = coef.reshape(7, T, K, eng.lpad).flip(2).reshape(7, T * K, eng.lpad).contiguous()
            if ntr:
                coefq = coefq.reshape(3 * ntr, T, K, eng.lpad).flip(2).reshape(3 * ntr, T * K, eng.lpad).contiguous()
        self._coef = coef
        zm = eng.synth_out(coef).reshape(7, T, K, eng.M)
        res = eng.tem_epilogue(zm, self.p, self._f_zm, self._coslat_zm, p0=self.p0)
        self._dev_results = {n: zm[i] for i, n in enumerate(_ZM_NAMES)}
        self._dev_results.update(res)
        self._cache = {}
        self._host_public = None
        self._dev_tracer = []
        for i in range(ntr):
            zmq = eng.synth_out(coefq[3 * i:3 * i + 3]).reshape(3, T, K, eng.M)
            tr = eng.tracer_epilogue(zmq)
            tr.update(qb=zmq[0], qpvpb=zmq[1], qpwappb=zmq[2])
            self._dev_tracer.append(tr)

    # ------------------------------------------------------------------
    def _result(self, name, like=None, cast_like=None, tracer=None):
        '''(lat, plev, time) array of one result, in the container kind of the inputs.'''
        key = name if tracer is None else (name, tracer)
        if key in self._cache:
            return self._cache[key]
        src_dict = self._dev_results if tracer is None else self._dev_tracer[tracer]
        src = self.ua if cast_like is None else cast_like
        dtype = ar.dtype_of(src)
        r = ar.raw(src)
        in_dev = r.device if isinstance(r, torch.Tensor) else None
        if tracer is None and name in _METHODS and self._kind != 'torch':
            # host-side outputs of the ten diagnostics methods: ONE device->host copy for all of them on first use
            # (ten separate permute + copy round trips cost 7 ms of a 244 ms config-2 call, the batch 1.5 ms)
            if self._host_public is None:
                blk = torch.stack([self._dev_results[n] for n in _METHODS]).permute(0, 3, 2, 1).contiguous()
                self._host_public = blk.cpu().numpy()                      # (10, M, K, T)
            out = self._host_public[_METHODS.index(name)].astype(dtype, copy=False)
        else:
            t = src_dict[name].permute(2, 1, 0).contiguous()           # [T][K][M] -> (M, K, T)
            out = ar.from_device(t, 'numpy' if self._kind == 'dataarray' else self._kind, dtype, in_dev)
        if self._kind == 'dataarray':
            coords = {'lat': self._lat_zm, self.plevname: self.plev, self.timename: self.time}
            out = ar.make_dataarray(self.ua, out, ('lat', self.plevname, self.timename), coords=coords, name=name)
        self._cache[key] = out
        return out

    def _qi(self, qi, who):
        '''tracer-index convention of the reference (e.g. tem_diagnostics.py:814-816)'''
        if qi is None and self.ntrac == 1:
            return 0
        if qi is None and self.ntrac > 1:
            raise RuntimeError('qi must be passed to {}() when len(q) > 1!'.format(who))
        if self.ntrac == 0:
            raise RuntimeError('{}() needs tracers: pass q= to TEMDiagnostics'.format(who))
        return qi

    def _tracer(self, name, qi, who=None):
        qi = self._qi(qi, who or name)
        return self._result(name, cast_like=self.q[qi], tracer=qi)

    def _tracer_list(self, name):
        return [self._result(name, cast_like=self.q[i], tracer=i) for i in range(self.ntrac)]

    # tracer intermediates (tem_diagnostics.py:458-475): lists, one entry per tracer
    qb = property(lambda self: self._tracer_list('qb'))
    qpvpb = property(lambda self: self._tracer_list('qpvpb'))
    qpwappb = property(lambda self: self._tracer_list('qpwappb'))
    dqb_dp = property(lambda self: self._tracer_list('dqb_dp'))
    qbcoslat = property(lambda self: self._tracer_list('qbcoslat'))
    dqbcoslat_dlat = property(lambda self: self._tracer_list('dqbcoslat_dlat'))

    def etfy(self, qi=None):
        '''northward eddy tracer flux (tem_diagnostics.py:801-832)'''
        return self._tracer('etfy', qi)

    def etfz(self, qi=None):
        '''upward eddy tracer flux (tem_diagnostics.py:836-866)'''
        return self._tracer('etfz', qi)

    def etdiv(self, qi=None):
        '''eddy tracer flux divergence (tem_diagnostics.py:870-905)'''
        return self._tracer('etdiv', qi)

    def qtendetfd(self, qi=None):
        '''tracer tendency due to eddy tracer flux divergence (tem_diagnostics.py:909-934)'''
        return self._tracer('qtendetfd', qi)

    def qtendvtem(self, qi=None):
        '''tracer tendency due to TEM northward advection (tem_diagnostics.py:938-965)'''
        return self._tracer('qtendvtem', qi)

    def qtendwtem(self, qi=None):
        '''tracer tendency due to TEM upward advection (tem_diagnostics.py:969-991)'''
        return self._tracer('qtendwtem', qi)

    # zonal means and derived intermediates (tem_diagnostics.py:412-457)
    ub = property(lambda self: self._result('ub'))
    vb = property(lambda self: self._result('vb', cast_like=self.va))
    thetab = property(lambda self: self._result('thetab', cast_like=self.ta))
    wapb = property(lambda self: self._result('wapb', cast_like=self.wap))
    upvpb = property(lambda self: self._result('upvpb'))
    upwappb = property(lambda self: self._result('upwappb'))
    vptpb = property(lambda self: self._result('vptpb'))
    dub_dp = property(lambda self: self._result('dub_dp'))
    dthetab_dp = property(lambda self: self._result('dthetab_dp'))
    ubcoslat = property(lambda self: self._result('ubcoslat'))
    dubcoslat_dlat = property(lambda self: self._result('dubcoslat_dlat'))
    psicoslat = property(lambda self: self._result('psicoslat'))
    dpsicoslat_dlat = property(lambda self: self._result('dpsicoslat_dlat'))
    int_vbdp = property(lambda self: self._result('int_vbdp'))
    psi = property(lambda self: self._result('psi'))
    dpsi_dp = property(lambda self: self._result('dpsi_dp'))

    # ---- native-grid eddies and products (tem_diagnostics.py:420-433, 517-529, 547-555): NOT kept by the fused
    #      path; rebuilt on demand, one field at a time, shaped (ncol, plev, time) like the reference's.
    def _native(self, which):
        key = ('native', which)
        if key in self._cache:
            return self._cache[key]
        eng = self.ZM._engine
        dev = eng.device
        K, T, N = self.NLEV, self.NT, self.NCOL
        src = {'up': ('ua', 0, False), 'vp': ('va', 1, False), 'thetap': ('ta', 2, True), 'wapp': ('wap', 3, False)}
        for i in range(self.ntrac):
            src['qp%d' % i] = ('q%d' % i, None, False)
        prod = {'upvp': ('up', 'vp'), 'upwapp': ('up', 'wapp'), 'vptp': ('vp', 'thetap')}
        for i in range(self.ntrac):
            prod['qpvp%d' % i] = ('qp%d' % i, 'vp')
            prod['qpwapp%d' % i] = ('qp%d' % i, 'wapp')

        def eddy(name):
            var, ci, scaled = src[name]
            x = self._slab(var, 0, T, dev)
            c = self._coef_in[ci] if ci is not None else self._coefq_in[3 * int(name[2:])]
            return eng.eddy_native(x, c, self._lev_scale if scaled else None, K)
        if which in src:
            t = eddy(which)
            like = self._vars[src[which][0]]
        else:
            a_, b_ = prod[which]
            t = eng.multiply(eddy(a_), eddy(b_))
            like = self._vars[src[a_][0]]
        t = t.reshape(T, K, N)
        if self._flip_lev:
            t = t.flip(1)
        t = t.permute(2, 1, 0).contiguous()                   # (ncol, plev, time)
        r = ar.raw(like)
        in_dev = r.device if isinstance(r, torch.Tensor) else None
        out = ar.from_device(t, 'numpy' if self._kind == 'dataarray' else self._kind, ar.dtype_of(like), in_dev)
        if self._kind == 'dataarray':
            coords = {self.plevname: self.plev, self.timename: self.time}
            out = ar.make_dataarray(self.ua, out, self.data_dims, coords=coords, name=which.rstrip('0123456789'))
        self._cache[key] = out
        return out

    up = property(lambda self: self._native('up'))
    vp = property(lambda self: self._native('vp'))
    thetap = property(lambda self: self._native('thetap'))
    wapp = property(lambda self: self._native('wapp'))
    upvp = property(lambda self: self._native('upvp'))
    upwapp = property(lambda self: self._native('upwapp'))
    vptp = property(lambda self: self._native('vptp'))
    qp = property(lambda self: [self._native('qp%d' % i) for i in range(self.ntrac)])
    qpvp = property(lambda self: [self._native('qpvp%d' % i) for i in range(self.ntrac)])
    qpwapp = property(lambda self: [self._native('qpwapp%d' % i) for i in range(self.ntrac)])

    @property
    def theta(self):
        """potential temperature on the native grid (tem_diagnostics.py:491-506), rebuilt on demand on the GPU
        (theta = lev_scale * T is the eddy kernel with zero coefficients)."""
        key = ('native', 'theta')
        if key not in self._cache:
            eng = self.ZM._engine
            K, T, N = self.NLEV, self.NT, self.NCOL
            x = self._slab('ta', 0, T, eng.device)
            zero = torch.zeros((T * K, eng.lpad), dtype=torch.float64, device=eng.device)
            t = eng.eddy_native(x, zero, self._lev_scale, K).reshape(T, K, N)
            if self._flip_lev:
                t = t.flip(1)
            t = t.permute(2, 1, 0).contiguous()
            r = ar.raw(self.ta)
            in_dev = r.device if isinstance(r, torch.Tensor) else None
            out = ar.from_device(t, 'numpy' if self._kind == 'dataarray' else self._kind, ar.dtype_of(self.ta), in_dev)
            if self._kind == 'dataarray':
                coords = {self.plevname: self.plev, self.timename: self.time}
                out = ar.make_dataarray(self.ua, out, self.data_dims, coords=coords, name='THETA',
                                        attrs={'long_name': 'potential temperature'})
            self._cache[key] = out
        return self._cache[key]

    @property
    def out_file(self):
        if self._out_file is None:
            warnings.warn('\'out_file\' is not set until to_netcdf() is called')
        return self._out_file

    # ---- diagnostics methods (tem_diagnostics.py:615-797); each is cast to the dtype of the input the
    #      reference casts to (:626,643,661,678,696,714,740,757,777,795)
    def vtem(self):
        '''TEM northward wind [m/s] (tem_diagnostics.py:615-628)'''
        return self._result('vtem', cast_like=self.va)

    def omegatem(self):
        '''TEM upward wind [Pa/s] (tem_diagnostics.py:632-645)'''
        return self._result('omegatem', cast_like=self.wap)

    def wtem(self):
        '''TEM upward wind [m/s] (tem_diagnostics.py:649-663)'''
        return self._result('wtem', cast_like=self.wap)

    def psitem(self):
        '''TEM mass stream function [kg/s] (tem_diagnostics.py:667-680)'''
        return self._result('psitem', cast_like=self.va)

    def epfy(self):
        '''northward EP flux [m3/s2] (tem_diagnostics.py:684-698)'''
        return self._result('epfy')

    def epfz(self):
        '''upward EP flux [m3/s2] (tem_diagnostics.py:702-716)'''
        return self._result('epfz')

    def epdiv(self):
        '''EP flux divergence [m2/s2] (tem_diagnostics.py:720-742)'''
        return self._result('epdiv')

    def utendepfd(self):
        '''eastward-wind tendency due to EP flux divergence [m/s2] (tem_diagnostics.py:746-759)'''
        return self._result('utendepfd')

    def utendvtem(self):
        '''eastward-wind tendency due to TEM northward advection + Coriolis [m/s2] (tem_diagnostics.py:763-779)'''
        return self._result('utendvtem')

    def utendwtem(self):
        '''eastward-wind tendency due to TEM upward advection [m/s2] (tem_diagnostics.py:783-797)'''
        return self._result('utendwtem')

    # ---- file output (tem_diagnostics.py:995-1103).  The reference writes through xarray/netCDF4; neither is a
    #      dependency here, so the files are NetCDF-3 (64-bit offset) written with scipy.io.netcdf_file: same file
    #      names, variable names and dims ('lat', plev, time) / ('ncol', plev, time).
    def _write_nc(self, path, output):
        from scipy.io import netcdf_file
        def _np(x):
            v = x.values if ar.is_dataarray(x) else x
            return v.cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        with netcdf_file(path, 'w', version=2) as nc:
            nc.createDimension('lat', self.ZM_N)
            nc.createDimension(self.plevname, self.NLEV)
            nc.createDimension(self.timename, self.NT)
            for dim, vals in (('lat', self._lat_zm), (self.plevname, self.plev), (self.timename, self.time)):
                vals = np.asarray(vals)
                if vals.dtype.kind in 'iuf':
                    v = nc.createVariable(dim, 'f8', (dim,))
                    v[:] = vals.astype(np.float64)
            for name, val in output.items():
                a_ = _np(val)
                if a_.shape[0] == self.ZM_N:
                    dims = ('lat', self.plevname, self.timename)
                else:
                    if self.ncolname not in nc.dimensions:
                        nc.createDimension(self.ncolname, self.NCOL)
                    dims = (self.ncolname, self.plevname, self.timename)
                v = nc.createVariable(name, a_.dtype.char if a_.dtype.kind == 'f' else 'f8', dims)
                v[:] = a_
        return path

    def to_netcdf(self, loc=None, prefix=None, include_attrs=False):
        '''Saves all TEM quantities to `{prefix_}TEM_{grid}_{gridout}_L{L}.nc` under `loc` (tem_diagnostics.py:995-1041).
        include_attrs=True also writes the intermediates (zonal means, eddies, fluxes, derivatives).'''
        import os
        loc = os.getcwd() if loc is None else loc
        results = {n: getattr(self, n)() for n in _METHODS}
        if include_attrs:
            attrs = {n: getattr(self, n) for n in ('ub', 'up', 'vb', 'vp', 'thetab', 'thetap', 'wapb', 'upvp', 'upvpb',
                                                   'upwapp', 'upwappb', 'vptp', 'vptpb', 'dub_dp', 'dthetab_dp', 'ubcoslat',
                                                   'dubcoslat_dlat', 'psi', 'psicoslat', 'dpsicoslat_dlat', 'dpsi_dp',
                                                   'int_vbdp')}
            attrs['wawpp'] = self.wapp          # key spelled as in the reference (:1011)
            output = dict(attrs, **results)
        else:
            output = results
        prefix = '{}_'.format(prefix) if prefix is not None else ''
        filename = '{}TEM_{}_{}_L{}.nc'.format(prefix, self.ZM.grid_name, self.ZM.grid_out_name, self.L)
        self._out_file = '{}/{}'.format(loc, filename)
        self._write_nc(self._out_file, output)
        self._log('wrote TEM data to {}'.format(self._out_file))
        return self._out_file

    @property
    def q_out_file(self):
        if len(self._q_out_file) == 0:
            warnings.warn('\'q_out_file\' is emtpy; no tracers currently present')
        elif self._q_out_file.count(None) == self.ntrac:
            warnings.warn('\'q_out_file\' is not set until q_to_netcdf() is called')
        return self._q_out_file

    def q_to_netcdf(self, loc=None, qi=None, prefix=None, include_attrs=False):
        '''One file per tracer, `{prefix_}TEM_{grid}_{gridout}_L{L}_TRACER-{name}.nc` (tem_diagnostics.py:1045-1103).'''
        import os
        assert self.ntrac > 0, 'No tracers to output (argument `q` not passed at object construction)'
        loc = os.getcwd() if loc is None else loc
        prefix = '{}_'.format(prefix) if prefix is not None else ''
        names = [getattr(qq, 'name', None) if ar.is_dataarray(qq) else None for qq in self.q]
        names = [n if n is not None else 'q{}'.format(i) for i, n in enumerate(names)]
        for i in (range(self.ntrac) if qi is None else [qi]):
            output = {"etfy": self.etfy(i), "etfz": self.etfz(i), "etdiv": self.etdiv(i), "qtendetfd": self.qtendetfd(i),
                      "qtendvtem": self.qtendvtem(i), "qtendwtem": self.qtendwtem(i)}
            if include_attrs:
                output.update({"qpvp": self.qpvp[i], "qpwapp": self.qpwapp[i], "qpvpb": self.qpvpb[i],
                               "qpwappb": self.qpwappb[i], "dqp_dp": self.dqb_dp[i], "qbcoslat": self.qbcoslat[i],
                               "dqbcoslat_dlat": self.dqbcoslat_dlat[i]})
            filename = '{}TEM_{}_{}_L{}_TRACER-{}.nc'.format(prefix, self.ZM.grid_name, self.ZM.grid_out_name, self.L, names[i])
            self._q_out_file[i] = '{}/{}'.format(loc, filename)
            self._write_nc(self._q_out_file[i], output)
        return self._q_out_file
