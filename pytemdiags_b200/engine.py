"""Thin host-side driver over libtemd: owns a `temd_plan`, hands torch device tensors to the C ABI.

PyTorch is used for device memory and streams only; every numerical operation on the hot path is a
libtemd kernel launch.  No CPU fallback: constructing an Engine without the library or without a
CUDA device raises.
"""
import ctypes as C
import threading

import numpy as np
import torch

from . import _lib
from .constants import P0, H, a, g0, pi


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def gradient_coefficients(x):
    """Interior coefficients of `np.gradient(f, x)` (NumPy's second-order non-uniform stencil) and its
    uniform-spacing branch flag, reproducing numpy/lib/function_base.py::gradient.

    Returns (coef[3][n] float64, uniform: bool, h: float).
    """
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    coef = np.zeros((3, n))
    dx = np.diff(x)
    uniform = bool((dx == dx[0]).all())
    if n > 2:
        dx1, dx2 = dx[:-1], dx[1:]
        coef[0, 1:-1] = -(dx2) / (dx1 * (dx1 + dx2))
        coef[1, 1:-1] = (dx2 - dx1) / (dx1 * dx2)
        coef[2, 1:-1] = dx1 / (dx2 * (dx1 + dx2))
    return coef, uniform, float(dx[0])


def _check_rank(lat, L):
    """Y0 (N x (L+1)) has rank min(L+1, number of distinct latitudes).  The reference's lstsq (gelsd) silently returns
    the minimum-norm solution when that is < L+1 (sph_zonal_mean.py:389), e.g. the default L=50 on a lat-lon grid with
    fewer than 51 latitudes; this build refuses, early and with the remedy (documented deviation, INTEGRATION.md)."""
    if L + 1 > 8 and np.unique(lat).shape[0] < L + 1:
        raise RuntimeError('basis is rank-deficient: L+1 = {} Legendre degrees but only {} distinct latitudes among the {} '
                           'native columns; lower L to at most {} (the reference would return a minimum-norm '
                           'least-squares fit here; this build does not)'.format(
                               L + 1, np.unique(lat).shape[0], lat.shape[0], np.unique(lat).shape[0] - 1))


def _unique_nodes(lat):
    """x = cos(colatitude) of every column, computed like the reference (sph_zonal_mean.py:358), and its distinct
    values: (x, x_unique, inverse, counts) as np.unique returns them."""
    x = np.cos(np.deg2rad(90 - lat))
    xu, inv, cnt = np.unique(x, return_inverse=True, return_counts=True)
    return x, xu, inv, cnt


class Engine:
    """One zonal-averaging plan (native grid, output grid, truncation L) on one GPU.

    `min_norm=True`: the basis is built by temd_basis_build_min_norm, so a rank-deficient Y0 gives NumPy's
    minimum-norm least-squares answer instead of an error; `rank` is then the number of directions kept."""

    def __init__(self, lat, lat_out, L, device=None, min_norm=False):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError('pytemdiags_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self.lat = np.ascontiguousarray(np.asarray(lat, dtype=np.float64))
        self.lat_out = np.ascontiguousarray(np.asarray(lat_out, dtype=np.float64))
        self.N, self.M, self.L = int(self.lat.shape[0]), int(self.lat_out.shape[0]), int(L)
        self.Mld = self.M + (self.M & 1)
        self.min_norm = bool(min_norm)
        if not self.min_norm:
            _check_rank(self.lat, self.L)
        self._plan = C.c_void_p(0)
        self._create_plan(self.N)
        self.built = False
        self.sanity = None
        self.rank = None
        self.lock = threading.RLock()   # serialises callers that share this (cached) engine's per-call state

    def _create_plan(self, ncol):
        create = self.lib.temd_plan_create_min_norm if self.min_norm else self.lib.temd_plan_create
        _lib.check(create(self.device.index or 0, ncol, self.L, self.M, C.byref(self._plan)),
                   'temd_plan_create_min_norm' if self.min_norm else 'temd_plan_create')
        self.lpad = self.lib.temd_plan_lpad(self._plan)

    def _build_min_norm(self, x, xu, cnt, x_out, sanity):
        """temd_basis_build_min_norm; x = None on a plan created on the unique nodes."""
        xu_d, mult = self._dev(xu), self._dev(cnt.astype(np.float64))
        san = (C.c_double * 2)()
        rank = C.c_int(0)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_basis_build_min_norm(self._plan, _ptr(x), _ptr(xu_d), _ptr(mult), int(xu.shape[0]),
                                                    _ptr(x_out), C.byref(rank), san if sanity else None, self.stream)
        _lib.check(rc, 'temd_basis_build_min_norm')
        self.built = True
        self.rank = int(rank.value)
        if sanity:
            self.sanity = (san[0], san[1])
        return self

    def __del__(self):
        try:
            if getattr(self, '_plan', None) and self._plan.value:
                self.lib.temd_plan_destroy(self._plan)
                self._plan = C.c_void_p(0)
        except Exception:
            pass

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, arr):
        return torch.as_tensor(np.ascontiguousarray(arr, dtype=np.float64)).to(self.device)

    # ---- sph_compute_matrices (sph_zonal_mean.py:302-422) ----
    def build_basis(self, sanity=False, weights=None):
        if self.min_norm and weights is not None:
            raise RuntimeError('min_norm=True is not available together with weights=')
        # x = cos(colatitude), computed exactly like the reference: coalt = deg2rad(90 - lat)
        x = self._dev(np.cos(np.deg2rad(90 - self.lat)))
        x_out = self._dev(np.cos(np.deg2rad(90 - self.lat_out)))
        if self.min_norm:
            _, xu, _, cnt = _unique_nodes(self.lat)
            return self._build_min_norm(x, xu, cnt, x_out, sanity)
        if weights is not None:
            # deprecated reference path: Y0inv = Y0^T diag(4 pi w)  (sph_zonal_mean.py:180-181,383-386)
            w = self._dev(4 * np.pi * np.asarray(weights, dtype=np.float64))
            with torch.cuda.device(self.device):
                rc = self.lib.temd_basis_build_weighted(self._plan, _ptr(x), _ptr(x_out), _ptr(w), self.stream)
            _lib.check(rc, 'temd_basis_build_weighted')
            self.built = True
            self.rank = self.L + 1
            return self
        san = (C.c_double * 2)()
        with torch.cuda.device(self.device):
            rc = self.lib.temd_basis_build(self._plan, _ptr(x), _ptr(x_out), san if sanity else None, self.stream)
        _lib.check(rc, 'temd_basis_build')
        self.built = True
        self.rank = self.L + 1
        if sanity:
            self.sanity = (san[0], san[1])
        return self

    def export_matrices(self, Y0=True, Y0inv=True, Y0p=True):
        """Dense Y0 (N,L+1), Y0inv (L+1,N), Y0p (M,L+1) as device tensors (reference attributes)."""
        Lp = self.L + 1
        o0 = torch.empty((self.N, Lp), dtype=torch.float64, device=self.device) if Y0 else None
        oi = torch.empty((Lp, self.N), dtype=torch.float64, device=self.device) if Y0inv else None
        op = torch.empty((self.M, Lp), dtype=torch.float64, device=self.device) if Y0p else None
        with torch.cuda.device(self.device):
            rc = self.lib.temd_basis_export(self._plan, _ptr(o0), _ptr(oi), _ptr(op), self.stream)
        _lib.check(rc, 'temd_basis_export')
        return o0, oi, op

    # ---- zonal-mean pieces ----
    def _check_field(self, x):
        if not (x.is_cuda and x.dtype == torch.float64 and x.dim() == 2 and x.shape[1] == self.N
                and x.stride(1) == 1 and x.stride(0) % 2 == 0 and x.data_ptr() % 16 == 0):
            raise RuntimeError('field must be a float64 CUDA tensor [rows][ncol], ncol contiguous, even row stride, '
                               '16-byte aligned')

    def project(self, fields, lev_scale=None, scale_field=-1, nlev=1):
        """coef[f][row][lpad] = Q^T fields[f][row][:]  (fields: list of [rows][N] device tensors)."""
        rows, ld = fields[0].shape[0], fields[0].stride(0)
        for x in fields:
            self._check_field(x)
            if x.shape[0] != rows or x.stride(0) != ld:
                raise RuntimeError('all fields must share shape and stride')
        coef = torch.empty((len(fields), rows, self.lpad), dtype=torch.float64, device=self.device)
        ptrs = (C.c_void_p * len(fields))(*[x.data_ptr() for x in fields])
        with torch.cuda.device(self.device):
            rc = self.lib.temd_project(self._plan, ptrs, len(fields), rows, ld, _ptr(lev_scale), scale_field, nlev,
                                       _ptr(coef), self.stream)
        _lib.check(rc, 'temd_project')
        return coef

    def synth_out(self, coef):
        """[.., rows, lpad] -> zonal means on the output latitudes [.., rows, M] (view of an Mld-strided buffer)."""
        c2 = coef.reshape(-1, self.lpad)
        out = torch.empty((c2.shape[0], self.Mld), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_synth_out(self._plan, _ptr(c2), c2.shape[0], _ptr(out), self.Mld, self.stream)
        _lib.check(rc, 'temd_synth_out')
        return out.reshape(tuple(coef.shape[:-1]) + (self.Mld,))[..., :self.M]

    def synth_out_dlat(self, coef):
        """[.., rows, lpad] -> d/dphi (per radian) of the zonal means on the output latitudes, by differentiating the
        Legendre basis (optional extra; the reference uses finite differences)."""
        c2 = coef.reshape(-1, self.lpad)
        out = torch.empty((c2.shape[0], self.Mld), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_synth_out_dlat(self._plan, _ptr(c2), c2.shape[0], _ptr(out), self.Mld, self.stream)
        _lib.check(rc, 'temd_synth_out_dlat')
        return out.reshape(tuple(coef.shape[:-1]) + (self.Mld,))[..., :self.M]

    def export_dY0p(self):
        """Dense dY0p (M, L+1): latitude derivative of the basis at the output latitudes."""
        out = torch.empty((self.M, self.L + 1), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_basis_export_dlat(self._plan, _ptr(out), self.stream)
        _lib.check(rc, 'temd_basis_export_dlat')
        return out

    def synth_native(self, coef, out=None):
        c2 = coef.reshape(-1, self.lpad)
        ld = self.N + (self.N & 1)
        if out is None:
            out = torch.empty((c2.shape[0], ld), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_synth_native(self._plan, _ptr(c2), c2.shape[0], _ptr(out), out.stride(0), self.stream)
        _lib.check(rc, 'temd_synth_native')
        return out[:, :self.N]

    def eddy_native(self, x, coef, lev_scale=None, nlev=1):
        """x: [rows][N] field, coef: [rows][lpad] -> eddy field [rows][N] (on-demand properties only)."""
        self._check_field(x)
        rows = x.shape[0]
        ld = self.N + (self.N & 1)
        out = torch.empty((rows, ld), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_eddy_native(self._plan, _ptr(x), x.stride(0), _ptr(coef), rows, _ptr(lev_scale), nlev,
                                           _ptr(out), ld, self.stream)
        _lib.check(rc, 'temd_eddy_native')
        return out[:, :self.N]

    def multiply(self, a_, b_):
        rows, n = a_.shape
        out = torch.empty((rows, n + (n & 1)), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_multiply(_ptr(a_), a_.stride(0), _ptr(b_), b_.stride(0), _ptr(out), out.stride(0), rows, n,
                                        self.stream)
        _lib.check(rc, 'temd_multiply')
        return out[:, :n]

    def scan_nonfinite(self, t):
        """'nan' if the device tensor holds a NaN, 'inf' if it holds infinities but no NaN, else None."""
        t = t if t.dtype == torch.float64 and t.is_contiguous() else t.to(torch.float64).contiguous()
        with torch.cuda.device(self.device):
            rc = self.lib.temd_check_finite(_ptr(t), t.numel(), self.stream)
        if rc == -2:
            return 'nan'
        if rc == -6:
            return 'inf'
        _lib.check(rc, 'temd_check_finite')
        return None

    def check_finite(self, t, what='input', classify=None):
        """NaN screen of sph_zonal_mean.py:219-221.  `t` is normally the small coefficient block (non-finite inputs
        propagate into it); `classify()` is then called on failure only and looks at the inputs themselves, because an
        infinity in a field also turns into NaN coefficients while the reference screens NaN only."""
        kind = self.scan_nonfinite(t)
        if kind is None:
            return
        if classify is not None:
            kind = classify()
        if kind == 'nan':
            # same failure the reference raises at sph_zonal_mean.py:219-221
            raise RuntimeError('Variable {} has nans! Spectral zonal averager cannot handle nans; '
                               'please replace or remove them'.format(what))
        if kind == 'inf':
            # the reference lets infinities through and returns inf/nan results; fail loudly instead
            raise RuntimeError('Variable {} has infinite values (no nans); the spectral zonal mean of such a field '
                               'is undefined'.format(what))
        raise RuntimeError('Variable {}: all inputs are finite but the projection overflowed'.format(what))

    def eddy_flux_project(self, u, v, t, w, coef4, lev_scale, nlev):
        for x in (u, v, t, w):
            self._check_field(x)
        rows, ld = u.shape[0], u.stride(0)
        out = torch.empty((3, rows, self.lpad), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_eddy_flux_project(self._plan, _ptr(u), _ptr(v), _ptr(t), _ptr(w), rows, ld, _ptr(coef4),
                                                 _ptr(lev_scale), nlev, _ptr(out), self.stream)
        _lib.check(rc, 'temd_eddy_flux_project')
        return out

    # ---- _decompose_zm_eddy + _compute_fluxes (tem_diagnostics.py:510-558) as coefficient blocks ----
    def tem_coefficients(self, xs, lev_scale, nlev):
        """xs = (u, v, T, omega) as [rows][N] device tensors -> ([4][rows][lpad] coefficients of ub, vb, thetab, wapb,
        [3][rows][lpad] coefficients of upvpb, upwappb, vptpb)."""
        c4 = self.project(list(xs[:4]), lev_scale=lev_scale, scale_field=2, nlev=nlev)
        # libtemd picks the implementation: the fully fused kernel for L + 1 <= 104, the split synth-eddy /
        # product-projection pipeline above that (eddies go through a bounded scratch buffer, a row batch at a time)
        return c4, self.eddy_flux_project(xs[0], xs[1], xs[2], xs[3], c4, lev_scale, nlev)

    def tracer_coefficients(self, qs, xs, c4, lev_scale, nlev):
        """Tracer TEM inputs (tem_diagnostics.py:532-538,560-570).  qs: list of [rows][N] tracers; xs, c4 as in
        tem_coefficients.  Returns [3 * len(qs)][rows][lpad]: per tracer the coefficients of qb, qpvpb, qpwappb.
        All tracers are projected in one launch; the fused kernel then runs per tracer on (q, v, theta, omega), whose
        first two product slots are q'v' and q'omega'."""
        rows = xs[0].shape[0]
        out = torch.empty((3 * len(qs), rows, self.lpad), dtype=torch.float64, device=self.device)
        cq_all = torch.cat([self.project(list(qs[i:i + 8])) for i in range(0, len(qs), 8)], 0)
        out[0::3] = cq_all
        i = 0
        while i + 1 < len(qs):       # two tracers per launch: v' and omega' are synthesised once for the pair
            c4p = torch.cat([cq_all[i:i + 2], c4[1:2], c4[3:4]], 0)
            fl = self.tracer_flux_project(qs[i], qs[i + 1], xs[1], xs[3], c4p)
            out[3 * i + 1:3 * i + 3] = fl[0:2]
            out[3 * i + 4:3 * i + 6] = fl[2:4]
            i += 2
        if i < len(qs):              # an odd tracer out: the TEM kernel on (q, v, theta, omega), first two product slots
            c4q = torch.cat([cq_all[i:i + 1], c4[1:]], 0)
            out[3 * i + 1:3 * i + 3] = self.eddy_flux_project(qs[i], xs[1], xs[2], xs[3], c4q, lev_scale, nlev)[:2]
        return out

    def tracer_flux_project(self, q1, q2, v, w, coef4):
        """coef4 = [4][rows][lpad] coefficients of (q1, q2, v, omega) -> [4][rows][lpad] of q1'v', q1'omega', q2'v', q2'omega'."""
        for x in (q1, q2, v, w):
            self._check_field(x)
        rows, ld = v.shape[0], v.stride(0)
        out = torch.empty((4, rows, self.lpad), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_tracer_flux_project(self._plan, _ptr(q1), _ptr(q2), _ptr(v), _ptr(w), rows, ld,
                                                   _ptr(coef4.contiguous()), _ptr(out), self.stream)
        _lib.check(rc, 'temd_tracer_flux_project')
        return out

    def tem_epilogue(self, zm, p_pa, f, coslat, p0=P0):
        """zm: [7][nt][nlev][Mld-strided M] device tensor (as returned by synth_out on a [7][nt*nlev][lpad]
        coefficient block).  Returns dict name -> [nt][nlev][M] device tensors."""
        nt, nlev = zm.shape[1], zm.shape[2]
        assert zm.shape[0] == 7 and zm.shape[3] == self.M and zm.stride(2) == self.Mld and zm.stride(3) == 1
        # the small coordinate / stencil-coefficient vectors are uploaded once per (p, f, coslat) and cached
        key = (np.asarray(p_pa, dtype=np.float64).tobytes(), np.asarray(f, dtype=np.float64).tobytes(),
               np.asarray(coslat, dtype=np.float64).tobytes())
        cached = getattr(self, '_epi_cache', None)
        if cached is None or cached[0] != key:
            latr = np.deg2rad(self.lat_out)
            gp, p_uni, hp = gradient_coefficients(p_pa)
            gl, l_uni, hl = gradient_coefficients(latr)
            packed = self._dev(np.concatenate([np.ravel(x) for x in (p_pa, latr, gp, gl, coslat, f)]))
            nl, nm = len(p_pa), self.M
            offs = np.cumsum([0, nl, nm, 3 * nl, 3 * nm, nm, nm])
            d = {n: packed[offs[i]:offs[i + 1]] for i, n in enumerate(('p', 'latr', 'gp', 'gl', 'coslat', 'f'))}
            d['_packed'] = packed
            self._epi_cache = (key, d, p_uni, hp, l_uni, hl)
        _, d, p_uni, hp, l_uni, hl = self._epi_cache
        nout = len(_lib.EPILOGUE_OUTPUTS)
        out = torch.empty((nout + 2, nt, nlev, self.Mld), dtype=torch.float64, device=self.device)
        args = _lib.EpilogueArgs(nt=nt, nlev=nlev, nlat=self.M, ld=self.Mld, zm=zm.data_ptr(), p=d['p'].data_ptr(),
                                 latr=d['latr'].data_ptr(), gp=d['gp'].data_ptr(), gl=d['gl'].data_ptr(),
                                 p_uniform=int(p_uni), lat_uniform=int(l_uni), hp=hp, hlat=hl,
                                 coslat=d['coslat'].data_ptr(), f=d['f'].data_ptr(),
                                 p0=float(p0), a=a, H=H, g0=g0, pi=pi, out=out.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.temd_tem_epilogue(self._plan, C.byref(args), self.stream)
        _lib.check(rc, 'temd_tem_epilogue')
        self._keepalive = d
        self._epi_full = out          # [nout+2][nt][nlev][Mld] (padded planes, needed by the tracer epilogue)
        self._epi_consts = (d, p_uni, hp, l_uni, hl, float(p0))
        return {name: out[i, :, :, :self.M] for i, name in enumerate(_lib.EPILOGUE_OUTPUTS)}

    def tracer_epilogue(self, zmq):
        """zmq: [3][nt][nlev][Mld-strided M] (qb, qpvpb, qpwappb) -> dict of tracer diagnostics.  Must follow
        tem_epilogue (uses its psi / vtem / omegatem planes)."""
        nt, nlev = zmq.shape[1], zmq.shape[2]
        assert zmq.shape[0] == 3 and zmq.stride(2) == self.Mld and zmq.stride(3) == 1
        d, p_uni, hp, l_uni, hl, p0 = self._epi_consts
        names = _lib.EPILOGUE_OUTPUTS
        full = self._epi_full
        nout = len(_lib.TRACER_OUTPUTS)
        out = torch.empty((nout + 2, nt, nlev, self.Mld), dtype=torch.float64, device=self.device)
        args = _lib.TracerArgs(nt=nt, nlev=nlev, nlat=self.M, ld=self.Mld, zmq=zmq.data_ptr(),
                               psi=full[names.index('psi')].data_ptr(), vtem=full[names.index('vtem')].data_ptr(),
                               omegatem=full[names.index('omegatem')].data_ptr(), p=d['p'].data_ptr(),
                               latr=d['latr'].data_ptr(), gp=d['gp'].data_ptr(), gl=d['gl'].data_ptr(),
                               p_uniform=int(p_uni), lat_uniform=int(l_uni), hp=hp, hlat=hl,
                               coslat=d['coslat'].data_ptr(), p0=p0, a=a, H=H, out=out.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.temd_tracer_epilogue(self._plan, C.byref(args), self.stream)
        _lib.check(rc, 'temd_tracer_epilogue')
        return {name: out[i, :, :, :self.M] for i, name in enumerate(_lib.TRACER_OUTPUTS)}

    def synth_fields(self, field, seed, t0, nt, plev_hpa, lat_rad_dev, lon_rad_dev, plev_dev, out=None):
        nlev = plev_dev.shape[0]
        ld = self.N + (self.N & 1)
        if out is None:
            out = torch.empty((nt * nlev, ld), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_synth_fields(_ptr(out), field, seed, t0, nt, nlev, self.N, out.stride(0),
                                            _ptr(lat_rad_dev), _ptr(lon_rad_dev), _ptr(plev_dev), self.stream)
        _lib.check(rc, 'temd_synth_fields')
        return out[:, :self.N]


class DedupEngine(Engine):
    """Structure-exploiting variant (SURVEY.md §8f-4, opt-in `dedup=True`): the plan lives on the U unique values of
    x = sin(lat); fields are reduced to per-group sums in ONE pass (csrc/temd_dedup.cu) and every tensor-core kernel
    runs on U columns instead of N.  Same method surface and the same coefficients (to rounding) as `Engine`."""

    def __init__(self, lat, lat_out, L, device=None, min_norm=False):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError('pytemdiags_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self.lat = np.ascontiguousarray(np.asarray(lat, dtype=np.float64))
        self.lat_out = np.ascontiguousarray(np.asarray(lat_out, dtype=np.float64))
        self.N, self.M, self.L = int(self.lat.shape[0]), int(self.lat_out.shape[0]), int(L)
        self.Mld = self.M + (self.M & 1)
        self.min_norm = bool(min_norm)
        # group the columns by the exact value of the basis argument (computed like the reference: sph_zonal_mean.py:358)
        x, xu, inv, cnt = _unique_nodes(self.lat)
        self.NU = int(xu.shape[0])
        if self.NU < self.L + 1 and not self.min_norm:
            _check_rank(self.lat, self.L)
        self.Uld = self.NU + (self.NU & 1)
        self.multiplicity = self.N / self.NU
        # number the groups by their first column instead of by x: consecutive groups then start at (nearly)
        # consecutive columns, and on symmetric grids (cubed sphere: mirror images in other faces) so do their other
        # members - the thread-per-group gather of k_gsum_thread touches full 32-byte sectors instead of 8 bytes of each.
        # The order of the unique nodes is irrelevant to the algebra.  Raveled lat-lon grids are already in this order.
        first = np.full(self.NU, self.N, dtype=np.int64)
        np.minimum.at(first, inv, np.arange(self.N))
        order = np.argsort(first, kind='stable')
        newid = np.empty(self.NU, dtype=np.int64)
        newid[order] = np.arange(self.NU)
        xu, cnt, inv = xu[order], cnt[order], newid[inv]
        contiguous = bool(np.all(np.diff(inv) >= 0))
        perm = None if contiguous else np.argsort(inv, kind='stable')
        goff = np.concatenate([[0], np.cumsum(cnt)])
        self._xu = xu
        self._cnt_minmax = (int(cnt.min()), int(cnt.max()))
        self._even_groups = int(bool(np.all(goff % 2 == 0)))
        i32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(self.device)
        self._perm = None if perm is None else i32(perm)
        self._goff, self._gid = i32(goff), i32(inv)
        self._mult = self._dev(cnt.astype(np.float64))
        self._rsq = self._dev(1.0 / np.sqrt(cnt.astype(np.float64)))
        self._cnt = cnt
        self._plan = C.c_void_p(0)
        self._create_plan(self.NU)
        self.built = False
        self.sanity = None
        self.rank = None
        self.lock = threading.RLock()

    def build_basis(self, sanity=False, weights=None):
        if weights is not None:
            raise RuntimeError('dedup=True is not available with the deprecated quadrature-weights inverse')
        x_out = self._dev(np.cos(np.deg2rad(90 - self.lat_out)))
        if self.min_norm:
            return self._build_min_norm(None, self._xu, self._cnt, x_out, sanity)
        xu = self._dev(self._xu)
        san = (C.c_double * 2)()
        with torch.cuda.device(self.device):
            rc = self.lib.temd_basis_build_dedup(self._plan, _ptr(xu), _ptr(x_out), _ptr(self._mult),
                                                 san if sanity else None, self.stream)
        _lib.check(rc, 'temd_basis_build_dedup')
        self.built = True
        self.rank = self.L + 1
        if sanity:
            self.sanity = (san[0], san[1])
        return self

    # ---- pieces on the unique grid ----
    def group_sums(self, fields, lev_scale=None, scale_field=-1, nlev=1, with_products=False):
        rows, ld = fields[0].shape[0], fields[0].stride(0)
        for x in fields:
            self._check_field(x)
            if x.shape[0] != rows or x.stride(0) != ld:
                raise RuntimeError('all fields must share shape and stride')
        nplanes = _lib.GS_NPLANES if with_products else len(fields)
        out = torch.empty((nplanes, rows, self.Uld), dtype=torch.float64, device=self.device)
        if self.Uld != self.NU:
            out[:, :, self.NU:].zero_()
        ptrs = (C.c_void_p * len(fields))(*[x.data_ptr() for x in fields])
        with torch.cuda.device(self.device):
            rc = self.lib.temd_group_sums(ptrs, len(fields), rows, ld, _ptr(self._perm), _ptr(self._goff), self.NU,
                                          self._cnt_minmax[1], self._cnt_minmax[0], self._even_groups, _ptr(self._rsq), _ptr(lev_scale),
                                          scale_field, nlev, int(with_products), _ptr(out), self.Uld, self.stream)
        _lib.check(rc, 'temd_group_sums')
        return out

    def _project_u(self, planes):
        """planes: [nf][rows][Uld] weighted group sums -> [nf][rows][lpad]."""
        nf, rows = planes.shape[0], planes.shape[1]
        coef = torch.empty((nf, rows, self.lpad), dtype=torch.float64, device=self.device)
        ptrs = (C.c_void_p * nf)(*[planes[f].data_ptr() for f in range(nf)])
        with torch.cuda.device(self.device):
            rc = self.lib.temd_project(self._plan, ptrs, nf, rows, self.Uld, None, -1, 1, _ptr(coef), self.stream)
        _lib.check(rc, 'temd_project')
        return coef

    def _synth_u(self, coef):
        """[.., rows, lpad] -> Qw c on the unique grid, [.., rows, Uld] (= sqrt(multiplicity) * native zonal mean)."""
        c2 = coef.reshape(-1, self.lpad)
        out = torch.empty((c2.shape[0], self.Uld), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_synth_native(self._plan, _ptr(c2), c2.shape[0], _ptr(out), self.Uld, self.stream)
        _lib.check(rc, 'temd_synth_native')
        return out.reshape(tuple(coef.shape[:-1]) + (self.Uld,))

    def _expand(self, mw, x=None, lev_scale=None, nlev=1, alpha=0.0, beta=1.0, rsq=True):
        rows = mw.shape[0]
        ld = self.N + (self.N & 1)
        out = torch.empty((rows, ld), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.temd_dedup_expand(_ptr(x), x.stride(0) if x is not None else 0, _ptr(lev_scale), nlev, _ptr(mw),
                                            mw.stride(0), _ptr(self._gid), _ptr(self._rsq) if rsq else None, alpha, beta,
                                            _ptr(out), ld, rows, self.N, self.stream)
        _lib.check(rc, 'temd_dedup_expand')
        return out[:, :self.N]

    # ---- Engine surface ----
    def project(self, fields, lev_scale=None, scale_field=-1, nlev=1):
        out = []
        for i in range(0, len(fields), 4):
            gs = self.group_sums(fields[i:i + 4], lev_scale, scale_field - i if i <= scale_field < i + 4 else -1, nlev)
            out.append(self._project_u(gs))
        return out[0] if len(out) == 1 else torch.cat(out, 0)

    def synth_native(self, coef, out=None):
        res = self._expand(self._synth_u(coef.reshape(-1, self.lpad)))
        if out is not None:
            out[:, :self.N] = res
            return out[:, :self.N]
        return res

    def eddy_native(self, x, coef, lev_scale=None, nlev=1):
        self._check_field(x)
        return self._expand(self._synth_u(coef), x, lev_scale, nlev, alpha=1.0, beta=-1.0)

    def _flux(self, gs, c4):
        rows = gs.shape[1]
        mw = self._synth_u(c4)                                   # [4][rows][Uld]
        fl = torch.empty((3, rows, self.Uld), dtype=torch.float64, device=self.device)
        if self.Uld != self.NU:
            fl[:, :, self.NU:].zero_()
        with torch.cuda.device(self.device):
            rc = self.lib.temd_dedup_flux(_ptr(gs), self.Uld, _ptr(mw), self.Uld, _ptr(self._goff), _ptr(self._rsq), rows,
                                          self.NU, _ptr(fl), self.Uld, self.stream)
        _lib.check(rc, 'temd_dedup_flux')
        return self._project_u(fl)

    def tem_coefficients(self, xs, lev_scale, nlev):
        gs = self.group_sums(list(xs[:4]), lev_scale, 2, nlev, with_products=True)      # the ONE pass over the fields
        c4 = self._project_u(gs[_lib.GS_SW:_lib.GS_SW + 4])
        return c4, self._flux(gs, c4)

    def eddy_flux_project(self, u, v, t, w, coef4, lev_scale, nlev):
        gs = self.group_sums([u, v, t, w], lev_scale, 2, nlev, with_products=True)
        return self._flux(gs, coef4)

    def tracer_coefficients(self, qs, xs, c4, lev_scale, nlev):
        rows = xs[0].shape[0]
        out = torch.empty((3 * len(qs), rows, self.lpad), dtype=torch.float64, device=self.device)
        for i, q in enumerate(qs):
            gs = self.group_sums([q, xs[1], xs[2], xs[3]], lev_scale, 2, nlev, with_products=True)
            cq = self._project_u(gs[_lib.GS_SW:_lib.GS_SW + 1])
            out[3 * i] = cq[0]
            out[3 * i + 1:3 * i + 3] = self._flux(gs, torch.cat([cq, c4[1:]], 0))[:2]
        return out

    def export_matrices(self, Y0=True, Y0inv=True, Y0p=True):
        """Dense Y0 (N,L+1), Y0inv (L+1,N), Y0p (M,L+1) of the FULL grid, expanded from the unique grid:
        Y0[i] = Y0_u[u(i)];  pinv(Y0)[:, i] = pinv(Yw)[:, u(i)] / sqrt(n_u)  (Yw = sqrt(n) Y0_u has the same Gram matrix)."""
        Lp = self.L + 1
        o0 = torch.empty((self.NU, Lp), dtype=torch.float64, device=self.device) if Y0 else None
        oi = torch.empty((Lp, self.NU), dtype=torch.float64, device=self.device) if Y0inv else None
        op = torch.empty((self.M, Lp), dtype=torch.float64, device=self.device) if Y0p else None
        with torch.cuda.device(self.device):
            rc = self.lib.temd_basis_export(self._plan, _ptr(o0), _ptr(oi), _ptr(op), self.stream)
        _lib.check(rc, 'temd_basis_export')
        if o0 is not None:
            o0 = self._expand(o0.t().contiguous(), rsq=False).t().contiguous()
        if oi is not None:
            oi = self._expand(oi).contiguous()
        return o0, oi, op
