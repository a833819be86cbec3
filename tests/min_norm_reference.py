"""Float64 NumPy reference of the minimum-norm zonal mean (`min_norm=True`), for the tests.

The result the feature promises is NumPy's minimum-norm least-squares solution, `np.linalg.lstsq(Y0, I, rcond=None)`:
Y0inv = pinv(Y0) with singular values sigma_i <= eps * max(N, L+1) * sigma_1 dropped.  SciPy's default cutoff
(eps * sigma_1, what the reference's `scipy.linalg.lstsq` uses) keeps rounding noise on rank-deficient grids, so
no implementation can match it and it is not the yardstick here.

For grids too large for an N x N identity the same matrix comes from the SVD of the weighted unique-node basis
Yw = diag(sqrt(n)) Y0(x_unique), which has the Gram matrix of Y0 and hence its singular values and right singular
vectors: pinv(Y0)[:, i] = pinv(Yw)[:, u(i)] / sqrt(n_u).
"""
import numpy as np

import oracle

EPS = np.finfo(np.float64).eps


def unique_nodes(lat):
    """x = cos(colatitude) exactly as the reference computes it, and its distinct values."""
    x = np.cos(np.deg2rad(90 - np.asarray(lat, dtype=np.float64)))
    xu, inv, cnt = np.unique(x, return_inverse=True, return_counts=True)
    return x, xu, inv, cnt


def weighted_spectrum(lat, L):
    """Singular values of Yw (= those of Y0) in decreasing order, NumPy's cutoff and rank."""
    _, xu, _, cnt = unique_nodes(lat)
    yw = np.sqrt(cnt)[:, None] * oracle.sph_basis_recurrence(xu, L)
    s = np.linalg.svd(yw, compute_uv=False)
    cutoff = EPS * max(len(lat), L + 1) * s[0]
    return s, cutoff, int(np.sum(s > cutoff))


def sph_matrices_lstsq_numpy(lat, lat_out, L, method='auto'):
    """Y0 (N, L+1), Y0inv (L+1, N), Y0p (M, L+1) and the rank, with Y0inv = np.linalg.lstsq(Y0, I, rcond=None)[0].

    method 'lstsq' is that call literally (an N x N identity); 'svd' is its SVD-of-Yw equivalent; 'auto' picks lstsq
    for N <= 3000."""
    lat = np.asarray(lat, dtype=np.float64)
    x, xu, inv, cnt = unique_nodes(lat)
    Y0 = oracle.sph_basis_recurrence(x, L)
    Y0p = oracle.sph_basis_recurrence(np.cos(np.deg2rad(90 - np.asarray(lat_out, dtype=np.float64))), L)
    if method == 'auto':
        method = 'lstsq' if lat.shape[0] <= 3000 else 'svd'
    if method == 'lstsq':
        Y0inv, _, rank, _ = np.linalg.lstsq(Y0, np.identity(lat.shape[0]), rcond=None)
        return Y0, Y0inv, Y0p, int(rank)
    if method != 'svd':
        raise ValueError(method)
    sq = np.sqrt(cnt.astype(np.float64))
    yw = sq[:, None] * oracle.sph_basis_recurrence(xu, L)
    u, s, vt = np.linalg.svd(yw, full_matrices=False)
    r = int(np.sum(s > EPS * max(lat.shape[0], L + 1) * s[0]))
    pinv_w = (vt[:r].T / s[:r]) @ u[:, :r].T               # (L+1, U)
    Y0inv = pinv_w[:, inv] / sq[inv]
    return Y0, Y0inv, Y0p, r


def latitude_means(lat, A):
    """Closed form on grids whose distinct x nodes are all kept: the per-node arithmetic mean of A (N, ...),
    expanded back to every column."""
    _, _, inv, cnt = unique_nodes(lat)
    A2 = np.asarray(A, dtype=np.float64).reshape(len(lat), -1)
    sums = np.zeros((cnt.shape[0], A2.shape[1]))
    np.add.at(sums, inv, A2)
    return (sums / cnt[:, None])[inv].reshape(np.shape(A))


def legendre_interpolant(lat, lat_out, L, A):
    """Closed form of the output-grid mean when all U distinct nodes are kept (U <= L+1): the minimum-norm Legendre
    coefficients c = pinv(Y_U) m of the per-node means m, evaluated on lat_out."""
    _, xu, inv, cnt = unique_nodes(lat)
    A2 = np.asarray(A, dtype=np.float64).reshape(len(lat), -1)
    sums = np.zeros((cnt.shape[0], A2.shape[1]))
    np.add.at(sums, inv, A2)
    m = sums / cnt[:, None]
    Yu = oracle.sph_basis_recurrence(xu, L)
    c = Yu.T @ np.linalg.solve(Yu @ Yu.T, m)
    Yp = oracle.sph_basis_recurrence(np.cos(np.deg2rad(90 - np.asarray(lat_out, dtype=np.float64))), L)
    return (Yp @ c).reshape((len(lat_out),) + np.shape(A)[1:])


def latlon_plus_row(nlat=72, nlon=144, row=30, dlat=1e-13):
    """Lat-lon grid without poles plus one extra row of nlon columns at lat[row] + dlat degrees: U = nlat + 1 distinct
    nodes, one of them 1e-13 degrees from its neighbour, so Y0 has numerical rank nlat."""
    from pytemdiags_b200 import synthetic as syn
    lat, lon = syn.latlon_grid(nlat, nlon, poles=False)
    lat1 = np.unique(lat)
    return np.concatenate([lat, np.full(nlon, lat1[row] + dlat)]), np.concatenate([lon, lon[:nlon]])
