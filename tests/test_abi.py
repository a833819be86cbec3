"""CPU: the C-ABI library loads and exports every symbol include/temd.h declares; host-side logic."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported(temd_lib):
    from pytemdiags_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'temd.h')).read()
    declared = set(re.findall(r'\b(temd_[a-z_0-9]+)\s*\(', hdr))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(temd_lib, name), name
    assert temd_lib.temd_version() >= 101


def test_epilogue_enum_matches_python():
    from pytemdiags_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'temd.h')).read()
    enum = re.search(r'enum\s*\{(.*?)TEMD_NOUT', hdr, re.S).group(1)
    names = [n.strip().split('=')[0].strip()[len('TEMD_OUT_'):].lower() for n in enum.split(',') if n.strip()]
    assert tuple(names) == _lib.EPILOGUE_OUTPUTS


def test_no_gpu_means_loud_failure():
    # in a child process that sees no CUDA device, so that this also runs on a machine with a GPU
    import subprocess
    import sys
    code = '\n'.join([
        'import sys; sys.path.insert(0, %r)' % ROOT,
        'import numpy as np, pytest, torch',
        'assert not torch.cuda.is_available()',
        'from pytemdiags_b200 import sph_zonal_averager',
        'with pytest.raises(RuntimeError, match="no CPU fallback"):',
        '    sph_zonal_averager(np.linspace(-80, 80, 100), np.arange(-89.5, 90, 1.0), 10)',
    ])
    subprocess.check_call([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))


def test_product_never_imports_oracle():
    import subprocess
    import sys
    code = "import sys; sys.path.insert(0, %r); import pytemdiags_b200, bench; assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules), 'oracle imported'" % ROOT
    subprocess.check_call([sys.executable, '-c', code])


def test_gradient_coefficients_reproduce_numpy():
    from pytemdiags_b200.engine import gradient_coefficients
    rng = np.random.default_rng(1)
    for x in (np.geomspace(1, 1000, 17) * 100, np.deg2rad(np.arange(-89.5, 90, 1.0)), np.arange(7.0) * 0.5):
        f = rng.standard_normal(x.shape[0])
        coef, uni, h = gradient_coefficients(x)
        ref = np.gradient(f, x)
        n = x.shape[0]
        got = np.empty(n)
        got[0] = (f[1] - f[0]) / (h if uni else x[1] - x[0])
        got[-1] = (f[-1] - f[-2]) / (h if uni else x[-1] - x[-2])
        for i in range(1, n - 1):
            got[i] = (f[i + 1] - f[i - 1]) / (2 * h) if uni else coef[0, i] * f[i - 1] + coef[1, i] * f[i] + coef[2, i] * f[i + 1]
        assert np.array_equal(got, ref)


def test_synthetic_grids():
    from pytemdiags_b200 import synthetic as syn
    lat, lon = syn.pg2_grid(30)
    assert lat.shape == (21600,) and abs(lat).max() < 90 and np.isclose(lat.mean(), 0, atol=1e-12)
    lat, lon = syn.latlon_grid(721, 1440)
    assert lat.shape == (1038240,) and lat[0] == -90 and lat[1440] == -89.75 and lon[1] == 0.25
    a = syn.hash_noise(3, 1, 5, 4, 100)
    assert np.array_equal(a, syn.hash_noise(3, 1, 5, 4, 100)) and abs(a.mean()) < 0.2 and abs(a.std() - 1) < 0.1
