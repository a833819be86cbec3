"""GPU: the time-sharded driver.  One NCCL rank in-process (torch.distributed and libtemd's own NCCL call); with >= 2
visible GPUs also `tools/sharded_check.py` under torchrun (uneven and empty slabs, both transports, tracers).  The
2-rank host logic is covered on CPU with gloo (tests/test_distributed_cpu.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    import socket
    with socket.socket() as sk:
        sk.bind(('127.0.0.1', 0))
        return sk.getsockname()[1]


def test_sharded_tem_single_rank_nccl():
    import torch
    import torch.distributed as dist
    from pytemdiags_b200 import TEMDiagnostics, synthetic as syn
    from pytemdiags_b200.distributed import PUBLIC_OUTPUTS, ShardedTEM, TemdComm, shard_bounds
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(_free_port())
    created = False
    if not dist.is_initialized():
        dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device('cuda:0'))
        created = True
    try:
        lat, lon = syn.pg2_grid(6)
        K, T, L = 6, 5, 20
        plev = syn.default_plev(K)
        f = syn.synth_fields(lat, lon, plev, T, seed=21)
        a, b = shard_bounds(T, 1)[0]
        kw = dict(L=L, dims=('time', 'lev', 'ncol'), debug_level=0)
        full = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, **kw)
        comm = TemdComm(1, 0, TemdComm.unique_id(), 'cuda:0')       # NCCL called from inside libtemd.so
        for c in (None, comm):
            sh = ShardedTEM(f['ua'][a:b], f['va'][a:b], f['ta'][a:b], f['wap'][a:b], plev, lat, T=T, comm=c, **kw)
            out = sh.gather_all()
            for n in PUBLIC_OUTPUTS:
                got = out[n].cpu().numpy()
                assert got.shape == (180, K, T)
                assert np.array_equal(got, getattr(full, n)()), n
            assert np.array_equal(sh.gather('vtem').cpu().numpy(), full.vtem())
        comm.close()
    finally:
        if created:
            dist.destroy_process_group()


def test_sharded_tem_two_gpus_torchrun():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs >= 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', str(_free_port()), os.path.join(ROOT, 'tools', 'sharded_check.py'), '--empty']
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'ALL 2 RANKS OK: True' in r.stdout, r.stdout                      # all-reduced verdict of every rank and case
    assert 'sharded == unsharded: False' not in r.stdout


def test_device_kwarg_other_than_current_device():
    """ADVICE r1: `device=` must work when it differs from the current CUDA device, and must not change it."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    from pytemdiags_b200 import TEMDiagnostics, sph_zonal_averager, synthetic as syn
    torch.cuda.set_device(0)
    lat, lon = syn.pg2_grid(5)
    K, T, L = 5, 2, 12
    plev = syn.default_plev(K)
    f = syn.synth_fields(lat, lon, plev, T, seed=4)
    kw = dict(L=L, dims=('time', 'lev', 'ncol'), debug_level=0)
    t0 = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, device='cuda:0', **kw)
    t1 = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, device='cuda:1', **kw)
    assert torch.cuda.current_device() == 0
    t1b = TEMDiagnostics(f['ua'], f['va'], f['ta'], f['wap'], plev, lat, device='cuda:1', **kw)   # cached engine reused
    assert torch.cuda.current_device() == 0
    for n in ('vtem', 'epfy', 'epdiv'):
        assert np.array_equal(getattr(t0, n)(), getattr(t1, n)())
        assert np.array_equal(getattr(t0, n)(), getattr(t1b, n)())
    zm = sph_zonal_averager(lat, np.arange(-89.5, 90, 1.0), L, device='cuda:1')
    zm.sph_compute_matrices()
    x = f['ua'][0].T.copy()          # (ncol, lev)
    bad = x.copy()
    bad[3, 1] = np.nan
    with pytest.raises(RuntimeError, match='nans'):
        zm.sph_zonal_mean(bad)
    assert zm.sph_zonal_mean(x).shape == (180, K)
    assert torch.cuda.current_device() == 0
    del t1, t1b, zm
    import gc
    gc.collect()                      # plan destruction must not move the current device either
    assert torch.cuda.current_device() == 0
