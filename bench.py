#!/usr/bin/env python
"""Benchmark of the TEM-suite hot path (BASELINE.json metric: column.level.steps/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config config2] [--dump-outputs DIR]

Headline (`value`, `ms_per_step`, `roofline`, `e2e`): one "step" = the full TEM suite (project -> fused
eddy/flux/project -> output-grid synthesis -> stencil epilogue) over ONE 73-step time slab of config 2 with the four
input fields already resident in HBM; `e2e` is the same thing through the public API with pinned HOST arrays
(`TEMDiagnostics(ua, va, ta, wap, p, lat)` at N = 1, `ShardedTEM(...).gather_all()` at N > 1, H2D + D2H inside the
timed region) next to a barrier-synchronised concurrent pinned-H2D ceiling of the box.  With N > 1 (torchrun) every
rank owns its own time slab (weak scaling, no collective on the data path) and the ten public outputs are gathered with
ONE NCCL all-gather per step.

Extra blocks in the same JSON line (`records`), each a whole BASELINE record time-sharded over the N ranks
(STRONG scaling; slabs generated on the device, kernels timed with CUDA events, max over ranks, final gather included):
  config3  ne256pg2 x 128 lev x 96 steps, L=200 (the north-star record)
  config4  0.25-degree lat-lon x 37 lev x 240 steps, L=300: dense path and the de-duplicated fast path (`dedup=True`)
  config2_dedup  the 365-step ne120pg2 record through the de-duplicated path (scattered groups of <= 8 columns)
  config5  zonal-mean-only sweep L in {25..800} on ne120pg2 x 72 lev x 24 steps (N = 1 only)
Each carries its roofline fractions and a spot check of one time step against tests/golden/scale_*.npz.

`--impl reference` times the reference's CPU algorithm (the NumPy oracle port, factored form: the literal N x N operator
of sph_zonal_mean.py:251 needs 956 GB at this grid) on a bounded sample.

`--steps K` is the number of timed headline steps and of timed public-API calls in `e2e`.  `--dump-outputs DIR` writes
what the last timed headline step computed (rank 0's slab) as DIR/<name>.npy, float64: every epilogue plane, on a fixed
seeded sample of the slab's time steps that keeps the files within 64 MB.  The inputs are generated from a fixed seed,
so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

if '--impl' in sys.argv and 'reference' in sys.argv:
    # the reference arm uses every host core (torchrun exports OMP_NUM_THREADS=1 for its workers)
    for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_v] = str(os.cpu_count())

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'tem_suite_column_level_steps_per_s'
UNIT = 'col*lev*steps/s'
FP64_PEAK_TFLOPS = 37.1   # measured DMMA m8n8k4 issue-rate peak on this pool (profiles/r01_microbench_fp64.log)
PUBLIC = ('vtem', 'omegatem', 'wtem', 'psitem', 'epfy', 'epfz', 'epdiv', 'utendepfd', 'utendvtem', 'utendwtem')
# (seed, time step) of the committed one-step expectations, tests/golden/make_scale_golden.py
FIXTURES = {'config2': ('scale_config2_t1', 1, 182), 'config3': ('scale_config3_t1', 2, 48), 'config4': ('scale_config4_t1', 3, 120)}
DUMP_BYTES = 64 * 10 ** 6       # cap on what --dump-outputs writes


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.max_mhz = None
        self.reasons = set()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {'hw_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwSlowdown', 0x8),
                 'hw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwThermalSlowdown', 0x40),
                 'sw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonSwThermalSlowdown', 0x20),
                 'sw_power_cap': getattr(nv, 'nvmlClocksThrottleReasonSwPowerCap', 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': ['unavailable']}
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def workload(name):
    from pytemdiags_b200 import synthetic as syn
    cfg = dict(syn.CONFIGS[name])
    L = cfg['L'] if not isinstance(cfg['L'], tuple) else cfg['L'][2]
    return cfg, L


def cpu_suite_sample(cfg, L, tsample, seed=0, repeat=1):
    """Times the oracle port (factored form) on `tsample` time steps of the workload.  Returns
    (points per second, seconds per suite, setup seconds, threads)."""
    import oracle
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass
    from pytemdiags_b200 import synthetic as syn
    lat, lon = syn.make_grid(cfg['grid'])
    plev = syn.default_plev(cfg['K'])
    t0 = time.time()
    mats = oracle.sph_matrices(lat, oracle.zm_latitudes(1), L, method='pinv')
    setup = time.time() - t0
    f = syn.synth_fields(lat, lon, plev, tsample, seed=seed)
    tr = lambda x: np.ascontiguousarray(x.transpose(2, 1, 0))
    args = [tr(f[n]) for n in ('ua', 'va', 'ta', 'wap')]
    best = None
    for _ in range(repeat):
        t0 = time.time()
        oracle.tem_suite(*args, plev, lat, L=L, literal=False, matrices=mats)
        dt = time.time() - t0
        best = dt if best is None else min(best, dt)
    pts = lat.shape[0] * cfg['K'] * tsample
    return pts / best, best, setup, os.cpu_count()


def run_reference(args):
    """The reference arm: NumPy oracle port of the reference algorithm on the host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cfg, L = workload(args.config)
    tsample = args.cpu_tsample
    import oracle
    from pytemdiags_b200 import synthetic as syn
    lat, lon = syn.make_grid(cfg['grid'])
    plev = syn.default_plev(cfg['K'])
    mats = oracle.sph_matrices(lat, oracle.zm_latitudes(1), L, method='pinv')
    f = syn.synth_fields(lat, lon, plev, tsample, seed=0)
    tr = lambda x: np.ascontiguousarray(x.transpose(2, 1, 0))
    a = [tr(f[n]) for n in ('ua', 'va', 'ta', 'wap')]
    for _ in range(args.warmup):
        oracle.tem_suite(*a, plev, lat, L=L, literal=False, matrices=mats)
    t0 = time.time()
    for _ in range(args.steps):
        oracle.tem_suite(*a, plev, lat, L=L, literal=False, matrices=mats)
    dt = (time.time() - t0) / args.steps
    pts = lat.shape[0] * cfg['K'] * tsample
    val = pts / dt
    sample = '%d of %d time steps per step of %s (factored NumPy oracle; literal N x N operator infeasible)' % (
        tsample, cfg['T'], args.config)
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': '%s: %s, K=%d, L=%d, %d-step sample' % (args.config, cfg['grid'], cfg['K'], L, tsample)},
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': 'port', 'sample': sample},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


# ----------------------------------------------------------------------------------------------------------------------
class Ctx:
    """Per-process context: rank / device / collectives."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(self.local)
        self.dev = torch.device('cuda', self.local)
        self.binding = bind_near_gpu(self.local) if self.world > 1 else None
        if self.world > 1:
            dist.init_process_group('nccl', device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def table(self, v):
        """every rank's value, in rank order"""
        if self.world == 1:
            return [float(v)]
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        out = self.torch.empty(self.world, dtype=self.torch.float64, device=self.dev)
        self.dist.all_gather_into_tensor(out, t)
        return [float(x) for x in out.cpu()]


def bind_near_gpu(local):
    """Pin this rank (and therefore the first-touch placement of its pinned buffers) to the CPUs of the NUMA node
    the GPU hangs off, read from sysfs (NVML's affinity mask is the whole machine on the virtualised boxes).
    Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if bus.startswith('00000000:'):
            bus = bus[4:]
        node = -1
        try:
            node = int(open('/sys/bus/pci/devices/%s/numa_node' % bus).read().strip())
        except Exception:
            pass
        nodes = sorted(d for d in os.listdir('/sys/devices/system/node') if d.startswith('node') and d[4:].isdigit())
        if node < 0 or len(nodes) <= 1:
            return {'gpu_pci': bus, 'numa_node': node, 'numa_nodes': len(nodes), 'bound': False,
                    'why': 'single (virtual) NUMA node: nothing to bind to'}
        cpus = open('/sys/devices/system/node/node%d/cpulist' % node).read().strip()
        ids = []
        for part in cpus.split(','):
            lo, _, hi = part.partition('-')
            ids += list(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, ids)
        return {'gpu_pci': bus, 'numa_node': node, 'numa_nodes': len(nodes), 'bound': True, 'cpus': cpus}
    except Exception as e:      # noqa: BLE001
        return {'bound': False, 'why': '%s: %s' % (type(e).__name__, e)}


def nerr(x, ref):
    return float(np.abs(np.asarray(x) - ref).max() / max(float(np.abs(ref).max()), 1e-300))


def spot_check(ctx, cfgname, res_planes, t_first, t_count):
    """Compares ONE time step of the outputs that were just timed (res_planes: name -> [T_local][K][M] device tensors of
    the steps [t_first, t_first + t_count)) with the committed CPU-oracle expectation of that step.  Max over ranks."""
    fname, _, tfix = FIXTURES[cfgname]
    path = os.path.join(ROOT, 'tests', 'golden', fname + '.npz')
    err = -1.0
    if os.path.exists(path) and t_first <= tfix < t_first + t_count:
        g = np.load(path)
        err = 0.0
        for n in PUBLIC:
            got = res_planes[n][tfix - t_first].permute(1, 0).cpu().numpy()       # (M, K)
            err = max(err, nerr(got, g[n][:, :, 0]))
    err = ctx.max(err)
    return {'fixture': 'tests/golden/%s.npz' % fname, 'time_step': tfix, 'outputs': len(PUBLIC), 'tol': 1e-10,
            'max_normwise_err': err if err >= 0 else None, 'ok': bool(0 <= err < 1e-10)}


def dump_outputs(path, res_planes, t_first):
    """Writes res_planes (name -> [T_local][K][M] device tensors of the steps [t_first, t_first + T_local)) as
    path/<name>.npy, float64, keeping a seeded sample of the time steps (the same one for every plane) so that the
    files stay within DUMP_BYTES."""
    import torch
    first = next(iter(res_planes.values()))
    step_bytes = sum(v[0].numel() * 8 for v in res_planes.values())
    keep = min(first.shape[0], DUMP_BYTES // step_bytes)
    assert keep >= 1, 'one time step of the outputs exceeds the --dump-outputs cap'
    idx = np.sort(np.random.default_rng(0).choice(first.shape[0], keep, replace=False))
    sel = torch.as_tensor(idx, device=first.device)
    os.makedirs(path, exist_ok=True)
    for n, v in res_planes.items():
        np.save(os.path.join(path, n + '.npy'), v.index_select(0, sel).to(torch.float64).cpu().numpy())
    return {'dir': path, 'arrays': sorted(res_planes), 'dtype': 'float64', 'time_steps': [t_first + int(i) for i in idx],
            'shape': [keep] + list(first.shape[1:]), 'bytes': keep * step_bytes}


def ev_pair(torch):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


# ----------------------------------------------------------------------------------------------------------------------
def headline(args, ctx):
    """config-2 slab per GPU: value, per-kernel times, roofline, spot check."""
    torch = ctx.torch
    from pytemdiags_b200 import synthetic as syn, constants as const
    from pytemdiags_b200.engine import Engine
    from pytemdiags_b200.distributed import gather_time_major
    cfg, L = workload(args.config)
    K = cfg['K']
    lat, lon = syn.make_grid(cfg['grid'])
    N = lat.shape[0]
    plev = syn.default_plev(K)
    lat_zm = np.arange(-89.5, 90.0, 1.0)
    Ts = args.slab_steps
    fname, seed, tfix = FIXTURES.get(args.config, (None, 0, 0))
    nslabs = max(1, cfg['T'] // Ts)
    t_off = ((ctx.rank + tfix // Ts) % nslabs) * Ts      # rank 0's slab contains the fixture's time step

    eng = Engine(lat, lat_zm, L, device=ctx.dev)
    t0 = time.time()
    eng.build_basis()
    torch.cuda.synchronize()
    basis_s = time.time() - t0

    latr, lonr = eng._dev(np.deg2rad(lat)), eng._dev(np.deg2rad(lon))
    plev_d = eng._dev(plev)
    xs = [eng.synth_fields(fi, seed, t_off, Ts, plev, latr, lonr, plev_d) for fi in range(4)]
    p_pa = plev * 100
    lev_scale = eng._dev((const.P0 / p_pa) ** const.k)
    f_zm = 2 * const.Om * np.sin(lat_zm * np.pi / 180)
    coslat = np.cos(lat_zm * np.pi / 180)
    torch.cuda.synchronize()
    ev = {}

    def timed(name, fn):
        a, b = ev_pair(torch)
        a.record()
        r = fn()
        b.record()
        ev.setdefault(name, []).append((a, b))
        return r

    def step():
        c4 = timed('project', lambda: eng.project(xs, lev_scale=lev_scale, scale_field=2, nlev=K))
        cf = timed('eddy_flux_project', lambda: eng.eddy_flux_project(xs[0], xs[1], xs[2], xs[3], c4, lev_scale, K))
        coef = torch.cat([c4, cf], 0)
        eng.check_finite(coef, 'fields')
        zm = timed('synth_out', lambda: eng.synth_out(coef)).reshape(7, Ts, K, eng.M)
        res = timed('epilogue', lambda: eng.tem_epilogue(zm, p_pa, f_zm, coslat))
        if ctx.world > 1:
            # the product's multi-GPU exchange: ONE all-gather of the ten stacked output planes
            timed('gather', lambda: gather_time_major(torch.stack([res[n] for n in PUBLIC]), Ts * ctx.world))
        return res
    launches_per_step = 2 + 2 + 1 + 1 + EPILOGUE_LAUNCHES   # project+reduce, eddy+reduce, check_finite, synth_out, epilogue

    for _ in range(args.warmup):
        step()
    ev.clear()
    ctx.barrier()
    sampler = ClockSampler(ctx.local)
    sampler.start()
    e0, e1 = ev_pair(torch)
    e0.record()
    for _ in range(args.steps):
        res = step()
    e1.record()
    ctx.barrier()
    clocks = sampler.result()
    ms = ctx.max(e0.elapsed_time(e1) / args.steps)
    value = N * K * Ts * ctx.world / (ms * 1e-3)
    kms = {n: float(np.mean([a.elapsed_time(b) for a, b in v])) for n, v in ev.items()}
    dump = dump_outputs(args.dump_outputs, res, t_off) if args.dump_outputs and ctx.rank == 0 else None
    check = spot_check(ctx, args.config, res, t_off, Ts) if fname else None

    Lp, rows = L + 1, Ts * K
    fl_eddy, fl_proj = 14.0 * Lp * N * rows, 8.0 * Lp * N * rows
    roof = {'bound': 'tensor', 'kernel': 'k_eddy (temd_eddy_flux_project)',
            'achieved': fl_eddy / (kms['eddy_flux_project'] * 1e-3) / 1e12, 'peak': FP64_PEAK_TFLOPS, 'unit': 'TFLOP/s',
            'traffic': None,
            'peak_source': 'FP64 is not in MEASURED_PEAKS.json; 37.1 TFLOP/s = DMMA.8x8x4 issue-rate peak measured on '
                           'this pool (profiles/r01_microbench_fp64.log), nominal 148 SM x 64 FMA/clk x 1.965 GHz = 37.2',
            'algorithmic_flops_per_launch': fl_eddy}
    roof['frac'] = roof['achieved'] / roof['peak']
    try:
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get('%s:%d' % (args.config, Ts))
        if tr:
            roof['traffic'] = tr['k_eddy']['dram_bytes']
            roof['traffic_unit'] = 'bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/traffic.json)'
            roof['algorithmic_bytes_per_launch'] = 32.0 * N * rows
    except Exception:
        pass
    roof_proj = {'bound': 'tensor', 'kernel': 'k_project (temd_project)',
                 'achieved': fl_proj / (kms['project'] * 1e-3) / 1e12, 'peak': FP64_PEAK_TFLOPS, 'unit': 'TFLOP/s'}
    roof_proj['frac'] = roof_proj['achieved'] / roof_proj['peak']
    out = dict(cfg=cfg, L=L, N=N, K=K, Ts=Ts, ms=ms, value=value, kms=kms, clocks=clocks, basis_s=basis_s, roof=roof,
               roof_proj=roof_proj, spot_check=check, launches_per_step=launches_per_step, dump=dump,
               step_tf=22.0 * Lp * N * rows / (ms * 1e-3) / 1e12,
               hbm={'bytes_per_point': 64, 'achieved_gbs': 64.0 * N * rows / (ms * 1e-3) / 1e9, 'peak_gbs': peaks().get('hbm_gbs')})
    return out, eng, xs, plev, lat


EPILOGUE_LAUNCHES = 2     # k_epi_1, k_epi_2


def h2d_ceiling(ctx, nbytes):
    """Pinned host->device copy bandwidth of this box: every rank alone in turn (`solo`), then all ranks at once after
    a barrier (`concurrent`), per GPU.  The concurrent aggregate / 32 B per point is the ceiling of the e2e metric."""
    torch = ctx.torch
    n = nbytes // 8
    h = torch.empty(n, dtype=torch.float64).pin_memory()
    h.zero_()
    d = torch.empty(n, dtype=torch.float64, device=ctx.dev)

    def one(reps=3):
        a, b = ev_pair(torch)
        a.record()
        for _ in range(reps):
            d.copy_(h, non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        return reps * nbytes / (a.elapsed_time(b) * 1e-3) / 1e9
    one(1)
    solo = 0.0
    for r in range(ctx.world):
        ctx.barrier()
        if r == ctx.rank:
            solo = one()
    ctx.barrier()
    conc = one()
    ctx.barrier()
    solo_t, conc_t = ctx.table(solo), ctx.table(conc)
    del h, d
    return {'bytes_per_copy': nbytes, 'solo_gbs_per_gpu': [round(x, 2) for x in solo_t],
            'concurrent_gbs_per_gpu': [round(x, 2) for x in conc_t], 'concurrent_aggregate_gbs': round(sum(conc_t), 2),
            'how': 'cudaMemcpyAsync from cudaHostAlloc memory, 3 copies, CUDA events; solo = one rank at a time, '
                   'concurrent = all ranks after a barrier'}


def e2e_leg(args, ctx, head, xs, plev, lat):
    """The public API on pinned HOST arrays, H2D + D2H inside the timed region.  N = 1: TEMDiagnostics; N > 1:
    ShardedTEM (each rank uploads its slab) + gather_all() (one collective) + D2H of the gathered outputs.  At N > 1
    the record of e2e_steps x N time steps is sharded twice: equally, and in proportion to the host->device bandwidth
    each GPU gets when all ranks copy at once (`ShardedTEM(weights=...)`): on this pool's 8-GPU boxes GPUs 0-3 get
    23 GB/s and GPUs 4-7 35 GB/s, so an equal split waits for the slow links."""
    torch = ctx.torch
    from pytemdiags_b200 import TEMDiagnostics
    from pytemdiags_b200.distributed import ShardedTEM, shard_bounds
    N, K, L, Te = head['N'], head['K'], head['L'], args.e2e_steps
    M = 180
    kw = dict(L=L, dims=('time', 'lev', 'ncol'), debug_level=0, device=ctx.dev)
    ceiling = h2d_ceiling(ctx, min(4 * Te * K * N * 8 // 4, 2 << 30))
    Ttot = Te * ctx.world

    def measure(weights):
        a_, b_ = shard_bounds(Ttot, ctx.world, weights)[ctx.rank]
        nloc = b_ - a_
        assert nloc * K <= xs[0].shape[0], 'e2e slab larger than the resident slab'
        host = []
        for fi in range(4):
            h = torch.empty((nloc, K, N), dtype=torch.float64).pin_memory()
            h.copy_(xs[fi][:nloc * K].reshape(nloc, K, N))
            host.append(h.numpy())
        torch.cuda.synchronize()
        local_s = []
        if ctx.world == 1:
            def call():
                tem = TEMDiagnostics(host[0], host[1], host[2], host[3], plev, lat, **kw)
                return [getattr(tem, n)() for n in PUBLIC]
        else:
            back = torch.empty((len(PUBLIC), Ttot, K, M), dtype=torch.float64).pin_memory()

            def call():
                sh = ShardedTEM(host[0], host[1], host[2], host[3], plev, lat, T=Ttot, weights=weights, **kw)
                local_s.append(sh.local_seconds)
                full, _ = sh.gather_all(PUBLIC, tracers=False, layout='stacked')
                back.copy_(full, non_blocking=True)          # ONE device->host copy of the ten gathered outputs
                torch.cuda.synchronize()
                return back
        for _ in range(2):
            call()
        ctx.barrier()
        nrep = args.steps
        a, b = ev_pair(torch)
        calls = []
        a.record()
        for _ in range(nrep):
            tc = time.time()
            call()
            torch.cuda.synchronize()
            calls.append(time.time() - tc)
        b.record()
        ctx.barrier()
        dt = ctx.max(a.elapsed_time(b) * 1e-3 / nrep)
        if os.environ.get('TEMD_BENCH_DEBUG'):
            print('e2e per-call ms:', [round(c * 1e3, 1) for c in calls], file=sys.stderr)
        del host
        # steps per second of each rank's own upload + compute (before the gather), for a refined split
        rates = ctx.table(nloc / max(float(np.median(local_s[-nrep:])), 1e-9)) if ctx.world > 1 else None
        return dt, [y - x for x, y in shard_bounds(Ttot, ctx.world, weights)], rates

    dt, steps, rates0 = measure(None)
    h2d = 4 * Ttot * K * N * 8                     # bytes all ranks upload per call
    d2h = 10 * M * K * Ttot * 8 * ctx.world        # every rank reads the gathered outputs back
    bound = ceiling['concurrent_aggregate_gbs'] * 1e9 / 32.0
    out = {'value': N * K * Ttot / dt, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
           'time_steps_per_call': Ttot, 'time_steps_per_gpu': steps, 'ms_per_call': dt * 1e3,
           'h2d_gbs_achieved_aggregate': h2d / dt / 1e9, 'h2d_ceiling': ceiling,
           'ceiling_value': bound, 'frac_of_h2d_ceiling': N * K * Ttot / dt / bound, 'cpu_binding': ctx.binding,
           'api': 'TEMDiagnostics(ua, va, ta, wap, p, lat)' if ctx.world == 1 else
                  'ShardedTEM(ua, va, ta, wap, p, lat, T=..., weights=...).gather_all()  (one NCCL all-gather of the 10 outputs)',
           'note': 'pinned host arrays; H2D of slab i+1 overlaps compute of slab i; basis cached across calls like the '
                   'reference\'s maps/ cache; the metric is bound by host->device bandwidth (32 B per point): ceiling_value = '
                   'concurrent aggregate H2D GB/s / 32 B'}
    if ctx.world > 1:
        equal = {'value': out['value'], 'ms_per_call': out['ms_per_call'], 'time_steps_per_gpu': steps,
                 'frac_of_h2d_ceiling': out['frac_of_h2d_ceiling'],
                 'frac_of_slowest_link_ceiling': N * K * Ttot / dt / (ctx.world * min(ceiling['concurrent_gbs_per_gpu']) * 1e9 / 32.0)}
        w = ceiling['concurrent_gbs_per_gpu']
        out['sharding'] = 'equal'
        if max(w) / min(w) > 1.1:       # heterogeneous host links: slabs proportional to the measured bandwidth
            dtw, stepsw, rates1 = measure(w)
            weighted = {'value': N * K * Ttot / dtw, 'ms_per_call': dtw * 1e3, 'time_steps_per_gpu': stepsw,
                        'frac_of_h2d_ceiling': N * K * Ttot / dtw / bound, 'weights': [round(x, 2) for x in w],
                        'weights_from': 'concurrent pinned-H2D GB/s per GPU (h2d_ceiling)'}
            # one refinement: weights = the steps/s every rank actually sustained in that run (upload + kernels)
            dtr, stepsr, _ = measure(rates1)
            refined = {'value': N * K * Ttot / dtr, 'ms_per_call': dtr * 1e3, 'time_steps_per_gpu': stepsr,
                       'frac_of_h2d_ceiling': N * K * Ttot / dtr / bound, 'weights': [round(x, 2) for x in rates1],
                       'weights_from': 'steps/s of each rank (ShardedTEM.local_steps / local_seconds) in the weighted run'}
            out['equal_split'], out['weighted_split'], out['refined_split'] = equal, weighted, refined
            best = max((weighted, refined), key=lambda r: r['value'])
            if best['value'] > out['value']:
                out.update(value=best['value'], ms_per_call=best['ms_per_call'], time_steps_per_gpu=best['time_steps_per_gpu'],
                           frac_of_h2d_ceiling=best['frac_of_h2d_ceiling'],
                           h2d_gbs_achieved_aggregate=h2d / (best['ms_per_call'] * 1e-3) / 1e9,
                           sharding='time slabs weighted by ' + best['weights_from'])
        else:
            out['equal_split'] = equal
    return out


# ----------------------------------------------------------------------------------------------------------------------
def run_record(ctx, cfgname, sub_steps, dedup=False):
    """One whole BASELINE record, time-sharded over the ranks (strong scaling): slabs are generated on the device
    (untimed), the suite kernels are timed with CUDA events slab by slab, the tail (output-grid synthesis, stencil
    epilogue, final all-gather of the ten outputs) once; total = max over ranks."""
    torch = ctx.torch
    from pytemdiags_b200 import synthetic as syn, constants as const
    from pytemdiags_b200.engine import DedupEngine, Engine
    from pytemdiags_b200.distributed import gather_time_major, shard_bounds
    cfg, L = workload(cfgname)
    K, T = cfg['K'], cfg['T']
    lat, lon = syn.make_grid(cfg['grid'])
    N = lat.shape[0]
    plev = syn.default_plev(K)
    lat_zm = np.arange(-89.5, 90.0, 1.0)
    fname, seed, tfix = FIXTURES[cfgname]
    a, b = shard_bounds(T, ctx.world)[ctx.rank]
    eng = (DedupEngine if dedup else Engine)(lat, lat_zm, L, device=ctx.dev)
    t0 = time.time()
    eng.build_basis()
    torch.cuda.synchronize()
    basis_s = time.time() - t0
    latr, lonr, plev_d = eng._dev(np.deg2rad(lat)), eng._dev(np.deg2rad(lon)), eng._dev(plev)
    p_pa = plev * 100
    lev_scale = eng._dev((const.P0 / p_pa) ** const.k)
    f_zm = 2 * const.Om * np.sin(lat_zm * np.pi / 180)
    coslat = np.cos(lat_zm * np.pi / 180)
    ld = N + (N & 1)
    bufs = [torch.empty((sub_steps * K, ld), dtype=torch.float64, device=ctx.dev) for _ in range(4)]
    coef = torch.zeros((7, (b - a) * K, eng.lpad), dtype=torch.float64, device=ctx.dev)
    ev = {}

    def timed(name, fn):
        e0, e1 = ev_pair(torch)
        e0.record()
        r = fn()
        e1.record()
        ev.setdefault(name, []).append((e0, e1))
        return r

    def slab(s0, s1):
        xs = [eng.synth_fields(fi, seed, s0, s1 - s0, plev, latr, lonr, plev_d, out=bufs[fi][:(s1 - s0) * K]) for fi in range(4)]
        r0, r1 = (s0 - a) * K, (s1 - a) * K
        if dedup:
            gs = timed('group_sums', lambda: eng.group_sums(xs, lev_scale, 2, K, with_products=True))
            c4 = timed('project_u', lambda: eng._project_u(gs[11:15]))
            cf = timed('flux_u', lambda: eng._flux(gs, c4))
        else:
            c4 = timed('project', lambda: eng.project(xs, lev_scale=lev_scale, scale_field=2, nlev=K))
            cf = timed('eddy_flux_project', lambda: eng.eddy_flux_project(xs[0], xs[1], xs[2], xs[3], c4, lev_scale, K))
        coef[:4, r0:r1] = c4
        coef[4:, r0:r1] = cf

    host_ms = {}

    def tail():
        h0 = time.time()
        timed('tail_check_finite', lambda: eng.check_finite(coef, 'fields'))
        h1 = time.time()
        zm = timed('tail_synth_out', lambda: eng.synth_out(coef)).reshape(7, b - a, K, eng.M)
        h2 = time.time()
        res = timed('tail_epilogue', lambda: eng.tem_epilogue(zm, p_pa, f_zm, coslat))
        h3 = time.time()
        full = timed('tail_gather', lambda: gather_time_major(torch.stack([res[n] for n in PUBLIC]), T)) if ctx.world > 1 else None
        host_ms.update(check_finite=(h1 - h0) * 1e3, synth_out=(h2 - h1) * 1e3, epilogue=(h3 - h2) * 1e3,
                       gather=(time.time() - h3) * 1e3)
        return res, full

    starts = list(range(a, b, sub_steps))
    if starts:                       # warm-up: first slab + tail (allocations, attribute calls, NCCL channel set-up)
        slab(starts[0], min(b, starts[0] + sub_steps))
    tail()
    tail()       # twice: the engine keeps the last epilogue planes alive, so only the third call finds a cached block
                 # (a fresh cudaMalloc of ~100 MB costs tens of ms once NCCL has enabled peer access)
    ev.clear()
    ctx.barrier()
    for s0 in starts:
        slab(s0, min(b, s0 + sub_steps))
    res, full = timed('tail', tail)
    ctx.barrier()
    kms = {n: float(np.sum([x.elapsed_time(y) for x, y in v])) for n, v in ev.items()}
    local_ms = sum(v for n, v in kms.items() if not n.startswith('tail_'))
    total_ms = ctx.max(local_ms)
    kmax = {n: ctx.max(v) for n, v in sorted(kms.items())}
    check = spot_check(ctx, cfgname, res, a, b - a)
    pts = float(N) * K * T
    Lp = L + 1
    out = {'workload': '%s: %s (%d cols) x %d lev x %d steps, L=%d, %s' % (cfgname, cfg['grid'], N, K, T, L,
                                                                         'dedup fast path' if dedup else 'dense path'),
           'scaling': 'strong', 'time_steps_per_gpu': [y - x for x, y in shard_bounds(T, ctx.world)], 'sub_slab_steps': sub_steps,
           'record_ms': total_ms, 'value': pts / (total_ms * 1e-3), 'unit': UNIT, 'kernel_ms_max_over_ranks': kmax,
           'basis_build_s': basis_s, 'spot_check': check, 'tail_host_ms': {k_: round(v, 3) for k_, v in host_ms.items()},
           'timing': 'CUDA events around every suite launch of every slab + the tail (synth_out, epilogue, all-gather); '
                     'on-device slab generation between slabs is not timed; max over ranks'}
    if dedup:
        g_ms = kmax['group_sums']
        gb = 32.0 * pts / ctx.world                      # bytes one rank's group-sum launches read
        hb = peaks().get('hbm_gbs') or 6522.7
        out['unique_latitudes'] = eng.NU
        out['roofline'] = {'bound': 'hbm', 'kernel': 'k_gsum_warp / k_gsum_thread (temd_group_sums)',
                           'achieved': gb / (g_ms * 1e-3) / 1e9, 'peak': hb, 'unit': 'GB/s',
                           'algorithmic_bytes': '32 B per col.lev.step (four float64 fields read once)'}
        out['roofline']['frac'] = out['roofline']['achieved'] / hb
        try:
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get('%s:%d:dedup' % (cfgname, sub_steps))
            if tr:      # ncu dram bytes of ONE launch over one sub-slab, next to its algorithmic bytes
                out['roofline']['traffic'] = tr['k_gsum_warp']['dram_bytes']
                out['roofline']['algorithmic_bytes_per_launch'] = tr['k_gsum_warp']['algorithmic_bytes']
        except Exception:
            pass
        out['suite_hbm'] = {'achieved_gbs': gb / (total_ms * 1e-3) / 1e9, 'frac': gb / (total_ms * 1e-3) / 1e9 / hb,
                            'note': 'whole suite incl. the tensor-core kernels on the unique grid and the tail'}
    else:
        per_gpu = pts / ctx.world
        for key, name, fl in (('eddy_flux_project', 'k_eddy', 14.0), ('project', 'k_project', 8.0)):
            tf = fl * Lp * per_gpu / (kmax[key] * 1e-3) / 1e12
            out['roofline_' + name] = {'bound': 'tensor', 'achieved': tf, 'peak': FP64_PEAK_TFLOPS, 'unit': 'TFLOP/s',
                                       'frac': tf / FP64_PEAK_TFLOPS}
        tf = 22.0 * Lp * per_gpu / (total_ms * 1e-3) / 1e12
        out['suite_fp64'] = {'achieved_tflops_per_gpu': tf, 'frac': tf / FP64_PEAK_TFLOPS}
    del bufs, coef, eng
    torch.cuda.empty_cache()
    return out


def run_sweep(ctx):
    """config 5: zonal-mean-only sweep on ne120pg2 x 72 lev x 24 steps (N = 1)."""
    torch = ctx.torch
    from pytemdiags_b200 import synthetic as syn
    from pytemdiags_b200.engine import Engine
    lat, lon = syn.pg2_grid(120)
    N, K, T = lat.shape[0], 72, 24
    rows = K * T
    lat_out = np.arange(-89.5, 90, 1.0)
    hbm = peaks().get('hbm_gbs') or 6522.7
    out, x = [], None

    def timeit(fn, reps=5):
        for _ in range(2):
            fn()
        a, b = ev_pair(torch)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    for L in (25, 50, 100, 200, 400, 800):
        eng = Engine(lat, lat_out, L, device=ctx.dev)
        t0 = time.time()
        eng.build_basis()
        torch.cuda.synchronize()
        tb = time.time() - t0
        if x is None:
            pl = syn.default_plev(K)
            x = eng.synth_fields(0, 4, 0, T, pl, eng._dev(np.deg2rad(lat)), eng._dev(np.deg2rad(lon)), eng._dev(pl))
        Lp, pts = L + 1, float(N) * rows
        coef = eng.project([x])
        nat = torch.empty((rows, N), dtype=torch.float64, device=ctx.dev)
        tp = timeit(lambda: eng.project([x]))
        to = timeit(lambda: eng.synth_out(coef))
        tn = timeit(lambda: eng.synth_native(coef[0], out=nat))
        r = {'L': L, 'basis_build_ms': tb * 1e3, 'project_ms': tp, 'synth_out_ms': to, 'synth_native_ms': tn,
             'project_tflops': 2.0 * Lp * pts / tp / 1e9, 'synth_native_tflops': 2.0 * Lp * pts / tn / 1e9,
             'project_read_gbs': 8.0 * pts / tp / 1e6, 'synth_native_write_gbs': 8.0 * pts / tn / 1e6}
        r['project_frac_fp64'] = r['project_tflops'] / FP64_PEAK_TFLOPS
        r['synth_native_frac_fp64'] = r['synth_native_tflops'] / FP64_PEAK_TFLOPS
        r['project_frac_hbm'] = r['project_read_gbs'] / hbm
        r['synth_native_frac_hbm'] = r['synth_native_write_gbs'] / hbm
        r['sph_zonal_mean_pts_per_s'] = pts / ((tp + to) * 1e-3)
        r['sph_zonal_mean_native_pts_per_s'] = pts / ((tp + tn) * 1e-3)
        out.append({k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()})
        del eng, coef, nat
        torch.cuda.empty_cache()
    return {'workload': 'config5: ne120pg2 (345600 cols) x 72 lev x 24 steps, one field, L sweep', 'n_gpus': 1,
            'peaks': {'fp64_tflops': FP64_PEAK_TFLOPS, 'hbm_gbs': hbm}, 'sweep': out}


def run_ours(args):
    ctx = Ctx()
    torch = ctx.torch
    head, eng, xs, plev, lat = headline(args, ctx)
    e2e = None
    if not args.no_e2e:
        e2e = e2e_leg(args, ctx, head, xs, plev, lat)
    del xs, eng
    import gc
    from pytemdiags_b200 import zonal
    zonal._ENGINE_CACHE.clear()
    gc.collect()
    torch.cuda.empty_cache()

    records = {}
    if not args.no_records:
        todo = [('config3', lambda: run_record(ctx, 'config3', 12)),
                ('config4', lambda: run_record(ctx, 'config4', 30)),
                ('config4_dedup', lambda: run_record(ctx, 'config4', 30, dedup=True)),
                ('config2_dedup', lambda: run_record(ctx, 'config2', 73, dedup=True))]
        for name, fn in todo:
            try:
                records[name] = fn()
            except Exception as e:      # noqa: BLE001  (a failed extra block must not lose the headline line)
                records[name] = {'error': '%s: %s' % (type(e).__name__, str(e)[:300])}
                if ctx.world > 1:
                    raise
            gc.collect()
            torch.cuda.empty_cache()
        if ctx.world == 1:
            try:
                records['config5'] = run_sweep(ctx)
            except Exception as e:      # noqa: BLE001
                records['config5'] = {'error': '%s: %s' % (type(e).__name__, str(e)[:300])}

    if ctx.rank != 0:
        if ctx.world > 1:
            ctx.dist.destroy_process_group()
        return

    cfg, L, N, K, Ts = head['cfg'], head['L'], head['N'], head['K'], head['Ts']
    cpu = None
    if not args.no_cpu and ctx.world == 1:
        v, secs, setup, cores = cpu_suite_sample(cfg, L, args.cpu_tsample)
        cpu = {'value': v, 'unit': UNIT, 'cores': cores, 'kind': 'port',
               'sample': '%d of %d time steps of %s, factored NumPy oracle (literal N x N form infeasible: %.0f GB); '
                         'suite %.1f s, matrix setup (pinv) %.1f s not included'
                         % (args.cpu_tsample, cfg['T'], args.config, 8.0 * N * N / 1e9, secs, setup)}
    line = {
        'metric': METRIC, 'value': head['value'], 'unit': UNIT, 'n_gpus': ctx.world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': head['ms'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': {'workload': '%s: grid %s (%d cols) x %d lev, L=%d, time slab of %d steps per GPU per step '
                               '(%d slabs = the %d-step record)' % (args.config, cfg['grid'], N, K, L, Ts,
                                                                   -(-cfg['T'] // Ts), cfg['T']),
                   'slab_steps': Ts, 'l2': 'inputs (%.1f GB per GPU) are far larger than the 126 MB L2'
                                           % (4 * 8.0 * N * Ts * K / 1e9),
                   'parallelism': 'time slabs, one per GPU; one NCCL all-gather of the outputs per step' if ctx.world > 1
                                  else 'single GPU'},
        'clocks': head['clocks'], 'e2e': e2e, 'gpu_launches': head['launches_per_step'] * args.steps,
        'roofline': head['roof'], 'roofline_project': head['roof_proj'],
        'step_fp64_tflops_per_gpu': head['step_tf'], 'hbm_algorithmic': head['hbm'],
        'kernel_ms': head['kms'], 'basis_build_s': head['basis_s'], 'spot_check': head['spot_check'],
        'cpu_baseline': cpu, 'records': records,
    }
    if head['dump']:
        line['dump_outputs'] = head['dump']
    print(json.dumps(line))
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='config2')
    ap.add_argument('--slab-steps', type=int, default=73)
    ap.add_argument('--e2e-steps', type=int, default=16)
    ap.add_argument('--cpu-tsample', type=int, default=8)
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-records', action='store_true', help='skip the config 3 / 4 / 5 record blocks')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed as DIR/<name>.npy (float64, at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
