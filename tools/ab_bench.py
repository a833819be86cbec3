"""A/B the headline step between two builds of libtemd.so on one GPU.

    python tools/ab_bench.py BASE_LIB [NEW_LIB] [--runs 3] [--out DIR] [-- extra bench.py arguments]

Runs `bench.py --no-cpu --no-e2e` alternately with TEMD_LIB=BASE_LIB and TEMD_LIB=NEW_LIB (default: the in-tree
build), --runs times each, and prints ms_per_step and kernel_ms.eddy_flux_project of every run with the spread of
each build.  Then runs bench.py --dump-outputs once per build and compares every dumped plane normwise
(max|new - base| / max|base|).  The per-run JSON lines and the summary go to --out/ab_summary.json (default: a temporary directory)."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(lib, extra):
    env = dict(os.environ, TEMD_LIB=os.path.abspath(lib))
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--no-cpu', '--no-e2e'] + extra, env=env,
                         cwd=ROOT, check=True, capture_output=True, text=True).stdout
    return json.loads([ln for ln in out.splitlines() if ln.startswith('{')][-1])


def main():
    argv = sys.argv[1:]
    extra = argv[argv.index('--') + 1:] if '--' in argv else []
    argv = argv[:argv.index('--')] if '--' in argv else argv
    runs, out_dir = 3, None
    if '--runs' in argv:
        i = argv.index('--runs')
        runs = int(argv[i + 1])
        del argv[i:i + 2]
    if '--out' in argv:
        i = argv.index('--out')
        out_dir = argv[i + 1]
        del argv[i:i + 2]
    base = argv[0]
    new = argv[1] if len(argv) > 1 else os.path.join(ROOT, 'pytemdiags_b200', 'libtemd.so')
    out_dir = out_dir or tempfile.mkdtemp(prefix='ab_bench_')
    os.makedirs(out_dir, exist_ok=True)

    res = {'base': [], 'new': []}
    for r in range(runs):
        for name, lib in (('base', base), ('new', new)):
            line = bench(lib, extra)
            res[name].append(line)
            print('run %d %-4s ms_per_step %8.2f  eddy_flux_project %7.2f ms  project %7.2f ms  spot_check %.2e %s'
                  % (r, name, line['ms_per_step'], line['kernel_ms']['eddy_flux_project'], line['kernel_ms']['project'],
                     line['spot_check']['max_normwise_err'], line['spot_check']['ok']), flush=True)
    summary = {}
    for name, lines in res.items():
        st = [x['ms_per_step'] for x in lines]
        ed = [x['kernel_ms']['eddy_flux_project'] for x in lines]
        summary[name] = {'ms_per_step': st, 'eddy_flux_project_ms': ed}
        print('%-4s ms_per_step min %.2f max %.2f | eddy_flux_project min %.2f max %.2f'
              % (name, min(st), max(st), min(ed), max(ed)))
    summary['every_new_run_beats_every_base_run'] = {
        'ms_per_step': max(summary['new']['ms_per_step']) < min(summary['base']['ms_per_step']),
        'eddy_flux_project_ms': max(summary['new']['eddy_flux_project_ms']) < min(summary['base']['eddy_flux_project_ms'])}
    print(json.dumps(summary['every_new_run_beats_every_base_run']))

    errs = {}
    with tempfile.TemporaryDirectory(prefix='ab_dump_') as tmp:   # 2 x 64 MB of planes: compared, not kept
        dirs = {name: os.path.join(tmp, name) for name in ('base', 'new')}
        for name, lib in (('base', base), ('new', new)):
            bench(lib, ['--no-records', '--dump-outputs', dirs[name]] + extra)
        for f in sorted(os.listdir(dirs['base'])):
            a, b = np.load(os.path.join(dirs['base'], f)), np.load(os.path.join(dirs['new'], f))
            errs[f[:-4]] = float(np.abs(b - a).max() / np.abs(a).max())
    for k, v in errs.items():
        print('%-12s %.2e' % (k, v))
    print('planes %d, worst normwise difference %.2e' % (len(errs), max(errs.values())))
    summary['dump_normwise_diff'] = errs
    with open(os.path.join(out_dir, 'ab_summary.json'), 'w') as fh:
        json.dump({'runs': res, 'summary': summary}, fh, indent=1)


if __name__ == '__main__':
    main()
