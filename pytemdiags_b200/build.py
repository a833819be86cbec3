"""Builds pytemdiags_b200/libtemd.so with nvcc for sm_100a (in-tree, so it ships with gpurun)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libtemd.so')
SOURCES = ['temd_api.cu', 'temd_project.cu', 'temd_basis.cu', 'temd_synth.cu', 'temd_synth_res.cu', 'temd_eddy.cu',
           'temd_epilogue.cu', 'temd_fields.cu', 'temd_comm.cu', 'temd_dedup.cu', 'temd_svd.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']


def _newest_source_mtime():
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, '..', 'include', 'temd.h')]
    return max(os.path.getmtime(f) for f in files)


def build(force=False, verbose=False):
    """Compile every .cu into objects (in parallel) and link the shared library."""
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_source_mtime():
        return LIB
    nvcc = os.environ.get('NVCC', 'nvcc')
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode != 0:
            sys.stderr.write(out)
        if pr.returncode != 0:
            raise RuntimeError('nvcc failed on %s' % src)
        objs.append(obj)
    cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-ldl']
    subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
