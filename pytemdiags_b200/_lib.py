"""ctypes binding of libtemd.so (the C ABI declared in include/temd.h).

There is NO CPU fallback: if the library is missing or no sm_100 device is visible, the compute entry
points raise.  PyTorch is used by callers only for device memory and streams.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('TEMD_LIB', os.path.join(_HERE, 'libtemd.so'))   # TEMD_LIB: A/B-test another build

# every symbol include/temd.h declares (checked by tests/test_abi.py)
SYMBOLS = (
    'temd_version', 'temd_last_error', 'temd_plan_create', 'temd_plan_destroy', 'temd_plan_lpad',
    'temd_basis_build', 'temd_basis_build_weighted', 'temd_basis_export', 'temd_project', 'temd_synth_out', 'temd_synth_native',
    'temd_eddy_native', 'temd_multiply', 'temd_eddy_flux_project', 'temd_tracer_flux_project', 'temd_tem_epilogue', 'temd_tracer_epilogue', 'temd_check_finite', 'temd_host_copy', 'temd_synth_fields',
    'temd_synth_out_dlat', 'temd_basis_export_dlat', 'temd_basis_build_dedup', 'temd_group_sums', 'temd_dedup_flux', 'temd_dedup_expand',
    'temd_comm_unique_id', 'temd_comm_init', 'temd_comm_destroy', 'temd_allgather_outputs',
    'temd_plan_create_min_norm', 'temd_plan_rank', 'temd_basis_build_min_norm',
)

# order of the output planes written by temd_tem_epilogue (enum TEMD_OUT_* in temd.h)
EPILOGUE_OUTPUTS = (
    'dub_dp', 'dthetab_dp', 'ubcoslat', 'dubcoslat_dlat', 'psi', 'psicoslat', 'dpsicoslat_dlat',
    'dpsi_dp', 'int_vbdp', 'vtem', 'omegatem', 'wtem', 'psitem', 'epfy', 'epfz', 'epdiv',
    'utendepfd', 'utendvtem', 'utendwtem',
)


class EpilogueArgs(C.Structure):
    _fields_ = [('nt', C.c_int), ('nlev', C.c_int), ('nlat', C.c_int), ('ld', C.c_size_t),
                ('zm', C.c_void_p), ('p', C.c_void_p), ('latr', C.c_void_p), ('gp', C.c_void_p), ('gl', C.c_void_p),
                ('p_uniform', C.c_int), ('lat_uniform', C.c_int), ('hp', C.c_double), ('hlat', C.c_double),
                ('coslat', C.c_void_p), ('f', C.c_void_p),
                ('p0', C.c_double), ('a', C.c_double), ('H', C.c_double), ('g0', C.c_double), ('pi', C.c_double),
                ('out', C.c_void_p)]


GS_NPLANES = 15          # TEMD_GS_NPLANES
GS_A0, GS_S, GS_P, GS_SW = 0, 4, 8, 11

TRACER_OUTPUTS = ('dqb_dp', 'qbcoslat', 'dqbcoslat_dlat', 'etfy', 'etfz', 'etdiv', 'qtendetfd', 'qtendvtem', 'qtendwtem')


class TracerArgs(C.Structure):
    _fields_ = [('nt', C.c_int), ('nlev', C.c_int), ('nlat', C.c_int), ('ld', C.c_size_t),
                ('zmq', C.c_void_p), ('psi', C.c_void_p), ('vtem', C.c_void_p), ('omegatem', C.c_void_p),
                ('p', C.c_void_p), ('latr', C.c_void_p), ('gp', C.c_void_p), ('gl', C.c_void_p),
                ('p_uniform', C.c_int), ('lat_uniform', C.c_int), ('hp', C.c_double), ('hlat', C.c_double),
                ('coslat', C.c_void_p), ('p0', C.c_double), ('a', C.c_double), ('H', C.c_double),
                ('out', C.c_void_p)]


_lib = None


def load():
    """Load libtemd.so (building is `python -m pytemdiags_b200.build` / `__graft_entry__.build()`)."""
    global _lib
    if _lib is not None:
        return _lib
    if 'TEMD_LIB' not in os.environ:
        # a library older than its sources is a stale build (e.g. an edit without `python -m pytemdiags_b200.build`):
        # rebuild rather than run yesterday's kernels.  nvcc is part of the image; failure to build is loud.
        from . import build as _build
        try:
            stale = (not os.path.exists(LIB_PATH)) or os.path.getmtime(LIB_PATH) < _build._newest_source_mtime()
        except OSError:
            stale = False
        if stale and os.environ.get('TEMD_NO_AUTOBUILD', '0') in ('', '0'):
            # one builder at a time (torchrun starts N ranks at once): the others wait on the lock and re-check
            import fcntl
            with open(os.path.join(_HERE, '.build.lock'), 'w') as lk:
                fcntl.flock(lk, fcntl.LOCK_EX)
                try:
                    if (not os.path.exists(LIB_PATH)) or os.path.getmtime(LIB_PATH) < _build._newest_source_mtime():
                        _build.build(force=True)
                finally:
                    fcntl.flock(lk, fcntl.LOCK_UN)
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('libtemd.so not found at %s: run `python -m pytemdiags_b200.build` '
                           '(there is no CPU fallback)' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i, sz, d = C.c_void_p, C.c_int, C.c_size_t, C.c_double
    lib.temd_version.restype = i
    lib.temd_last_error.restype = C.c_char_p
    lib.temd_plan_create.argtypes = [i, i, i, i, C.POINTER(vp)]
    lib.temd_plan_destroy.argtypes = [vp]
    lib.temd_plan_lpad.argtypes = [vp]
    lib.temd_plan_create_min_norm.argtypes = [i, i, i, i, C.POINTER(vp)]
    lib.temd_plan_rank.argtypes = [vp]
    lib.temd_basis_build_min_norm.argtypes = [vp, vp, vp, vp, i, vp, C.POINTER(i), C.POINTER(d), vp]
    lib.temd_basis_build.argtypes = [vp, vp, vp, C.POINTER(d), vp]
    lib.temd_basis_build_weighted.argtypes = [vp, vp, vp, vp, vp]
    lib.temd_basis_export.argtypes = [vp, vp, vp, vp, vp]
    lib.temd_project.argtypes = [vp, C.POINTER(vp), i, i, sz, vp, i, i, vp, vp]
    lib.temd_synth_out.argtypes = [vp, vp, i, vp, sz, vp]
    lib.temd_synth_native.argtypes = [vp, vp, i, vp, sz, vp]
    lib.temd_synth_out_dlat.argtypes = [vp, vp, i, vp, sz, vp]
    lib.temd_basis_export_dlat.argtypes = [vp, vp, vp]
    lib.temd_eddy_native.argtypes = [vp, vp, sz, vp, i, vp, i, vp, sz, vp]
    lib.temd_multiply.argtypes = [vp, sz, vp, sz, vp, sz, i, i, vp]
    lib.temd_eddy_flux_project.argtypes = [vp, vp, vp, vp, vp, i, sz, vp, vp, i, vp, vp]
    lib.temd_tracer_flux_project.argtypes = [vp, vp, vp, vp, vp, i, sz, vp, vp, vp]
    lib.temd_tem_epilogue.argtypes = [vp, C.POINTER(EpilogueArgs), vp]
    lib.temd_tracer_epilogue.argtypes = [vp, C.POINTER(TracerArgs), vp]
    lib.temd_check_finite.argtypes = [vp, sz, vp]
    lib.temd_host_copy.argtypes = [vp, vp, sz, i]
    lib.temd_synth_fields.argtypes = [vp, i, i, i, i, i, i, sz, vp, vp, vp, vp]
    lib.temd_basis_build_dedup.argtypes = [vp, vp, vp, vp, C.POINTER(d), vp]
    lib.temd_group_sums.argtypes = [C.POINTER(vp), i, i, sz, vp, vp, i, i, i, i, vp, vp, i, i, i, vp, sz, vp]
    lib.temd_dedup_flux.argtypes = [vp, sz, vp, sz, vp, vp, i, i, vp, sz, vp]
    lib.temd_dedup_expand.argtypes = [vp, sz, vp, i, vp, sz, vp, vp, d, d, vp, sz, i, i, vp]
    lib.temd_comm_unique_id.argtypes = [C.c_char_p]
    lib.temd_comm_init.argtypes = [i, i, i, C.c_char_p, C.POINTER(vp)]
    lib.temd_comm_destroy.argtypes = [vp]
    lib.temd_allgather_outputs.argtypes = [vp, vp, vp, sz, vp]
    for name in SYMBOLS:
        fn = getattr(lib, name)
        if name not in ('temd_last_error',):
            fn.restype = i
    _lib = lib
    return lib


class TemdError(RuntimeError):
    pass


def check(rc, what=''):
    """Map a libtemd return code to the reference's exception type (RuntimeError)."""
    if rc != 0:
        msg = load().temd_last_error().decode('utf-8', 'replace')
        raise TemdError('%s failed (code %d): %s' % (what or 'libtemd call', rc, msg))
