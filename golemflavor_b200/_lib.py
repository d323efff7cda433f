"""ctypes binding of ``libgolemflavor_b200.so`` (the C ABI of ``include/golemflavor_b200.h``).

torch is used for device memory and streams only: tensors are handed to the library as raw
device pointers.  There is no fallback: if the library has not been built (``python -c
"import __graft_entry__ as g; g.build()"``) or no CUDA device is present, compute calls raise.
"""

import ctypes as C
import os

import numpy as np

GF_MAX_DIM = 16
GF_MAX_BINS = 64
GF_SRC_MAX = 256   # sources per gf_scan_evidence_sources / gf_profile_sources call (csrc/gf_sources_dev.cuh)
GF_EVS_MAX_UNITS = 4096   # sources x groups per gf_scan_evidence_sources_groups call (csrc/gf_sources.cu)
GF_EVIDENCE_MAX_GROUPS = 32   # sample groups of the grouped evidence grids: a power of two in [2, 32]

GF_OK, GF_ERR_ARG, GF_ERR_CUDA = 0, 1, 2
ST_OUT_OF_PRIOR, ST_NON_UNITARY, ST_NON_FINITE, ST_ILL_COND, ST_REFINED = 1, 2, 4, 8, 16
PRIOR_UNIFORM, PRIOR_GAUSSIAN, PRIOR_LIMITEDGAUSS = 0, 1, 2
LLH_FLAT, LLH_GAUSSIAN = 0, 1

LIB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'lib')
# GOLEMFLAVOR_B200_LIB: developer override used to A/B kernel build variants (scratch/variants)
LIB_PATH = os.environ.get('GOLEMFLAVOR_B200_LIB') or os.path.join(LIB_DIR, 'libgolemflavor_b200.so')


class GolemFlavorError(RuntimeError):
    """CUDA-side failure (GF_ERR_CUDA) or a missing library / device."""


class PriorDim(C.Structure):
    _fields_ = [('lo', C.c_double), ('hi', C.c_double), ('mu', C.c_double), ('sigma', C.c_double),
                ('kind', C.c_int32), ('reserved', C.c_int32)]


class Model(C.Structure):
    """``gf_model`` -- field order and types must match the C header exactly."""
    _fields_ = [
        ('ndim', C.c_int32),
        ('col_sm', C.c_int32 * 4),
        ('col_mass', C.c_int32 * 2),
        ('col_src', C.c_int32 * 2),
        ('col_np', C.c_int32 * 4),
        ('col_scale', C.c_int32),
        ('col_x', C.c_int32),
        ('col_src3', C.c_int32 * 3),
        ('no_bsm', C.c_int32),
        ('dimension', C.c_int32),
        ('nbins', C.c_int32),
        ('llh_kind', C.c_int32),
        ('emulate_underflow', C.c_int32),
        ('fixed_sm', C.c_double * 4),
        ('fixed_mass', C.c_double * 2),
        ('fixed_src', C.c_double * 3),
        ('fixed_np', C.c_double * 4),
        ('fixed_loglam', C.c_double),
        ('bin_edges', C.c_double * (GF_MAX_BINS + 1)),
        ('fr_bf', C.c_double * 3),
        ('smearing', C.c_double),
        ('offset', C.c_double),
        ('llh_const', C.c_double),
        ('epsilon', C.c_double),
        ('prior', PriorDim * GF_MAX_DIM),
    ]


class ScanConfig(C.Structure):
    _fields_ = [('seed', C.c_uint64), ('first_index', C.c_uint64), ('count', C.c_uint64),
                ('nb', C.c_int32), ('reserved', C.c_int32)]


class EnsembleConfig(C.Structure):
    _fields_ = [('nchains', C.c_int64), ('nwalkers', C.c_int32), ('nfree', C.c_int32), ('nsteps', C.c_int64),
                ('step0', C.c_int64), ('thin', C.c_int64), ('a', C.c_double), ('seed', C.c_uint64), ('chain0', C.c_int64), ('mode', C.c_int32), ('cluster_blocks', C.c_int32)]


class ProfileConfig(C.Structure):
    _fields_ = [('seed', C.c_uint64), ('task0', C.c_int64), ('nstarts', C.c_int32), ('max_evals', C.c_int32),
                ('ftol', C.c_double), ('xtol', C.c_double)]


_P = C.c_void_p
_SIGNATURES = {
    'gf_abi_version': (C.c_int, []),
    'gf_sizeof': (C.c_uint64, [C.c_int32]),
    'gf_last_error': (C.c_char_p, []),
    'gf_launch_count': (C.c_uint64, []),
    'gf_device_info': (C.c_int, [C.POINTER(C.c_int32)] * 4),
    'gf_host_alloc': (C.c_int, [C.POINTER(C.c_void_p), C.c_uint64]),
    'gf_host_alloc_wc': (C.c_int, [C.POINTER(C.c_void_p), C.c_uint64]),
    'gf_host_free': (C.c_int, [_P]),
    'gf_model_check': (C.c_int, [C.POINTER(Model)]),
    'gf_angles_to_u': (C.c_int, [_P, C.c_int64, _P, _P]),
    'gf_angles_to_fr': (C.c_int, [_P, C.c_int64, _P, _P]),
    'gf_u_to_fr': (C.c_int, [_P, C.c_int64, _P, C.c_int64, _P, _P]),
    'gf_eigvec_herm3': (C.c_int, [_P, C.c_int64, _P, _P, _P, _P]),
    'gf_params_to_bsmu': (C.c_int, [_P, C.c_int32, _P, _P, C.c_int64, _P, C.c_int64, C.c_int32, C.c_double,
                                    C.c_int64, _P, _P, _P]),
    'gf_flux_averaged_fr': (C.c_int, [C.POINTER(Model), _P, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P]),
    'gf_lnprior': (C.c_int, [C.POINTER(Model), _P, C.c_int64, C.c_int64, C.c_int64, _P, _P]),
    'gf_multi_gaussian': (C.c_int, [_P, C.c_int64, C.POINTER(C.c_double), C.c_double, C.c_double, C.c_int32, _P, _P]),
    'gf_lnprob': (C.c_int, [C.POINTER(Model), _P, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P, _P]),
    'gf_lnprob_host': (C.c_int, [C.POINTER(Model), _P, C.c_int64, _P, _P, _P]),
    'gf_scan_hist': (C.c_int, [C.POINTER(Model), C.POINTER(ScanConfig), _P, _P, _P]),
    'gf_scan_samples': (C.c_int, [C.POINTER(Model), C.POINTER(ScanConfig), _P, _P, _P, _P]),
    'gf_ternary_hist': (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P]),
    'gf_scan_evidence': (C.c_int, [C.POINTER(Model), C.POINTER(ScanConfig), _P, _P]),
    'gf_scan_evidence_grid_workspace': (C.c_uint64, [C.c_int32]),
    'gf_scan_evidence_grid': (C.c_int, [C.POINTER(Model), C.POINTER(ScanConfig), _P, C.c_int32, _P, _P, C.c_uint64, _P]),
    'gf_scan_evidence_sources_workspace': (C.c_uint64, [C.c_int32, C.c_int32]),
    'gf_scan_evidence_sources': (C.c_int, [C.POINTER(Model), C.POINTER(ScanConfig), _P, C.c_int32, _P, _P, C.c_int32, _P, _P, C.c_uint64,
                                           _P]),
    'gf_scan_evidence_grid_groups_workspace': (C.c_uint64, [C.c_int32, C.c_int32]),
    'gf_scan_evidence_grid_groups': (C.c_int, [C.POINTER(Model), C.POINTER(ScanConfig), _P, C.c_int32, C.c_int32, _P, _P, C.c_uint64, _P]),
    'gf_scan_evidence_sources_groups_workspace': (C.c_uint64, [C.c_int32, C.c_int32, C.c_int32]),
    'gf_scan_evidence_sources_groups': (C.c_int, [C.POINTER(Model), C.POINTER(ScanConfig), _P, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P,
                                                  C.c_uint64, _P]),
    'gf_profile_grid': (C.c_int, [C.POINTER(Model), C.POINTER(ProfileConfig), _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    'gf_profile_sources': (C.c_int, [C.POINTER(Model), C.POINTER(ProfileConfig), _P, C.c_int32, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    'gf_coverage_mask': (C.c_int, [_P, C.c_int64, C.c_double, _P, C.POINTER(C.c_uint64), _P]),
    'gf_hist_smooth': (C.c_int, [_P, C.c_int32, C.c_uint64, _P, C.c_int32, _P, _P, _P]),
    'gf_coverage_mask_f64': (C.c_int, [_P, C.c_int64, C.c_double, _P, C.POINTER(C.c_double), C.POINTER(C.c_uint64), _P]),
    'gf_ensemble_run': (C.c_int, [C.POINTER(Model), C.POINTER(EnsembleConfig), _P, _P, _P, _P, _P, _P]),
    'gf_selftest_math': (C.c_int, [_P, C.c_int64, _P, _P, _P]),
    'gf_selftest_trig': (C.c_int, [_P, C.c_int64, _P, _P, _P, _P]),
    'gf_selftest_log': (C.c_int, [_P, C.c_int64, _P, _P]),
    'gf_fp64_peak_probe': (C.c_int, [C.c_int32, C.c_int64, _P, C.POINTER(C.c_double), _P]),
}
EXPORTS = tuple(sorted(_SIGNATURES))

_lib = None


def load():
    """dlopen the library once and attach the prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GolemFlavorError(
                'golemflavor_b200: {0} is missing -- build it first (python -c "import __graft_entry__ as g; '
                'g.build()" or python -m golemflavor_b200.build); there is no CPU fallback'.format(LIB_PATH))
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.gf_abi_version() != 1:
            raise GolemFlavorError('golemflavor_b200: ABI version mismatch, rebuild the library')
        for which, struct in enumerate((Model, ScanConfig, PriorDim, EnsembleConfig, ProfileConfig)):
            if lib.gf_sizeof(which) != C.sizeof(struct):
                raise GolemFlavorError('golemflavor_b200: layout of {0} differs between _lib.py ({1} B) and the '
                                       'library ({2} B)'.format(struct.__name__, C.sizeof(struct), lib.gf_sizeof(which)))
        _lib = lib
    return _lib


TORCH_OPS_PATH = os.path.join(LIB_DIR, 'libgolemflavor_b200_torch.so')
TORCH_OPS = ('abi_version', 'lnprob', 'lnprior', 'flux_averaged_fr', 'angles_to_u', 'angles_to_fr', 'u_to_fr', 'multi_gaussian', 'scan_hist')
_ops = None


def torch_ops():
    """``torch.ops.golemflavor``: the C ABI registered as torch operators (csrc/gf_torch_ops.cpp -- tensors in, tensors
    out, torch's current stream), loaded once with ``torch.ops.load_library``.  Raises if it has not been built."""
    global _ops
    if _ops is None:
        import torch
        load()   # the C-ABI library first: same checks, and the operator library links against it
        if not os.path.exists(TORCH_OPS_PATH):
            raise GolemFlavorError('golemflavor_b200: {0} is missing -- build it first (python -m golemflavor_b200.build); '
                                   'there is no fallback'.format(TORCH_OPS_PATH))
        torch.ops.load_library(TORCH_OPS_PATH)
        ops = torch.ops.golemflavor
        if int(ops.abi_version()) != 1:
            raise GolemFlavorError('golemflavor_b200: ABI version mismatch between the operator library and _lib.py')
        _ops = ops
    return _ops


def check(rc):
    """Map a C return code onto the reference's exception conventions
    (bad arguments -> ValueError, as ``fr.py:198-202``; runtime -> GolemFlavorError)."""
    if rc == GF_OK:
        return
    msg = load().gf_last_error().decode('utf-8', 'replace')
    if rc == GF_ERR_ARG:
        raise ValueError(msg)
    raise GolemFlavorError(msg)


_torch_ok = None


def torch_cuda():
    """Import torch and insist on a CUDA device (the check is made once per process: emcee-sized
    batches are latency-bound and torch.cuda.is_available() costs microseconds per call)."""
    global _torch_ok
    if _torch_ok is not None:
        return _torch_ok
    import torch
    if not torch.cuda.is_available():
        raise GolemFlavorError('golemflavor_b200: no CUDA device available; this package has no CPU path')
    _torch_ok = torch
    return torch


def ptr(t):
    """Device (or host) pointer of a tensor / None."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(torch):
    """Raw handle of torch's current CUDA stream (the private fast accessor when this torch has it:
    torch.cuda.current_stream() alone costs ~14 us per call)."""
    try:
        return C.c_void_p(torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))
    except AttributeError:
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def to_device(x, torch, shape_last=None):
    """Contiguous float64 CUDA tensor from array-like / tensor input."""
    if isinstance(x, torch.Tensor):
        t = x.to(device='cuda', dtype=torch.float64)
    else:
        t = torch.as_tensor(np.ascontiguousarray(np.asarray(x, dtype=np.float64))).cuda()
    t = t.contiguous()
    if shape_last is not None and (t.ndim == 0 or t.shape[-1] != shape_last):
        raise ValueError('expected trailing dimension {0}, got shape {1}'.format(shape_last, tuple(t.shape)))
    return t


def device_info():
    lib = load()
    v = [C.c_int32() for _ in range(4)]
    check(lib.gf_device_info(*[C.byref(x) for x in v]))
    return dict(sm_count=v[0].value, cc=(v[1].value, v[2].value), clock_khz=v[3].value)


class HostBuffer(object):
    """Page-locked host memory from the library (``gf_host_alloc`` / ``gf_host_alloc_wc``) as a NumPy array
    (``.array``); freed with the object.  ``write_combined=True`` is meant for input buffers the host only writes."""

    def __init__(self, shape, dtype=np.float64, write_combined=False):
        lib = load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._ptr = C.c_void_p()
        check((lib.gf_host_alloc_wc if write_combined else lib.gf_host_alloc)(C.byref(self._ptr), self.nbytes))
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            if self._ptr:
                load().gf_host_free(self._ptr)
                self._ptr = None
        except Exception:  # noqa: BLE001  (interpreter shutdown)
            pass
