"""ctypes binding of the engine's C ABI (include/sgdml_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` (or ``make -C
sgdml_b200/csrc``).  There is no CPU fallback: if the library is missing, or no CUDA
device is visible, every compute call raises.
"""

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libsgdml_b200.so')

_lib = None

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)
c_void_p = C.c_void_p
i64 = C.c_int64

# name -> (restype, argtypes); mirrors include/sgdml_b200.h one to one
SIGNATURES = {
    'sgdml_b200_abi_version': (C.c_int, []),
    'sgdml_b200_release_workspaces': (C.c_int, []),
    'sgdml_b200_last_error': (C.c_char_p, []),
    'sgdml_b200_device_count': (C.c_int, []),
    'sgdml_b200_tril_perms_lin': (C.c_int, [c_void_p, i64, i64, c_void_p]),
    'sgdml_b200_desc_from_R': (C.c_int, [c_void_p, i64, i64, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_d_desc_dot_vec': (C.c_int, [c_void_p, c_void_p, i64, i64, c_void_p, c_void_p]),
    'sgdml_b200_vec_dot_d_desc': (C.c_int, [c_void_p, c_void_p, i64, i64, c_void_p, c_void_p]),
    'sgdml_b200_model_create': (
        C.c_int,
        [C.POINTER(c_void_p), i64, i64, i64, c_void_p, c_void_p, c_void_p, C.c_double, C.c_double, C.c_double],
    ),
    'sgdml_b200_model_destroy': (C.c_int, [c_void_p]),
    'sgdml_b200_predict': (C.c_int, [c_void_p, c_void_p, i64, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_predict_hessian': (C.c_int, [c_void_p, c_void_p, i64, c_void_p, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_model_set_R_d_desc': (C.c_int, [c_void_p, c_void_p]),
    'sgdml_b200_model_set_alphas': (C.c_int, [c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_predict_train': (C.c_int, [c_void_p, i64, i64, C.c_int, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_model_get_R_d_desc_alpha': (C.c_int, [c_void_p, c_void_p]),
    'sgdml_b200_assemble': (
        C.c_int,
        [c_void_p, c_void_p, c_void_p, i64, i64, i64, C.c_double, c_void_p, i64, C.c_double, c_void_p, i64, c_void_p],
    ),
    'sgdml_b200_assemble_rows': (
        C.c_int,
        [c_void_p, c_void_p, c_void_p, i64, i64, i64, C.c_double, c_void_p, i64, C.c_double, i64, i64, c_void_p, i64,
         c_void_p],
    ),
    'sgdml_b200_assemble_ecstr': (
        C.c_int, [c_void_p, c_void_p, c_void_p, i64, i64, i64, C.c_double, C.c_double, c_void_p, i64, c_void_p]),
    'sgdml_b200_set_assemble_variant': (C.c_int, [C.c_int]),
    'sgdml_b200_potrf': (C.c_int, [c_void_p, i64, i64, c_void_p]),
    'sgdml_b200_potrs': (C.c_int, [c_void_p, i64, i64, c_void_p, i64, i64, c_void_p]),
    'sgdml_b200_solve_analytic': (C.c_int, [c_void_p, i64, i64, C.c_double, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_dgemm_nt': (
        C.c_int,
        [i64, i64, i64, C.c_double, c_void_p, i64, c_void_p, i64, C.c_double, c_void_p, i64, c_void_p],
    ),
    'sgdml_b200_ozaki_gemm_nt': (
        C.c_int,
        [i64, i64, i64, C.c_double, c_void_p, i64, c_void_p, i64, c_void_p, i64, C.c_int, C.c_int, c_void_p],
    ),
    'sgdml_b200_ozaki_debug': (
        C.c_int,
        [i64, i64, i64, c_void_p, i64, c_void_p, i64, c_void_p, i64, C.c_int, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p],
    ),
    'sgdml_b200_gather_rows_neg': (C.c_int, [c_void_p, i64, i64, c_void_p, c_void_p, i64, c_void_p]),
    'sgdml_b200_add_diag': (C.c_int, [c_void_p, i64, i64, C.c_double, c_void_p]),
    'sgdml_b200_trsm_right_lt': (C.c_int, [c_void_p, i64, i64, c_void_p, i64, i64, c_void_p]),
    'sgdml_b200_gram_tn': (C.c_int, [c_void_p, i64, i64, i64, C.c_double, c_void_p, i64, c_void_p]),
    'sgdml_b200_row_sqnorms': (C.c_int, [c_void_p, i64, i64, i64, c_void_p, c_void_p]),
    'sgdml_b200_nystroem_apply': (C.c_int, [c_void_p, i64, i64, i64, C.c_double, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_nystroem_project': (C.c_int, [c_void_p, i64, i64, i64, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_nystroem_expand': (
        C.c_int,
        [c_void_p, i64, i64, i64, C.c_double, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    'sgdml_b200_desc_from_R_pbc': (C.c_int, [c_void_p, i64, i64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_model_set_lattice': (C.c_int, [c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_model_set_alphas_E': (C.c_int, [c_void_p, c_void_p, c_void_p]),
    'sgdml_b200_model_set_contraction_slices': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    'sgdml_b200_set_predict_variant': (C.c_int, [C.c_int]),
    'sgdml_b200_model_dims': (C.c_int, [c_void_p, c_int64_p, c_int64_p, c_int64_p]),
    'sgdml_b200_pcg_workspace_doubles': (C.c_int64, [i64, i64, i64, i64]),
    'sgdml_b200_pcg': (
        C.c_int,
        [c_void_p, i64, i64, c_void_p, i64, i64, C.c_double, c_void_p, c_void_p, C.c_int, C.c_double, i64, i64,
         c_void_p, i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64_p, c_double_p, c_void_p],
    ),
    'sgdml_b200_set_solve_slices': (C.c_int, [C.c_int]),
    'sgdml_b200_set_gemm_variant': (C.c_int, [C.c_int]),
    'sgdml_b200_profile_enable': (C.c_int, [C.c_int]),
    'sgdml_b200_profile_reset': (C.c_int, []),
    'sgdml_b200_profile_get': (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    'sgdml_b200_fp64_peak_tflops': (C.c_int, [C.POINTER(C.c_double)]),
    'sgdml_b200_fp64_peak_tflops_sustained': (C.c_int, [C.c_double, C.POINTER(C.c_double)]),
}


# callback types of sgdml_b200_pcg (include/sgdml_b200.h)
EXCHANGE_FN = C.CFUNCTYPE(C.c_int, c_void_p, C.c_int, c_void_p, i64)
PROGRESS_FN = C.CFUNCTYPE(C.c_int, c_void_p, i64, c_double_p, i64)


class EngineError(RuntimeError):
    pass


def lib():
    """Loads libsgdml_b200.so (once).  Fails loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EngineError(
                'sgdml_b200: %s not found -- build it with `python -c "import __graft_entry__ as g; g.build()"` '
                'or `make -C sgdml_b200/csrc`.  There is no CPU fallback.' % LIB_PATH
            )
        handle = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def last_error():
    msg = lib().sgdml_b200_last_error()
    return msg.decode() if msg else ''


def check(rc, what):
    """Maps C-ABI return codes onto the exceptions the reference's callers catch:
    info > 0 -> np.linalg.LinAlgError('... not positive definite') (analytic.py:101,
    iterative.py:451-459); CUDA OOM -> RuntimeError('... out of memory')
    (torchtools.py:352)."""
    if rc == 0:
        return
    msg = last_error()
    if rc > 0:
        raise np.linalg.LinAlgError(msg or '%d-th leading minor of the array is not positive definite' % rc)
    if rc == -2:  # cudaErrorMemoryAllocation
        raise RuntimeError('CUDA out of memory in %s: %s' % (what, msg))
    raise EngineError('%s failed (rc=%d): %s' % (what, rc, msg))


def ptr(x):
    """Address of a NumPy array (host) or torch tensor (host or CUDA), or None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        if not x.flags.c_contiguous:
            raise ValueError('array must be C-contiguous')
        return x.ctypes.data
    # torch tensor
    if not x.is_contiguous():
        raise ValueError('tensor must be contiguous')
    return x.data_ptr()


_stream_state = None  # (cuda available, torch._C._cuda_getCurrentRawStream or None, torch._C._cuda_getDevice or None)


def current_stream():
    """cudaStream_t of torch's current stream (so that the engine's kernels are ordered
    with torch work and visible to torch.cuda.Event timing).  This sits on the B = 1 latency path (MD): the
    availability check is cached and the raw-stream accessor is used where torch has it (~0.3 us instead of ~4)."""
    global _stream_state
    if _stream_state is None:
        import torch

        avail = torch.cuda.is_available()
        _stream_state = (
            avail,
            getattr(torch._C, '_cuda_getCurrentRawStream', None) if avail else None,
            getattr(torch._C, '_cuda_getDevice', None) if avail else None,
        )
    avail, raw, dev = _stream_state
    if not avail:
        return None
    if raw is not None and dev is not None:
        return raw(dev())
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_gpu():
    if lib().sgdml_b200_device_count() < 1:
        raise EngineError('sgdml_b200: no CUDA device visible; this engine has no CPU fallback')


KERNEL_FAMILIES = ['predict_main', 'predict_aux', 'assemble', 'gemm', 'potf2', 'trsm', 'trsv', 'desc', 'misc', 'hessian']


def profile_snapshot():
    """{family: (device_ms_total, timed_scopes, launches)} since the last reset."""
    out = {}
    for i, name in enumerate(KERNEL_FAMILIES):
        ms, sc, ln = C.c_double(), C.c_int64(), C.c_int64()
        lib().sgdml_b200_profile_get(i, C.byref(ms), C.byref(sc), C.byref(ln))
        out[name] = (ms.value, sc.value, ln.value)
    return out


def launches_total():
    return sum(v[2] for v in profile_snapshot().values())
