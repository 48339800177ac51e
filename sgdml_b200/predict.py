"""``GDMLPredict`` -- the reference's public prediction API (sgdml/predict.py:248-1294)
backed by the B200 engine.

Drop-in for ``sgdml.predict.GDMLPredict`` on the hot path: same constructor signature,
``predict(R, return_E)``, ``set_R_desc``, ``set_R_d_desc``, ``set_alphas``,
``prepare_parallel``; same model dict / .npz layout (train.py:793-830).  Inputs stay
float64 end to end (the reference's torch path downcasts R to float32,
predict.py:1197-1201).  No CPU path: without the CUDA library or a GPU it raises.
"""

import logging
import timeit

import numpy as np

from . import _lib
from .desc import Desc


class GDMLPredict(object):
    def __init__(
        self,
        model,
        batch_size=None,
        num_workers=None,
        max_memory=None,
        max_processes=None,
        use_torch=False,
        log_level=None,
    ):
        """predict.py:249-463.  `batch_size`, `num_workers`, `max_memory`, `max_processes`
        and `use_torch` are accepted for signature compatibility; they only steer the
        reference's CPU/torch engines."""
        self.log = logging.getLogger(__name__)
        if log_level is not None:
            self.log.setLevel(log_level)

        if 'type' not in model or not (model['type'] == 'm' or model['type'] == b'm'):
            raise ValueError('The provided data structure is not a valid model.')  # predict.py:326-328

        _lib.require_gpu()

        self.n_atoms = int(np.asarray(model['z']).shape[0])
        self.desc = Desc(self.n_atoms, max_processes=max_processes)
        self.lat_and_inv = None
        if 'lattice' in model:  # predict.py:332-334
            lat = np.ascontiguousarray(model['lattice'], dtype=np.float64)
            self.lat_and_inv = (lat, np.ascontiguousarray(np.linalg.inv(lat)))

        self.n_train = int(model['R_desc'].shape[1])
        self.sig = float(model['sig'])  # as stored (predict.py:346); no int() truncation (torchtools.py:476)
        self.std = float(model['std']) if 'std' in model else 1.0
        self.c = float(model['c'])
        self.n_perms = int(np.asarray(model['perms']).shape[0])
        self.tril_perms_lin = np.ascontiguousarray(model['tril_perms_lin'], dtype=np.int64)

        # Cache for iterative training mode (predict.py:335-337).
        self.R_desc = None
        self.R_d_desc = None

        # knobs of the reference's CPU engine that its callers read back (cli.py:1526-1530, predict.py:462-509):
        # there are no worker processes and no chunking here
        self.num_workers = 0
        self.chunk_size = self.n_train
        self.bulk_mp = False
        self.use_torch = use_torch

        R_desc = np.ascontiguousarray(np.asarray(model['R_desc'], dtype=np.float64).T)  # (M, D); stored (D, M)
        R_d_desc_alpha = np.ascontiguousarray(model['R_d_desc_alpha'], dtype=np.float64)
        import ctypes

        handle = ctypes.c_void_p()
        _lib.check(
            _lib.lib().sgdml_b200_model_create(
                ctypes.byref(handle),
                self.n_atoms,
                self.n_train,
                self.n_perms,
                _lib.ptr(R_desc),
                _lib.ptr(R_d_desc_alpha),
                _lib.ptr(self.tril_perms_lin),
                self.sig,
                self.std,
                self.c,
            ),
            'model_create',
        )
        self._handle = handle
        if self.lat_and_inv is not None:
            _lib.check(
                _lib.lib().sgdml_b200_model_set_lattice(handle, _lib.ptr(self.lat_and_inv[0]), _lib.ptr(self.lat_and_inv[1])),
                'model_set_lattice',
            )
        if 'alphas_E' in model:  # energy constraints in the kernel (predict.py:443-447)
            self._set_alphas_E(model['alphas_E'])

    def __del__(self):
        h = getattr(self, '_handle', None)
        if h is not None and h.value:
            try:
                _lib.lib().sgdml_b200_model_destroy(h)
            except Exception:
                pass
            self._handle = None

    def set_contraction_slices(self, slices):
        """Extension (large descriptors, D > 256): run the predictor's four GEMMs on the tcgen05 tensor cores through
        `slices` exact int8 slices per operand (4..7) instead of FP64 DMMA (0).  See include/sgdml_b200.h."""
        _lib.check(
            _lib.lib().sgdml_b200_model_set_contraction_slices(self._handle, int(slices), _lib.current_stream()),
            'model_set_contraction_slices',
        )

    # ------------------------------------------------------------------ training-mode hooks
    def set_R_desc(self, R_desc):
        """predict.py:511-525."""
        self.R_desc = R_desc

    def set_R_d_desc(self, R_d_desc):
        """predict.py:527-549: uploads the training descriptor Jacobians once."""
        self.R_d_desc = R_d_desc
        if R_d_desc is not None:
            a = np.ascontiguousarray(R_d_desc, dtype=np.float64)
            if a.shape != (self.n_train, self.desc.dim, 3):
                raise ValueError('R_d_desc must have shape (n_train, D, 3)')
            _lib.check(_lib.lib().sgdml_b200_model_set_R_d_desc(self._handle, _lib.ptr(a)), 'model_set_R_d_desc')

    def _set_alphas_E(self, alphas_E):
        a = np.ascontiguousarray(np.asarray(alphas_E, dtype=np.float64).ravel())
        if a.shape != (self.n_train,):
            raise ValueError('alphas_E must have one entry per training point')
        _lib.check(_lib.lib().sgdml_b200_model_set_alphas_E(self._handle, _lib.ptr(a), _lib.current_stream()), 'model_set_alphas_E')

    def set_alphas(self, alphas_F, alphas_E=None):
        """predict.py:551-601: new regression coefficients (used once per CG iteration)."""
        if alphas_E is not None:
            self._set_alphas_E(alphas_E)  # predict.py:594-601
        assert self.R_d_desc is not None  # predict.py:575
        a = alphas_F if not isinstance(alphas_F, np.ndarray) else np.ascontiguousarray(alphas_F, dtype=np.float64)
        _lib.check(
            _lib.lib().sgdml_b200_model_set_alphas(self._handle, _lib.ptr(a), _lib.current_stream()),
            'model_set_alphas',
        )

    def get_R_d_desc_alpha(self):
        out = np.empty((self.n_train, self.desc.dim))
        _lib.check(_lib.lib().sgdml_b200_model_get_R_d_desc_alpha(self._handle, _lib.ptr(out)), 'get_R_d_desc_alpha')
        return out

    def _set_num_workers(self, num_workers=None, force_reset=False):
        """predict.py:603-649 (CPU worker pool): nothing to configure on the engine."""
        self.num_workers = 0

    def _set_chunk_size(self, chunk_size=None):
        """predict.py:651-673."""
        self.chunk_size = self.n_train

    def _set_bulk_mp(self, bulk_mp=False):
        """predict.py:710-725."""
        self.bulk_mp = False

    # ------------------------------------------------------------------ CPU autotuner stubs
    def prepare_parallel(self, n_bulk=1, n_reps=1, return_is_from_cache=False):
        """predict.py:770-1042 tunes CPU workers/chunks; nothing to tune here.  Returns the
        measured throughput (geometries/s) like the reference."""
        M = max(int(n_bulk), 1)
        R = np.tile(self._train_like_geometry(), (M, 1))
        self.predict(R)
        t0 = timeit.default_timer()
        for _ in range(max(int(n_reps), 1)):
            self.predict(R)
        gps = M * max(int(n_reps), 1) / (timeit.default_timer() - t0)
        return (gps, False) if return_is_from_cache else gps

    def _train_like_geometry(self):
        # any non-degenerate geometry will do for a throughput probe: atoms on a line 1.5 A apart
        r = np.zeros((self.n_atoms, 3))
        r[:, 0] = 1.5 * np.arange(self.n_atoms)
        r[:, 1] = 0.1 * np.arange(self.n_atoms) ** 2
        return r.reshape(1, -1)

    # ------------------------------------------------------------------ prediction
    def predict(self, R=None, return_E=True, out=None):
        """predict.py:1146-1294.  R (B, 3N) [or (3N,)] float64 -> (E (B,), F (B, 3N)) or (F,).
        With R=None the cached training descriptors are evaluated (predict.py:1219-1235).
        `out=(E, F)` (extension): preallocated outputs of the right shape/dtype on the same device as R
        (e.g. pinned host tensors), filled in place and returned.
        NumPy in -> NumPy out; torch tensor in (CUDA, or pinned/pageable host) -> torch tensors out on the
        same device (CUDA tensors are used in place, no copies)."""
        L = _lib.lib()
        dim_i = 3 * self.n_atoms
        if R is None:
            if self.R_d_desc is None:
                raise RuntimeError(
                    'A reference to the training geometry descriptors needs to be set (using '
                    "'set_R_d_desc()') for this function to work without arguments."
                )
            n = self.n_train
            F = np.empty((n, dim_i))
            E = np.empty(n) if return_E else None
            _lib.check(
                L.sgdml_b200_predict_train(self._handle, 0, n, 1, _lib.ptr(E), _lib.ptr(F), _lib.current_stream()),
                'predict_train',
            )
            return (E, F) if return_E else (F,)

        if isinstance(R, np.ndarray) or not hasattr(R, 'data_ptr'):
            R = np.ascontiguousarray(R, dtype=np.float64)
            if R.ndim == 1:
                R = R[None, :]  # predict.py:1183-1184
            if R.size % dim_i != 0 or (R.ndim == 2 and R.shape[1] != dim_i):
                raise ValueError('R must have 3*n_atoms columns')
            R = R.reshape(-1, dim_i)
            n = R.shape[0]
            if out is not None:
                E, F = out
            else:
                F = np.empty((n, dim_i))
                E = np.empty(n) if return_E else None
        else:
            import torch

            if R.dtype != torch.float64:
                raise ValueError('torch inputs must be float64')
            R = R.contiguous().reshape(-1, dim_i) if R.dim() != 1 else R.contiguous().reshape(1, dim_i)
            n = R.shape[0]
            if out is not None:
                E, F = out
            else:
                pin = (not R.is_cuda) and R.is_pinned()  # pinned host tensor in -> pinned host tensors out
                F = torch.empty((n, dim_i), dtype=torch.float64, device=R.device, pin_memory=pin)
                E = torch.empty((n,), dtype=torch.float64, device=R.device, pin_memory=pin) if return_E else None
        if not return_E:
            E = None  # the engine skips the energy output entirely
        if out is not None:  # (buffers allocated above are right by construction)
            self._check_out(R, E, F, n, dim_i)
        _lib.check(
            L.sgdml_b200_predict(self._handle, _lib.ptr(R), n, _lib.ptr(E), _lib.ptr(F), _lib.current_stream()),
            'predict',
        )
        return (E, F) if return_E else (F,)

    def predict_hessian(self, R, out=None):
        """Extension: analytic Hessian.  R (B, 3N) [or (3N,)] float64 -> (E (B,), F (B, 3N), H (B, 3N, 3N)), with
        H = d^2 E / dR^2 full and symmetric in model units (energy / length^2); E and F as ``predict`` gives them.
        Lattices and alphas_E are honoured.  NumPy in -> NumPy out; torch tensor in (CUDA, or pinned/pageable host)
        -> torch tensors out on the same device.  `out=(E, F, H)`: preallocated outputs, checked as in ``predict``.
        All contractions run in FP64, whatever ``set_contraction_slices`` chose."""
        dim_i = 3 * self.n_atoms
        if isinstance(R, np.ndarray) or not hasattr(R, 'data_ptr'):
            R = np.ascontiguousarray(R, dtype=np.float64)
            if R.ndim == 1:
                R = R[None, :]
            if R.size % dim_i != 0 or (R.ndim == 2 and R.shape[1] != dim_i):
                raise ValueError('R must have 3*n_atoms columns')
            R = R.reshape(-1, dim_i)
            n = R.shape[0]
            alloc = lambda shape: np.empty(shape)  # noqa: E731
        else:
            import torch

            if R.dtype != torch.float64:
                raise ValueError('torch inputs must be float64')
            R = R.contiguous().reshape(-1, dim_i) if R.dim() != 1 else R.contiguous().reshape(1, dim_i)
            n = R.shape[0]
            pin = (not R.is_cuda) and R.is_pinned()  # pinned host tensor in -> pinned host tensors out
            alloc = lambda shape: torch.empty(shape, dtype=torch.float64, device=R.device, pin_memory=pin)  # noqa: E731
        if out is None:
            E, F, H = alloc((n,)), alloc((n, dim_i)), alloc((n, dim_i, dim_i))
        else:
            if len(out) != 3 or out[2] is None:
                raise ValueError('out must be (E, F, H) with H given (E, F may be None)')
            E, F, H = out
            self._check_out(R, E, F, n, dim_i)
            self._check_buf(R, H, (n, dim_i, dim_i), 'H')
        _lib.check(
            _lib.lib().sgdml_b200_predict_hessian(
                self._handle, _lib.ptr(R), n, _lib.ptr(E), _lib.ptr(F), _lib.ptr(H), _lib.current_stream()
            ),
            'predict_hessian',
        )
        return E, F, H

    @staticmethod
    def _check_out(R, E, F, n, dim_i):
        """Output buffers go to the engine as raw double*: wrong dtype / layout / device would corrupt memory."""
        for buf, shape, name in ((F, (n, dim_i), 'F'), (E, (n,), 'E')):
            if buf is not None:
                GDMLPredict._check_buf(R, buf, shape, name)

    @staticmethod
    def _check_buf(R, buf, shape, name):
        if tuple(buf.shape) != shape:
            raise ValueError('out buffer %s has the wrong shape %s (expected %s)' % (name, tuple(buf.shape), shape))
        if isinstance(buf, np.ndarray):
            if buf.dtype != np.float64 or not buf.flags['C_CONTIGUOUS'] or not buf.flags['WRITEABLE']:
                raise ValueError('out buffer %s must be a writeable C-contiguous float64 array' % name)
            if not isinstance(R, np.ndarray) and R.is_cuda:
                raise ValueError('out buffer %s is a host array but R is a CUDA tensor' % name)
        else:
            import torch

            if buf.dtype != torch.float64 or not buf.is_contiguous():
                raise ValueError('out buffer %s must be a contiguous float64 tensor' % name)
            r_dev = None if isinstance(R, np.ndarray) else R.device
            if buf.is_cuda and (r_dev is None or buf.device != r_dev):
                raise ValueError('out buffer %s lives on %s but R does not' % (name, buf.device))
            if (not buf.is_cuda) and r_dev is not None and r_dev.type == 'cuda':
                raise ValueError('out buffer %s is a host tensor but R is a CUDA tensor' % name)

    def kmatvec_train(self, m_begin=0, m_end=None, out=None):
        """Raw (std = 1, c = 0) force sums on training points [m_begin, m_end): the K.v operator
        of the iterative solver (iterative.py:183-204) for alphas = v set via set_alphas."""
        if m_end is None:
            m_end = self.n_train
        n = m_end - m_begin
        F = out if out is not None else np.empty((n, 3 * self.n_atoms))
        _lib.check(
            _lib.lib().sgdml_b200_predict_train(
                self._handle, m_begin, m_end, 0, None, _lib.ptr(F), _lib.current_stream()
            ),
            'predict_train',
        )
        return F
