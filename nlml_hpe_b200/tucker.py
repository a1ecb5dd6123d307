"""Batched Tucker-fit pose inversion on B200 (host side).

Python face of the C ABI in include/nlml_hpe_b200.h for the Tucker half of the hot path:
the fixed-iteration fit of TD_Tester.optimize_with_sgd (/root/reference/TD_Tester.py:127-159)
for a whole batch of feature vectors.  The reference-compatible single-sample entry points
live in nlml_hpe_b200/TD_Tester.py.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib

KERNEL_HINTS = {"auto": 0, "thread_per_sample": 1, "cta_per_sample": 2, "warp_per_sample": 3,
                "thread_per_sample_tmem": 4, "tensor_core": 5, "tensor_core_generic": 6}


def _flatten_landmarks(X, landmarks):
    """Raw MediaPipe landmarks [N,468,3] -> [N,1404] (x,y,z of landmark i at columns 3i..3i+2); anything else as given."""
    if landmarks and X.ndim == 3 and X.shape[2] == 3:
        return X.reshape(X.shape[0], X.shape[1] * 3)
    return X


def _device_index(device):
    if device is None:
        return torch.cuda.current_device() if torch.cuda.is_available() else 0
    d = torch.device(device)
    if d.type != "cuda":
        raise _lib.NlmlError(f"nlml_hpe_b200 runs on CUDA devices only (got {d}); there is no CPU fallback")
    return d.index if d.index is not None else torch.cuda.current_device()


class TuckerFitter:
    """Holds the device-resident constants for one Tucker tensor W and cosine-row fit.

    W: float32 [R_id, R_y, R_p, R_r, F] (Trained_data.npz 'W', TD_Inference.py:47);
    params_*: [R_a, 4] rows (a,b,c,d) of optimized_{yaw,pitch,roll} (TD_Inference.py:43-45);
    ranks are taken from W, and the first R_a rows of each params array are used
    (the reference hard-slices [0:3,:], TD_Inference.py:56-57).

    Every fit / solve / powell entry point takes landmarks=True for RAW MediaPipe landmarks ([N,468,3] or [N,>=F],
    x,y,z of landmark i at columns 3i..3i+2): the IPD normalisation of
    FeatureExtractor.Read_Landmarks_and_Normalizing_using_IPD (helpers/FeatureExtractor.py:30-66) then runs inside the
    kernels' reads of X, in float64 as the reference, and the result equals the call on the normalised features bit
    for bit.  Needs F >= 792 (landmark 263).
    """

    def __init__(self, W, params_y, params_p, params_r, device=None):
        lib = _lib.load()
        W = np.ascontiguousarray(np.asarray(W, dtype=np.float32))
        if W.ndim != 5:
            raise ValueError(f"W must be [R_id,R_y,R_p,R_r,F], got shape {W.shape}")
        self.ranks = tuple(int(r) for r in W.shape[:4])
        self.F = int(W.shape[4])
        rows = []
        for name, P, r in (("yaw", params_y, self.ranks[1]), ("pitch", params_p, self.ranks[2]),
                           ("roll", params_r, self.ranks[3])):
            P = np.asarray(P, dtype=np.float64)
            if P.ndim != 2 or P.shape[1] != 4 or P.shape[0] < r:
                raise ValueError(f"{name} cosine rows must be [>={r},4], got {P.shape}")
            rows.append(np.ascontiguousarray(P[:r]))
        self.device_index = _device_index(device)
        self.device = torch.device("cuda", self.device_index)
        self.n_params = 3 + self.ranks[0]
        handle = ctypes.c_void_p()
        _lib.check(lib.nlml_tucker_plan_create(W.ctypes.data, *self.ranks, self.F, rows[0].ctypes.data,
                                               rows[1].ctypes.data, rows[2].ctypes.data, self.device_index,
                                               ctypes.byref(handle)))
        self._lib, self._h = lib, handle

    def close(self):
        if getattr(self, "_h", None):
            self._lib.nlml_tucker_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return int(self._lib.nlml_tucker_launch_count(self._h))

    def fit(self, X, iters=3000, lr=1e-3, clip=1.0, kernel="auto", out=None, landmarks=False):
        """X: CUDA float32 tensor [N, >=F] (row stride arbitrary, unit column stride); with landmarks=True raw
        landmarks [N,468,3] or [N,>=F] (see the class docstring).

        Returns a CUDA tensor [N, 3+R_id]: (yaw, pitch, roll) in radians + identity coefficients,
        the vector optimize_with_sgd returns (TD_Tester.py:159).  Asynchronous on the current stream.
        """
        if not (isinstance(X, torch.Tensor) and X.is_cuda):
            raise TypeError("fit() takes a CUDA tensor; use fit_host() for numpy / CPU tensors")
        X = _flatten_landmarks(X, landmarks)
        if X.dtype != torch.float32 or X.dim() != 2 or X.shape[1] < self.F:
            raise ValueError(f"X must be float32 [N, >={self.F}], got {X.dtype} {tuple(X.shape)}")
        if X.device.index != self.device_index:
            raise ValueError(f"X is on {X.device}, plan is on {self.device}")
        if X.shape[0] > 0 and X.stride(1) != 1:
            X = X.contiguous()
        n = X.shape[0]
        if out is None:
            out = torch.empty((n, self.n_params), dtype=torch.float32, device=X.device)
        stream = torch.cuda.current_stream(X.device).cuda_stream
        ldx = X.stride(0) if n > 1 else max(X.shape[1], self.F)
        call = self._lib.nlml_tucker_fit_landmarks_f32 if landmarks else self._lib.nlml_tucker_fit_f32
        _lib.check(call(self._h, X.data_ptr(), n, ldx, int(iters), float(lr), float(clip),
                        out.data_ptr(), out.stride(0) if n > 1 else self.n_params, KERNEL_HINTS[kernel], stream))
        return out

    def solve(self, X, max_evals=0, return_evals=False, out=None, landmarks=False):
        """Converged fit (what TD_Tester.Test computes with scipy Powell, TD_Tester.py:191-199): damped Newton
        from p = 0 to the local minimum, one thread per sample.  X (and landmarks) as in fit().  Returns [N, 3+R_id]
        (radians + identity coefficients) and, with return_evals, the int32 [N] evaluations used.
        Ranks (5,3,3,3) only.  Asynchronous on the current stream."""
        if not (isinstance(X, torch.Tensor) and X.is_cuda):
            raise TypeError("solve() takes a CUDA tensor; use solve_host() for numpy / CPU tensors")
        X = _flatten_landmarks(X, landmarks)
        if X.dtype != torch.float32 or X.dim() != 2 or X.shape[1] < self.F:
            raise ValueError(f"X must be float32 [N, >={self.F}], got {X.dtype} {tuple(X.shape)}")
        if X.device.index != self.device_index:
            raise ValueError(f"X is on {X.device}, plan is on {self.device}")
        if X.shape[0] > 0 and X.stride(1) != 1:
            X = X.contiguous()
        n = X.shape[0]
        if out is None:
            out = torch.empty((n, self.n_params), dtype=torch.float32, device=X.device)
        evals = torch.zeros((n,), dtype=torch.int32, device=X.device) if return_evals else None
        stream = torch.cuda.current_stream(X.device).cuda_stream
        ldx = X.stride(0) if n > 1 else max(X.shape[1], self.F)
        call = self._lib.nlml_tucker_solve_landmarks_f32 if landmarks else self._lib.nlml_tucker_solve_f32
        _lib.check(call(self._h, X.data_ptr(), n, ldx, int(max_evals), out.data_ptr(),
                        out.stride(0) if n > 1 else self.n_params,
                        evals.data_ptr() if return_evals and n > 0 else None, stream))
        return (out, evals) if return_evals else out

    def powell(self, X, return_info=False, landmarks=False):
        """The reference's shipped default fit, bit for bit: scipy Powell from p = 0 over TD_Tester.objective
        (TD_Tester.py:31-58, :191-194; algorithm restated from scipy 1.18.1 in csrc/powell_math.h, objective evaluated in
        the reference's own operation order).  X: CUDA float32 [N, >=F].  Returns a CUDA float64 tensor [N, 3+R_id] =
        result.x (radians + identity coefficients) and, with return_info, (result.fun float64 [N], result.nfev int32 [N]).
        One CTA per sample, float64: ~10^4 poses/s -- use solve() / fit() for throughput.  Asynchronous.
        With landmarks=True (see the class docstring) it equals the reference's
        FE.get_feature_vector(..., normalize=True) -> Test() chain."""
        if not (isinstance(X, torch.Tensor) and X.is_cuda):
            raise TypeError("powell() takes a CUDA tensor")
        X = _flatten_landmarks(X, landmarks)
        if X.dtype != torch.float32 or X.dim() != 2 or X.shape[1] < self.F:
            raise ValueError(f"X must be float32 [N, >={self.F}], got {X.dtype} {tuple(X.shape)}")
        if X.device.index != self.device_index:
            raise ValueError(f"X is on {X.device}, plan is on {self.device}")
        if X.shape[0] > 0 and X.stride(1) != 1:
            X = X.contiguous()
        n = X.shape[0]
        out = torch.empty((n, self.n_params), dtype=torch.float64, device=X.device)
        fun = torch.empty((n,), dtype=torch.float64, device=X.device) if return_info else None
        nfev = torch.empty((n,), dtype=torch.int32, device=X.device) if return_info else None
        stream = torch.cuda.current_stream(X.device).cuda_stream
        ldx = X.stride(0) if n > 1 else max(X.shape[1], self.F)
        call = self._lib.nlml_tucker_powell_landmarks_f64 if landmarks else self._lib.nlml_tucker_powell_f64
        _lib.check(call(self._h, X.data_ptr(), n, ldx, out.data_ptr(), self.n_params,
                        fun.data_ptr() if return_info and n > 0 else None,
                        nfev.data_ptr() if return_info and n > 0 else None, stream))
        return (out, fun, nfev) if return_info else out

    def solve_host(self, X, max_evals=0, out=None, landmarks=False):
        """solve() for numpy / CPU float32 [N, F] in host memory (or raw landmarks with landmarks=True); pipelined like
        fit_host()."""
        if isinstance(X, torch.Tensor):
            X = X.detach().numpy()
        X = _flatten_landmarks(np.asarray(X), landmarks)
        if X.dtype != np.float32 or X.ndim != 2 or X.shape[1] < self.F or (X.size and X.strides[1] != 4):
            raise ValueError(f"X must be float32 [N, >={self.F}] with unit column stride")
        n = X.shape[0]
        if out is None:
            out = np.empty((n, self.n_params), dtype=np.float32)
        ldx = X.strides[0] // 4 if n > 1 else X.shape[1]
        call = self._lib.nlml_tucker_solve_landmarks_host_f32 if landmarks else self._lib.nlml_tucker_solve_host_f32
        _lib.check(call(self._h, X.ctypes.data, n, ldx, int(max_evals), out.ctypes.data, self.n_params))
        return out

    def fit_host(self, X, iters=3000, lr=1e-3, clip=1.0, out=None, landmarks=False):
        """X: numpy / CPU tensor float32 [N, F] in host memory (pinned memory makes the copies
        asynchronous); with landmarks=True raw landmarks [N,468,3] or [N,>=F].  Host->device copy, fit and
        device->host copy are pipelined inside the library.  Returns numpy float32 [N, 3+R_id]."""
        if isinstance(X, torch.Tensor):
            X = X.detach().numpy()
        X = _flatten_landmarks(np.asarray(X), landmarks)
        if X.dtype != np.float32 or X.ndim != 2 or X.shape[1] < self.F or (X.size and X.strides[1] != 4):
            raise ValueError(f"X must be float32 [N, >={self.F}] with unit column stride")
        n = X.shape[0]
        if out is None:
            out = np.empty((n, self.n_params), dtype=np.float32)
        ldx = X.strides[0] // 4 if n > 1 else X.shape[1]
        call = self._lib.nlml_tucker_fit_landmarks_host_f32 if landmarks else self._lib.nlml_tucker_fit_host_f32
        _lib.check(call(self._h, X.ctypes.data, n, ldx, int(iters), float(lr), float(clip), out.ctypes.data, self.n_params))
        return out
