"""Host wrapper of the batched GCN actor (C ABI in ``include/tactor.h``): the batched counterpart of
``multimodals_OneAgent.act`` (``train/code/truss2D_RL.py:328-354``).  PyTorch only provides the device
buffers and the stream; the forward pass runs in ``libtfem.so``."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import capi
from .tf_checkpoint import ACTOR_LAYERS


class _Weights(C.Structure):
    _fields_ = [("kernel", C.c_void_p * 13), ("bias", C.c_void_p * 13)]


class _Inputs(C.Structure):
    _fields_ = [("x_n", C.c_void_p), ("A_n", C.c_void_p), ("A_s", C.c_void_p), ("A_n_ts", C.c_void_p),
                ("A_n_cs", C.c_void_p), ("x_p", C.c_void_p), ("A_p", C.c_void_p), ("n_pf", C.c_void_p),
                ("P", C.c_int32)]


ACTOR_EXPORTS = ("tactor_last_error", "tactor_create", "tactor_destroy", "tactor_set_weights", "tactor_set_weights_device",
                 "tactor_forward", "tactor_act",
                 "tactor_act_dev", "tactor_reserve_calls", "tactor_launch_count", "tactor_status",
                 "tactor_selftest_tmem_layout")

_lib = capi.lib
_lib.tactor_last_error.restype = C.c_char_p
_lib.tactor_create.argtypes = [C.POINTER(_Weights), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
_lib.tactor_destroy.argtypes = [C.c_void_p]
_lib.tactor_set_weights.argtypes = [C.c_void_p, C.POINTER(_Weights)]
_lib.tactor_set_weights_device.argtypes = [C.c_void_p, C.POINTER(_Weights), C.c_void_p]
_lib.tactor_forward.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Inputs), C.c_void_p, C.c_void_p, C.c_void_p]
_lib.tactor_act.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Inputs), C.c_void_p, C.c_void_p, C.c_float, C.c_float,
                            C.c_float, C.c_uint64, C.c_void_p]
_lib.tactor_launch_count.argtypes = [C.c_void_p]
_lib.tactor_launch_count.restype = C.c_int64
_lib.tactor_status.argtypes = [C.c_void_p]
_lib.tactor_selftest_tmem_layout.argtypes = [C.c_int]


def _check(rc):
    if rc != 0:
        raise capi.TfemError("libtfem actor error %d: %s" % (rc, _lib.tactor_last_error().decode()))


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def selftest_tmem_layout(device: int = 0) -> None:
    """raises unless ``tcgen05.st.16x128b`` places the mma accumulator fragment in tensor memory the way the actor kernel's
    operand generators assume (hardware check, one tiny launch)"""
    _check(_lib.tactor_selftest_tmem_layout(int(device)))


class BatchedActor:
    """One agent's actor for up to ``max_batch`` environments of ``nodes`` nodes (2 num_x: any even count
    from 6 to 32) on ``device``.

    ``weights``: ``{layer name: (kernel [in,out], bias [out])}`` as returned by
    :func:`mop_truss_marl_b200.tf_checkpoint.load_actor_weights`."""

    def __init__(self, weights, nodes: int, max_batch: int, device="cuda:0", mu=0.1, theta=0.1, sigma=0.1, seed=20):
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise capi.TfemError("BatchedActor needs a CUDA device: there is no CPU path")
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", index)
        self.nodes, self.max_batch = int(nodes), int(max_batch)
        self.mu, self.theta, self.sigma, self.seed = float(mu), float(theta), float(sigma), int(seed)
        w = self._pack(weights)
        self._h = C.c_void_p()
        _check(_lib.tactor_create(C.byref(w), self.nodes, self.max_batch, index, C.byref(self._h)))
        self.update_num = 0                        # multimodals_OneAgent.update_num (:352)

    def _pack(self, weights):
        w = _Weights()
        self._keep = []
        for i, name in enumerate(ACTOR_LAYERS):
            k = np.ascontiguousarray(weights[name][0], dtype=np.float32)
            b = np.ascontiguousarray(weights[name][1], dtype=np.float32)
            self._keep += [k, b]
            w.kernel[i] = k.ctypes.data
            w.bias[i] = b.ctypes.data
        return w

    def set_weights(self, weights):
        """replace all 13 layers (``actor_model.set_weights`` / ``load_weights`` on a live actor)"""
        w = self._pack(weights)
        _check(_lib.tactor_set_weights(self._h, C.byref(w)))

    def set_weights_device(self, weights):
        """the same from tensors that already live on the actor's device -- ``{layer: (kernel [in,out], bias [out])}`` of
        contiguous float32 CUDA tensors, e.g. a learner's parameters -- on the current stream: no host round trip and no
        device-wide synchronisation (``tactor_set_weights_device``)"""
        w = _Weights()
        for i, name in enumerate(ACTOR_LAYERS):
            k, b = weights[name]
            for t in (k, b):
                if not (isinstance(t, torch.Tensor) and t.device == self.device and t.dtype == torch.float32 and t.is_contiguous()):
                    raise ValueError("layer %s: expected contiguous float32 tensors on %s" % (name, self.device))
            w.kernel[i], w.bias[i] = k.data_ptr(), b.data_ptr()
        _check(_lib.tactor_set_weights_device(self._h, C.byref(w), self._stream()))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.tactor_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _inputs(self, x_n, A_n, A_s, A_n_ts, A_n_cs, x_p, A_p, n_pf):
        B, N = x_n.shape[0], self.nodes
        P = x_p.shape[1]
        for t, shape in ((x_n, (B, N, 13)), (A_n, (N, N)), (A_s, (B, N, N)), (A_n_ts, (B, N, N)),
                         (A_n_cs, (B, N, N)), (x_p, (B, P, 4)), (A_p, (B, P, P))):
            if t.dtype != torch.float32 or tuple(t.shape) != shape or not t.is_contiguous() or t.device != self.device:
                raise ValueError("expected contiguous float32 CUDA tensor of shape %s, got %s" % (shape, tuple(t.shape)))
        if n_pf is not None and (n_pf.dtype != torch.int32 or tuple(n_pf.shape) != (B,) or n_pf.device != self.device):
            raise ValueError("n_pf must be int32 [B] on the actor's device")
        inp = _Inputs(_ptr(x_n), _ptr(A_n), _ptr(A_s), _ptr(A_n_ts), _ptr(A_n_cs), _ptr(x_p), _ptr(A_p), _ptr(n_pf), P)
        return B, inp

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def forward(self, x_n, A_n, A_s, A_n_ts, A_n_cs, x_p, A_p, n_pf=None, out=None):
        """sigmoid outputs (geo [B,N,2], topo [B,N,3]) without exploration noise"""
        B, inp = self._inputs(x_n, A_n, A_s, A_n_ts, A_n_cs, x_p, A_p, n_pf)
        geo, topo = out if out is not None else (torch.empty(B, self.nodes, 2, device=self.device),
                                                 torch.empty(B, self.nodes, 3, device=self.device))
        _check(_lib.tactor_forward(self._h, B, C.byref(inp), _ptr(geo), _ptr(topo), self._stream()))
        return geo, topo

    def act(self, x_n, A_n, A_s, A_n_ts, A_n_cs, x_p, A_p, n_pf=None, out=None):
        """``act``: forward + OU noise on every entry (the reference adds it at test time too)."""
        B, inp = self._inputs(x_n, A_n, A_s, A_n_ts, A_n_cs, x_p, A_p, n_pf)
        geo, topo = out if out is not None else (torch.empty(B, self.nodes, 2, device=self.device),
                                                 torch.empty(B, self.nodes, 3, device=self.device))
        _check(_lib.tactor_act(self._h, B, C.byref(inp), _ptr(geo), _ptr(topo), self.mu, self.theta, self.sigma,
                               self.seed, self._stream()))
        self.update_num += 1
        return geo, topo

    def launch_count(self) -> int:
        return int(_lib.tactor_launch_count(self._h))

    def check(self) -> None:
        """synchronise and raise if a kernel reported a timed-out barrier wait or an activation outside the fp16 range
        of the split tensor-core product"""
        _check(_lib.tactor_status(self._h))
