"""Batched truss environment: B independent copies of the reference ``Game_research04`` state machine
(``test/*/code/truss2D_ENV.py:232-604``) resident on one GPU.

PyTorch is only the allocator / stream provider here: every computation goes through the C ABI of
``libtfem.so`` (``include/tfem.h``).  Field names follow the reference's state tuple
``(x_n, A_n, A_s, A_n_ts, A_n_cs, mask, x_pf, A_pf, nN_x_n, nN_x_e, nC_e)`` (``truss2D_ENV.py:354``).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import capi
from .families import FAMILIES, FamilySpec, family_desc


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class BatchedTrussEnv:
    """``batch`` environments of one geometry family on ``device``.

    ``reset()`` = ``_game_get_1_state()`` for every environment (``truss2D_ENV.py:339-354``);
    ``step(a_geo, a_topo, coin)`` = ``_game_modify(nN_x_n, nN_x_e, nC_e, [a_geo, a_topo])`` applied to each
    environment's own current state (``:373-589``), the stale move range carried explicitly.
    """

    STATE_FIELDS = ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e")
    FP64_FIELDS = ("point64", "d", "axial", "ratio", "U", "reactions")

    def __init__(self, family, batch: int, device="cuda:0", fp64_outputs: bool = True):
        self.spec: FamilySpec = FAMILIES[family] if isinstance(family, str) else family
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise capi.TfemError("BatchedTrussEnv needs a CUDA device: libtfem has no CPU path")
        if not torch.cuda.is_available():
            raise capi.TfemError("CUDA is not available: libtfem has no CPU path")
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", index)
        self.handle = self._open_handle(index)
        d = self.handle.dims
        self.B, self.N, self.E, self.ndof, self.nres = int(batch), d.N, d.E, d.ndof, d.nres
        self.fp64_outputs = fp64_outputs
        # topology constants of the state tuple
        self.A_n = torch.from_numpy(self.handle.table("A_n")).to(self.device)
        self.mask = torch.from_numpy(self.handle.table("mask")).to(self.device)
        self.nC_e = torch.from_numpy(self.handle.table("nC_e")).to(self.device)
        self.int_obj = self._int_obj()
        self.game_step = 1                     # Game_research04.game_step (:242)
        self._alloc(self.B)

    def _open_handle(self, index):
        return capi.Handle(family_desc(self.spec), index)

    def _int_obj(self):
        return self.handle.table("int_obj")

    # ------------------------------------------------------------------------------------------------
    def _alloc(self, B):
        N, E, dev = self.N, self.E, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        self.x_n = torch.empty(B, N, 13, **f32)
        self.A_s = torch.empty(B, N, N, **f32)
        self.A_n_ts = torch.empty(B, N, N, **f32)
        self.A_n_cs = torch.empty(B, N, N, **f32)
        self.nN_x_n = torch.empty(B, N, 12, **f32)
        self.nN_x_e = torch.empty(B, E, 21, **f32)
        self.move_range = torch.zeros(B, N, 2, **f32)
        self.point = torch.empty(B, 4, **f32)
        self.status = torch.zeros(B, dtype=torch.int32, device=dev)
        self.y = torch.empty(B, N, dtype=torch.float64, device=dev) if self.fp64_outputs else None
        self.y_weak = torch.empty(B, N, dtype=torch.uint8, device=dev) if self.fp64_outputs else None
        if self.fp64_outputs:
            self.point64 = torch.empty(B, 4, **f64)
            self.d = torch.empty(B, self.ndof, **f64)
            self.axial = torch.empty(B, E, **f64)
            self.ratio = torch.empty(B, E, **f64)
            self.U = torch.empty(B, **f64)
            self.reactions = torch.empty(B, self.nres, **f64)
        else:
            self.point64 = self.d = self.axial = self.ratio = self.U = self.reactions = None
        self._out = self._make_out()

    def _make_out(self, lo=0, hi=None):
        o = capi.StepOut()
        for name in ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "point", "point64", "d", "axial",
                     "ratio", "U", "reactions", "status", "y", "y_weak"):
            t = getattr(self, name)
            setattr(o, name, _ptr(t if (t is None or (lo == 0 and hi is None)) else t[lo:hi]))
        return o

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------------------------------------
    def reset(self):
        capi.check(capi.lib.tfem_reset(self.handle.ptr, self.B, _ptr(self.move_range), C.byref(self._out),
                                       self._stream()))
        self.game_step = 1
        return self.state()

    def step(self, a_geo: torch.Tensor, a_topo: torch.Tensor, coin: torch.Tensor | None = None,
             rows: tuple | None = None, parent: "BatchedTrussEnv | None" = None):
        """a_geo [B,N,2], a_topo [B,N,3] float32 CUDA tensors (clipped in place, like the reference);
        coin [B] uint8/bool (1 = ``random.random() >= 0.5``).  Updates the state in place and returns
        ``point`` [B,4].  ``rows=(lo, hi)`` steps only environments lo..hi-1 (the action / coin tensors then
        hold hi-lo environments): the environments are independent, so a batch can be stepped in pieces on
        different streams (``host_pipeline.HostRollout``).  ``parent``: read the parent geometry (raw tables + the
        stale move range) from another environment batch of the same family and size and leave it untouched -- the
        driver's "three agents act on the same parent state" (``master_DDPG_truss2D_MO.py:262-330``): this batch
        becomes the child state."""
        lo, hi = (0, self.B) if rows is None else rows
        if not (0 <= lo < hi <= self.B):
            raise ValueError("rows must satisfy 0 <= lo < hi <= batch")
        nb = hi - lo
        self._check(a_geo, (nb, self.N, 2))
        self._check(a_topo, (nb, self.N, 3))
        if coin is not None:
            if coin.dtype == torch.bool:
                coin = coin.to(torch.uint8)
            if coin.dtype != torch.uint8 or coin.shape != (nb,) or coin.device != self.device or not coin.is_contiguous():
                raise ValueError("coin must be a contiguous uint8 [B] tensor on the env device")
        src = self
        if parent is not None:
            self._inherit(parent, lo, hi)
            src = parent
        sin = capi.StepIn()
        sin.set_node = _ptr(src.nN_x_n[lo:hi])
        sin.set_element = _ptr(src.nN_x_e[lo:hi])
        sin.a_geo = _ptr(a_geo)
        sin.a_topo = _ptr(a_topo)
        sin.coin = _ptr(coin)
        sin.move_range = _ptr(self.move_range[lo:hi])
        out = self._out if rows is None else self._make_out(lo, hi)
        self._launch_step(lo, hi, sin, out)
        if rows is None or hi == self.B:
            self.game_step += 1
        return self.point if rows is None else self.point[lo:hi]

    def _inherit(self, parent, lo, hi):
        """the per-environment state a child batch takes from its parent besides the raw tables"""
        if parent.B != self.B or parent.N != self.N or parent.E != self.E or parent.device != self.device:
            raise ValueError("parent must be a batch of the same family, size and device")
        self.move_range[lo:hi].copy_(parent.move_range[lo:hi])

    def _launch_step(self, lo, hi, sin, out):
        capi.check(capi.lib.tfem_step(self.handle.ptr, hi - lo, C.byref(sin), C.byref(out), self._stream()))

    def _check(self, t, shape):
        if not (isinstance(t, torch.Tensor) and t.dtype == torch.float32 and tuple(t.shape) == shape
                and t.device == self.device and t.is_contiguous()):
            raise ValueError("expected a contiguous float32 CUDA tensor of shape %s" % (shape,))

    def state(self):
        """the reference's state tuple, batched (x_pf/A_pf are host-side Pareto bookkeeping)"""
        return {"x_n": self.x_n, "A_n": self.A_n, "A_s": self.A_s, "A_n_ts": self.A_n_ts, "A_n_cs": self.A_n_cs,
                "mask": self.mask, "nN_x_n": self.nN_x_n, "nN_x_e": self.nN_x_e, "nC_e": self.nC_e,
                "point": self.point, "move_range": self.move_range, "status": self.status}

    # ------------------------------------------------------------------------------------------------
    def solve_only(self, y: torch.Tensor, section: torch.Tensor):
        """``Model.restore(); Model.gen_all()`` on explicit FP64 heights ``y`` [B,N] and int32 sections
        [B,E] (``FEM_2Dtruss.py:434-459``)."""
        B = y.shape[0]
        if y.dtype != torch.float64 or section.dtype != torch.int32 or tuple(y.shape) != (B, self.N) \
                or tuple(section.shape) != (B, self.E) or not y.is_contiguous() or not section.is_contiguous():
            raise ValueError("y must be float64 [B,N] and section int32 [B,E], contiguous")
        f64 = dict(dtype=torch.float64, device=self.device)
        out = {"d": torch.empty(B, self.ndof, **f64), "axial": torch.empty(B, self.E, **f64),
               "ratio": torch.empty(B, self.E, **f64), "U": torch.empty(B, **f64),
               "reactions": torch.empty(B, self.nres, **f64),
               "status": torch.zeros(B, dtype=torch.int32, device=self.device)}
        capi.check(capi.lib.tfem_solve_only(self.handle.ptr, B, _ptr(y), _ptr(section), _ptr(out["d"]),
                                            _ptr(out["axial"]), _ptr(out["ratio"]), _ptr(out["U"]),
                                            _ptr(out["reactions"]), _ptr(out["status"]), self._stream()))
        return out

    def solve_dense_dmma(self, y: torch.Tensor, section: torch.Tensor):
        """the same solve as ``solve_only`` by the dense blocked Cholesky with DMMA trailing updates
        (``tfem_solve_dense_dmma``): returns ``d`` [B,ndof] in reference DOF order and ``status`` [B]"""
        B = y.shape[0]
        if y.dtype != torch.float64 or section.dtype != torch.int32 or tuple(y.shape) != (B, self.N) \
                or tuple(section.shape) != (B, self.E) or not y.is_contiguous() or not section.is_contiguous():
            raise ValueError("y must be float64 [B,N] and section int32 [B,E], contiguous")
        d = torch.empty(B, self.ndof, dtype=torch.float64, device=self.device)
        status = torch.zeros(B, dtype=torch.int32, device=self.device)
        capi.check(capi.lib.tfem_solve_dense_dmma(self.handle.ptr, B, _ptr(y), _ptr(section), _ptr(d), _ptr(status),
                                                  self._stream()))
        return d, status

    def launch_count(self) -> int:
        return self.handle.launch_count()


class MixedTrussEnv(BatchedTrussEnv):
    """``batch`` environments on ``device``, each of its own family among ``families`` (names or FamilySpecs that share
    num_x and support_case, at most ``capi.MAX_FAMILIES``; the large meshes fit fewer, see ``tfem_create_mixed``).  This is
    the reference's training batch: ``train/code/master_DDPG_truss2D_MO.py:787-815`` draws a shape and a truss type for
    every episode (``families.TRAIN_FAMILIES``).  One ``tfem_step_mixed`` launch steps the whole batch; environment b is
    bit for bit what a ``BatchedTrussEnv`` of family ``families[family_ids[b]]`` computes from the same inputs.

    ``reset(family_ids)`` takes a uint8 CUDA tensor [B] of indices into ``families`` and keeps a copy as
    ``self.family_ids``; ``step`` has the signature of ``BatchedTrussEnv.step`` (``parent=`` children copy the parent's
    family ids).  ``int_obj`` is [F, 2].  The single-family calls (``solve_only``, ``solve_dense_dmma``) and
    ``host_pipeline.HostRollout`` refuse a batch of more than one family; ``host_pipeline.MixedHostRollout`` steps it
    from host-resident state."""

    def __init__(self, families, batch: int, device="cuda:0", fp64_outputs: bool = True):
        self.specs = tuple(FAMILIES[f] if isinstance(f, str) else f for f in families)
        if not self.specs:
            raise ValueError("at least one family is needed")
        super().__init__(self.specs[0], batch, device, fp64_outputs)
        self.family_ids = torch.full((self.B,), 255, dtype=torch.uint8, device=self.device)   # no family until reset

    def _open_handle(self, index):
        return capi.MixedHandle([family_desc(s) for s in self.specs], index)

    def _int_obj(self):
        return np.stack([capi.Handle(family_desc(s), -1).table("int_obj") for s in self.specs])

    def reset(self, family_ids: torch.Tensor):
        if not (isinstance(family_ids, torch.Tensor) and family_ids.dtype == torch.uint8 and tuple(family_ids.shape) == (self.B,)
                and family_ids.device == self.device and family_ids.is_contiguous()):
            raise ValueError("family_ids must be a contiguous uint8 [B] tensor on the env device")
        self.family_ids.copy_(family_ids)
        capi.check(capi.lib.tfem_reset_mixed(self.handle.ptr, self.B, _ptr(self.family_ids), _ptr(self.move_range),
                                             C.byref(self._out), self._stream()))
        self.game_step = 1
        return self.state()

    def _inherit(self, parent, lo, hi):
        if not isinstance(parent, MixedTrussEnv) or parent.specs != self.specs:
            raise ValueError("parent must be a mixed batch over the same families")
        super()._inherit(parent, lo, hi)
        self.family_ids[lo:hi].copy_(parent.family_ids[lo:hi])

    def _launch_step(self, lo, hi, sin, out):
        capi.check(capi.lib.tfem_step_mixed(self.handle.ptr, hi - lo, _ptr(self.family_ids[lo:hi]), C.byref(sin),
                                            C.byref(out), self._stream()))


def step_host(handle: capi.Handle, set_node, set_element, move_range, a_geo, a_topo, coin=None,
              want_fp64: bool = True, out: dict | None = None, stream: int = 0):
    """``_game_modify`` with HOST numpy arrays in and out, batched over the leading axis
    (``tfem_step_host``).  ``a_geo``/``a_topo``/``move_range`` are updated in place like the reference
    updates the caller's action arrays and the model's move range."""
    d = handle.dims
    B = set_node.shape[0]
    N, E = d.N, d.E

    def chk(a, shape, dtype):
        if a.dtype != dtype or tuple(a.shape) != shape or not a.flags["C_CONTIGUOUS"]:
            raise ValueError("expected C-contiguous %s array of shape %s" % (np.dtype(dtype).name, shape))
        return a
    chk(set_node, (B, N, 12), np.float32); chk(set_element, (B, E, 21), np.float32)
    chk(move_range, (B, N, 2), np.float32); chk(a_geo, (B, N, 2), np.float32); chk(a_topo, (B, N, 3), np.float32)
    if out is None:
        out = {"x_n": np.empty((B, N, 13), np.float32), "A_s": np.empty((B, N, N), np.float32),
               "A_n_ts": np.empty((B, N, N), np.float32), "A_n_cs": np.empty((B, N, N), np.float32),
               "nN_x_n": np.empty((B, N, 12), np.float32), "nN_x_e": np.empty((B, E, 21), np.float32),
               "point": np.empty((B, 4), np.float32), "status": np.zeros((B,), np.int32)}
        if want_fp64:
            out.update(point64=np.empty((B, 4)), d=np.empty((B, d.ndof)), axial=np.empty((B, E)),
                       ratio=np.empty((B, E)), U=np.empty((B,)), reactions=np.empty((B, d.nres)),
                       y=np.empty((B, N)), y_weak=np.empty((B, N), np.uint8))
    sin = capi.StepIn()
    vp = lambda a: C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)  # noqa: E731
    sin.set_node, sin.set_element, sin.a_geo, sin.a_topo = vp(set_node), vp(set_element), vp(a_geo), vp(a_topo)
    sin.move_range = vp(move_range)
    if coin is not None:
        coin = np.ascontiguousarray(coin, dtype=np.uint8)
    sin.coin = vp(coin)
    sout = capi.StepOut()
    for name, _ in capi.StepOut._fields_:
        setattr(sout, name, vp(out.get(name)))
    capi.check(capi.lib.tfem_step_host(handle.ptr, B, C.byref(sin), C.byref(sout), C.c_void_p(stream)))
    return out
