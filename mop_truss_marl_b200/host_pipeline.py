"""Host-resident rollouts: the caller keeps the reference's state tuple in (pinned) host memory, like the reference
driver does (``master_DDPG_truss2D_MO.py:167-260``), and every step moves it to the GPU, lets the actor act, steps
the environments and brings the new state tuple, the objective point and the actions back.

The work is done by ``trollout_step_host`` (``include/trollout.h``): the environments are independent, so the batch
is cut into pieces and the three legs -- host->device copies, the two kernels-with-C-ABI (``tactor_act``,
``tfem_step``) and device->host copies -- run on three CUDA streams: piece i+1 is uploading while piece i computes
and piece i-1 downloads (PCIe is full duplex).  PyTorch only provides the pinned host buffers here.

``HostRollout(env, [actor0, actor1, actor2])`` runs the driver's whole inner step in one call
(``trollout_step_agents_host``): every agent acts on the same parent and steps its own child
(``master_DDPG_truss2D_MO.py:249-260``), and the parent crosses the link once instead of once per agent.

``MixedHostRollout(mix_env, actors)`` does the same over a ``batched_env.MixedTrussEnv``, the training driver's batch
of episodes of different shapes and truss types (``trollout_step_host_mixed`` / ``trollout_step_agents_host_mixed``):
the state tuple carries each environment's family id as ``"family"``.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import capi

STATE_IN = ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "move_range")
STATE_OUT = ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "move_range", "point", "status")
# compact copies of the two table columns ``_set_model`` reads (``nN_x_n[:, :, 1]``, ``nN_x_e[:, :, 0]``): a state tuple
# that carries them uploads 208 instead of 3 792 bytes per small environment for the two raw tables
COMPACT = ("node_y", "element_section")
ROLLOUT_EXPORTS = ("trollout_last_error", "trollout_create", "trollout_destroy", "trollout_step_host",
                   "trollout_bytes_per_env", "trollout_forget_buffers", "trollout_set_pieces", "trollout_create_agents",
                   "trollout_step_agents_host", "trollout_step_host_mixed", "trollout_step_agents_host_mixed")
MAX_AGENTS = 3                                   # TROLLOUT_MAX_AGENTS


class _State(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in STATE_IN + COMPACT]


class _IO(C.Structure):
    _fields_ = [("inp", _State), ("coin", C.c_void_p), ("x_p", C.c_void_p), ("A_p", C.c_void_p), ("n_pf", C.c_void_p),
                ("P", C.c_int32), ("out", _State), ("point", C.c_void_p), ("status", C.c_void_p),
                ("a_geo", C.c_void_p), ("a_topo", C.c_void_p)]


class _Child(C.Structure):
    _fields_ = [("out", _State), ("coin", C.c_void_p), ("point", C.c_void_p), ("status", C.c_void_p),
                ("a_geo", C.c_void_p), ("a_topo", C.c_void_p)]


class _AgentsIO(C.Structure):
    _fields_ = [("inp", _State), ("x_p", C.c_void_p), ("A_p", C.c_void_p), ("n_pf", C.c_void_p), ("P", C.c_int32),
                ("child", _Child * MAX_AGENTS)]


_lib = capi.lib
_lib.trollout_last_error.restype = C.c_char_p
_lib.trollout_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
_lib.trollout_destroy.argtypes = [C.c_void_p]
_lib.trollout_create_agents.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
_lib.trollout_step_host.argtypes = [C.c_void_p, C.c_int, C.POINTER(_IO), C.c_float, C.c_float, C.c_float, C.c_uint64]
_lib.trollout_step_agents_host.argtypes = [C.c_void_p, C.c_int, C.POINTER(_AgentsIO), C.POINTER(C.c_float),
                                           C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint64)]
_lib.trollout_step_host_mixed.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(_IO), C.c_float, C.c_float,
                                          C.c_float, C.c_uint64]
_lib.trollout_step_agents_host_mixed.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(_AgentsIO),
                                                 C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float),
                                                 C.POINTER(C.c_uint64)]
_lib.trollout_bytes_per_env.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
_lib.trollout_forget_buffers.argtypes = [C.c_void_p]
_lib.trollout_set_pieces.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.c_int]


def _check(rc):
    if rc != 0:
        raise capi.TfemError("libtfem rollout error %d: %s" % (rc, _lib.trollout_last_error().decode()))


def _hp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class HostRollout:
    """``env``: BatchedTrussEnv (family, device), ``actor``: BatchedActor of the env's node count on the same device, or
    a list of 1..3 distinct such actors (the driver's agents, stepped together by :meth:`step_agents`); ``pieces``: how many
    pieces the batch is cut into (each should still fill the GPU: about 148 tiles of 128 actor rows, i.e. ~1000
    small / ~500 large environments), or a list of piece sizes (multiples of 32 but the last, adding up to the batch):
    a small first piece starts the downloads -- the longest of the three legs -- early.  ``"auto"`` (default): about 5.7 MB of
    download per piece, at most 8 pieces -- the optimum measured with the zero-copy transfer kernels of the captured step
    (6 pieces for 4096 small bridges; ``profiles/README.md``); 2 when ``TROLLOUT_ZEROCOPY=0`` sends every array through the
    copy engines, whose per-copy cost makes more pieces a loss.  With several agents "auto" counts the download of one
    child, which is what one transfer of a piece carries: the pieces are those of a one-agent rollout."""

    _mixed = False                             # steps through the _mixed calls (MixedHostRollout)

    def __init__(self, env, actor, pieces="auto"):
        self.env, self.actor = env, actor
        self.actors = list(actor) if isinstance(actor, (list, tuple)) else [actor]
        self._h = C.c_void_p()
        if len(getattr(env, "specs", ())) > 1 and not self._mixed:
            raise capi.TfemError("the env batch holds several families (%d): step it with MixedHostRollout"
                                 % len(env.specs))
        for a in self.actors:                  # the actor ABI cannot tell its node count or device: checked here
            if getattr(a, "nodes", None) != env.N or getattr(a, "device", None) != env.device:
                raise ValueError("every actor must be a BatchedActor of the env's %d nodes on %s (got %s nodes on %s)"
                                 % (env.N, env.device, getattr(a, "nodes", None), getattr(a, "device", None)))
        auto = isinstance(pieces, str)
        if auto and pieces != "auto":
            raise ValueError("pieces: an int, a list of sizes or 'auto'")
        sizes = None if (auto or isinstance(pieces, int)) else [int(v) for v in pieces]
        n0 = 1 if (sizes or auto) else int(pieces)
        with torch.cuda.device(env.device):
            if isinstance(actor, (list, tuple)):
                hs = (C.c_void_p * max(1, len(self.actors)))(*[a._h.value for a in self.actors])
                _check(_lib.trollout_create_agents(env.handle.ptr, hs, len(self.actors), env.B, n0, C.byref(self._h)))
            else:
                _check(_lib.trollout_create(env.handle.ptr, actor._h, env.B, n0, C.byref(self._h)))
        if auto:
            pieces = 2
            if os.environ.get("TROLLOUT_ZEROCOPY", "1") != "0":
                down = C.c_size_t()
                _check(_lib.trollout_bytes_per_env(self._h, 1, 1, None, C.byref(down)))
                down = down.value // len(self.actors)
                pieces = max(1, min(8, int(round(env.B * down / 5.7e6))))
            pieces = max(1, min(pieces, env.B // 128)) if env.B >= 128 else 1
            step = -(-(-(-env.B // pieces)) // 32) * 32
            sizes = []
            while sum(sizes) < env.B:
                sizes.append(min(step, env.B - sum(sizes)))
        if sizes:
            if sum(sizes) != env.B:
                raise ValueError("the piece sizes must add up to the batch (%d)" % env.B)
            _check(_lib.trollout_set_pieces(self._h, (C.c_int32 * len(sizes))(*sizes), len(sizes)))
            edges = [0]
            for v in sizes:
                edges.append(edges[-1] + v)
            self.ranges = list(zip(edges[:-1], edges[1:]))
        else:
            step = -(-env.B // max(1, int(pieces)))
            step = -(-step // 32) * 32
            self.ranges = [(lo, min(lo + step, env.B)) for lo in range(0, env.B, step)]

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.trollout_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def alloc_host(self, compact: bool = True, raw_tables: bool = True):
        """pinned host buffers for one state tuple (+ point, status, actions); ``compact``: also the compact copies of
        the two live table columns (``COMPACT``), which the next step uploads instead of the full raw tables;
        ``raw_tables=False`` (needs ``compact``): a state tuple WITHOUT ``nN_x_n`` / ``nN_x_e`` -- the driver only ever feeds
        them back into ``_game_modify`` / ``_set_model`` (``master_DDPG_truss2D_MO.py:250-260, 755``), which read one column
        of each, so the compact columns carry everything it uses and the step downloads 3.8 KB less per small environment"""
        env = self.env
        if not raw_tables and not compact:
            raise ValueError("a state tuple without the raw tables needs their compact columns")
        h = {k: torch.empty(getattr(env, k).shape, dtype=getattr(env, k).dtype).pin_memory() for k in STATE_OUT
             if raw_tables or k not in ("nN_x_n", "nN_x_e")}
        h["a_geo"] = torch.empty(env.B, env.N, 2).pin_memory()
        h["a_topo"] = torch.empty(env.B, env.N, 3).pin_memory()
        if compact:
            h["node_y"] = torch.empty(env.B, env.N).pin_memory()
            h["element_section"] = torch.empty(env.B, env.E).pin_memory()
        return h

    def alloc_host_children(self, compact: bool = True, raw_tables: bool = True):
        """one :meth:`alloc_host` output set per agent: the ``outs_host`` of :meth:`step_agents`"""
        return [self.alloc_host(compact, raw_tables) for _ in self.actors]

    @staticmethod
    def fill_compact(state_host: dict):
        """(re)derive the compact columns of a host state tuple from its raw tables (after the caller edited them)"""
        state_host["node_y"].copy_(state_host["nN_x_n"][:, :, 1])
        state_host["element_section"].copy_(state_host["nN_x_e"][:, :, 0])

    def forget_buffers(self):
        """drop the CUDA graphs cached for host buffers seen so far (call before freeing such buffers)"""
        _check(_lib.trollout_forget_buffers(self._h))

    def bytes_per_step(self, P: int = 1, compact: bool = True, raw_tables: bool = True):
        a, b = C.c_size_t(), C.c_size_t()
        _check(_lib.trollout_bytes_per_env(self._h, int(P), 1 if compact else 0, C.byref(a), C.byref(b)))
        down = b.value - (0 if raw_tables else len(self.actors) * 4 * (12 * self.env.N + 21 * self.env.E))
        return a.value * self.env.B, down * self.env.B

    def _shapes(self, P):
        B, N, E = self.env.B, self.env.N, self.env.E
        return {"x_n": (B, N, 13), "A_s": (B, N, N), "A_n_ts": (B, N, N), "A_n_cs": (B, N, N), "nN_x_n": (B, N, 12),
                "nN_x_e": (B, E, 21), "move_range": (B, N, 2), "point": (B, 4), "a_geo": (B, N, 2), "a_topo": (B, N, 3),
                "node_y": (B, N), "element_section": (B, E)}

    @staticmethod
    def _chk(t, shape, dtype=torch.float32):
        if not (isinstance(t, torch.Tensor) and t.device.type == "cpu" and t.dtype == dtype
                and tuple(t.shape) == shape and t.is_contiguous()):
            raise ValueError("expected a contiguous host %s tensor of shape %s" % (dtype, shape))
        return _hp(t)

    def _parent(self, io, state_host, x_p_host, A_p_host, n_pf_host):
        """the parent half of the call: state tuple, Pareto-front graph"""
        B, P = self.env.B, int(x_p_host.shape[1])
        shapes, chk = self._shapes(P), self._chk
        compact_in = all(k in state_host for k in COMPACT)
        for k in STATE_IN:
            if not (compact_in and k in ("nN_x_n", "nN_x_e")):     # not read when the compact columns travel
                setattr(io.inp, k, chk(state_host[k], shapes[k]))
        if compact_in:
            for k in COMPACT:
                setattr(io.inp, k, chk(state_host[k], shapes[k]))
        io.x_p, io.A_p, io.P = chk(x_p_host, (B, P, 4)), chk(A_p_host, (B, P, P)), P
        io.n_pf = chk(n_pf_host, (B,), torch.int32) if n_pf_host is not None else C.c_void_p(0)

    def _child(self, blk, out_host, coin_host):
        """one child block: the coin and the outputs (a ``_Child``, or the child half of an ``_IO``)"""
        B = self.env.B
        shapes, chk = self._shapes(1), self._chk
        if not isinstance(out_host, dict):
            raise ValueError("an output set is a dict of host tensors (HostRollout.alloc_host)")
        compact_out = all(k in out_host for k in COMPACT)
        for k in STATE_IN:
            if k in out_host:
                setattr(blk.out, k, chk(out_host[k], shapes[k]))
            elif not (compact_out and k in ("nN_x_n", "nN_x_e")):
                raise ValueError("out_host lacks %r (only the raw tables may be left out, when their compact columns are there)" % k)
        for k in COMPACT:
            if k in out_host:
                setattr(blk.out, k, chk(out_host[k], shapes[k]))
        for k in ("point", "status", "a_geo", "a_topo"):
            if k not in out_host:
                raise ValueError("out_host lacks %r" % k)
        blk.coin = chk(coin_host, (B,), torch.uint8) if coin_host is not None else C.c_void_p(0)
        blk.point = chk(out_host["point"], shapes["point"])
        blk.status = chk(out_host["status"], (B,), torch.int32)
        blk.a_geo, blk.a_topo = chk(out_host["a_geo"], shapes["a_geo"]), chk(out_host["a_topo"], shapes["a_topo"])

    def step(self, state_host: dict, coin_host, x_p_host: torch.Tensor, A_p_host: torch.Tensor, out_host: dict,
             n_pf_host=None):
        """state_host[k] for k in STATE_IN, coin_host [B] uint8 (or None), x_p_host [B,P,4], A_p_host [B,P,P] and
        n_pf_host [B] int32 (or None): contiguous HOST tensors (pinned for overlap).  Fills out_host (STATE_OUT +
        a_geo, a_topo) and returns it once the last piece has landed.  A rollout of several actors steps with
        :meth:`step_agents`."""
        if len(self.actors) > 1:
            raise ValueError("this rollout runs %d actors: step it with step_agents" % len(self.actors))
        act = self.actors[0]
        io = _IO()
        self._parent(io, state_host, x_p_host, A_p_host, n_pf_host)
        self._child(io, out_host, coin_host)
        self._step_call(state_host, io, act.mu, act.theta, act.sigma, act.seed)
        act.update_num += 1
        return out_host

    def step_agents(self, state_host: dict, coins_host, x_p_host: torch.Tensor, A_p_host: torch.Tensor, outs_host,
                    n_pf_host=None):
        """every actor acts on the parent ``state_host`` and steps its own child: ``coins_host`` holds one coin tensor
        [B] uint8 (or None) per actor, ``outs_host`` one output set per actor (:meth:`alloc_host_children`); the rest
        as in :meth:`step`.  Child k is bit for bit what :meth:`step` of a rollout of actor k alone gives on the same
        parent with coin k.  Returns ``outs_host`` once the last piece of the last child has landed."""
        K = len(self.actors)
        if len(coins_host) != K or len(outs_host) != K:
            raise ValueError("step_agents needs one coin (or None) and one output set per actor: %d actors, %d coins, "
                             "%d output sets" % (K, len(coins_host), len(outs_host)))
        io = _AgentsIO()
        self._parent(io, state_host, x_p_host, A_p_host, n_pf_host)
        for k in range(K):
            self._child(io.child[k], outs_host[k], coins_host[k])
        acts = self.actors
        mu = (C.c_float * K)(*[a.mu for a in acts])
        theta = (C.c_float * K)(*[a.theta for a in acts])
        sigma = (C.c_float * K)(*[a.sigma for a in acts])
        seed = (C.c_uint64 * K)(*[a.seed for a in acts])
        self._step_call(state_host, io, mu, theta, sigma, seed)
        for a in acts:
            a.update_num += 1
        return outs_host

    def _step_call(self, state_host, io, *noise):
        """the C call of one step: an ``_IO`` goes to trollout_step_host, an ``_AgentsIO`` to trollout_step_agents_host"""
        fn = _lib.trollout_step_agents_host if isinstance(io, _AgentsIO) else _lib.trollout_step_host
        with torch.cuda.device(self.env.device):
            _check(fn(self._h, self.env.B, C.byref(io), *noise))


class MixedHostRollout(HostRollout):
    """:class:`HostRollout` over a ``batched_env.MixedTrussEnv``: every environment has its own family (the training
    driver draws a shape and a truss type per episode, ``train/code/master_DDPG_truss2D_MO.py:787-815``), and one call
    steps them all -- one env-step launch per piece and agent over every family.  The host state tuple carries the
    family ids as ``state_host["family"]`` (uint8 [B], indices into ``env.specs``), which :meth:`alloc_host` adds.
    ``step`` / ``step_agents`` copy the parent's ids into every output set that has a ``"family"`` tensor of its own,
    so a child can be fed back as the next parent.  Environment b of a child is bit for bit what a ``HostRollout``
    over a batch of family ``env.specs[family[b]]`` gives with the same pieces.  The ids are read when a captured step
    is replayed: they may be rewritten in the same buffer between steps.  An id out of range sets
    ``capi.STATUS_BAD_FAMILY`` in that environment's ``status``; its other outputs are then unspecified."""

    _mixed = True

    def __init__(self, env, actor, pieces="auto"):
        from .batched_env import MixedTrussEnv
        if not isinstance(env, MixedTrussEnv):
            raise ValueError("MixedHostRollout steps a batched_env.MixedTrussEnv (got %s): use HostRollout"
                             % type(env).__name__)
        super().__init__(env, actor, pieces)

    def alloc_host(self, compact: bool = True, raw_tables: bool = True):
        """:meth:`HostRollout.alloc_host` plus ``"family"``: pinned uint8 [B]"""
        h = super().alloc_host(compact, raw_tables)
        h["family"] = torch.empty(self.env.B, dtype=torch.uint8).pin_memory()
        return h

    def step(self, state_host: dict, coin_host, x_p_host: torch.Tensor, A_p_host: torch.Tensor, out_host: dict,
             n_pf_host=None):
        """:meth:`HostRollout.step`; ``state_host["family"]`` is required"""
        super().step(state_host, coin_host, x_p_host, A_p_host, out_host, n_pf_host)
        self._pass_family(state_host, [out_host])
        return out_host

    def step_agents(self, state_host: dict, coins_host, x_p_host: torch.Tensor, A_p_host: torch.Tensor, outs_host,
                    n_pf_host=None):
        """:meth:`HostRollout.step_agents`; ``state_host["family"]`` is required"""
        super().step_agents(state_host, coins_host, x_p_host, A_p_host, outs_host, n_pf_host)
        self._pass_family(state_host, outs_host)
        return outs_host

    def _step_call(self, state_host, io, *noise):
        fam = state_host.get("family")
        if fam is None:
            raise ValueError("state_host lacks 'family': the uint8 [B] family ids (MixedHostRollout.alloc_host)")
        fam = self._chk(fam, (self.env.B,), torch.uint8)
        fn = _lib.trollout_step_agents_host_mixed if isinstance(io, _AgentsIO) else _lib.trollout_step_host_mixed
        with torch.cuda.device(self.env.device):
            _check(fn(self._h, self.env.B, fam, C.byref(io), *noise))

    @staticmethod
    def _pass_family(state_host, outs_host):
        """every child has its parent's families"""
        fam = state_host["family"]
        for o in outs_host:
            if "family" in o and o["family"].data_ptr() != fam.data_ptr():
                o["family"].copy_(fam)
