"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the node-agent GCN actor forward pass.

Follows ``multimodes_actor.call`` (``train/code/truss2D_RL.py:75-127``) with spektral 1.2.0's published
``GCNConv`` (``output = A . (X . W) + b``, ``use_bias=True``, no activation) and ``GlobalSumPool`` (sum over
the node axis); ``act`` adds Ornstein-Uhlenbeck noise to every entry (``:41-48, 328-354``).

Parity status: **unpinned** -- TensorFlow / spektral are not installable here and the reference holds no
recorded actor output, so this restatement can only be checked against itself (shapes, determinism,
float32 CUDA vs float64 numpy agreement).  SURVEY.md section 8c.
"""
from __future__ import annotations

import numpy as np


def _gcn(X, A, W, b):
    return np.matmul(A, np.matmul(X, W)) + b


def _relu(x):
    return np.maximum(x, 0)


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def actor_forward(weights, x_n, A_n, A_s, A_n_ts, A_n_cs, x_p, A_p, n_pf=None, dtype=np.float64, operand_max=False):
    """Batched forward.  x_n [B,N,13]; A_* [B,N,N] (A_n may be [N,N]); x_p [B,P,4]; A_p [B,P,P];
    n_pf [B] = number of valid Pareto rows (rows >= n_pf[b] are ignored, i.e. ``act`` on the unpadded
    graph).  Returns (geo [B,N,2], topo [B,N,3]).

    ``operand_max=True``: returns (geo, topo, m) with the largest |entry| over the batch of the operands the CUDA kernel
    splits into fp16 hi + lo (DESIGN.md section 3.3): m["Z"] for Z = A_n x_n (layer 1's input), m["layer2"] for the
    inputs X and the products Y = A X of the five mixes ``gcn_l2_*`` (X is x11, x12, x13 or the scrambled Pareto
    embedding) and m["layer3"] for those of the two mixes ``gcn_l3_*`` (X is the five-way sum)."""
    w = {k: (np.asarray(a, dtype=dtype), np.asarray(b, dtype=dtype)) for k, (a, b) in weights.items()}
    x_n = np.asarray(x_n, dtype=dtype)
    B, N, _ = x_n.shape
    A_n = np.broadcast_to(np.asarray(A_n, dtype=dtype), (B, N, N))
    A_s, A_ts, A_cs = (np.asarray(a, dtype=dtype) for a in (A_s, A_n_ts, A_n_cs))
    x_p, A_p = np.asarray(x_p, dtype=dtype), np.asarray(A_p, dtype=dtype)
    x11 = _relu(_gcn(x_n, A_n, *w["gcn_l1_1"]))
    x12 = _relu(_gcn(x_n, A_n, *w["gcn_l1_2"]))
    x13 = _relu(_gcn(x_n, A_n, *w["gcn_l1_3"]))
    x14 = _relu(_gcn(x_p, A_p, *w["gcn_l1_4"]))                     # [B,P,H]
    if n_pf is not None:
        valid = (np.arange(x_p.shape[1])[None, :] < np.asarray(n_pf)[:, None]).astype(dtype)
        x14 = x14 * valid[:, :, None]
    pooled = x14.sum(axis=1)                                         # GlobalSumPool -> [B,H]
    H = pooled.shape[1]
    # tf.ragged.stack([pooled]*N, axis=-1) -> [B,H,N]; tf.reshape(..., (B,N,H)): NOT a transpose (:89-95)
    x14b = np.stack([pooled] * N, axis=-1).reshape(B, N, H)
    x21 = _relu(_gcn(x11, A_n, *w["gcn_l2_1"]))
    x22 = _relu(_gcn(x12, A_ts, *w["gcn_l2_2"]))
    x23 = _relu(_gcn(x12, A_cs, *w["gcn_l2_3"]))
    x24 = _relu(_gcn(x13, A_s, *w["gcn_l2_4"]))
    x25 = _relu(_gcn(x14b, A_n, *w["gcn_l2_5"]))
    s = x21 + x22 + x23 + x24 + x25
    x31 = _relu(_gcn(s, A_n, *w["gcn_l3_1"]))
    x32 = _relu(_gcn(s, A_s, *w["gcn_l3_2"]))
    geo = _sigmoid(_gcn(x31, A_n, *w["gcn_l4_1"]))
    topo = _sigmoid(_gcn(x32, A_n, *w["gcn_l4_2"]))
    if not operand_max:
        return geo, topo
    amax = lambda t: float(np.abs(t).max()) if t.size else 0.0      # noqa: E731
    mix = lambda *pairs: max(max(amax(X), amax(np.matmul(A, X))) for A, X in pairs)      # noqa: E731
    return geo, topo, {"Z": amax(np.matmul(A_n, x_n)),
                       "layer2": mix((A_n, x11), (A_ts, x12), (A_cs, x12), (A_s, x13), (A_n, x14b)),
                       "layer3": mix((A_n, s), (A_s, s))}


def rescale_weights(weights, k):
    """The same network with its hidden activations scaled by 2^k: layer 1 (``gcn_l1_1..4``, the Pareto branch included)
    and the hidden biases (``gcn_l2_*``, ``gcn_l3_*``) times 2^k, the output-head kernels (``gcn_l4_*``) times 2^-k.  ReLU
    is positively homogeneous and the factors are powers of two, so the function is unchanged (exactly, barring float32
    overflow or underflow of the weights); what moves is the magnitude of every activation between the input and the
    heads -- the operands of the kernel's fp16 split."""
    c = 2.0 ** int(k)
    out = {}
    for name, (W, b) in weights.items():
        W, b = np.asarray(W, np.float32), np.asarray(b, np.float32)
        if name.startswith("gcn_l1_"):
            W, b = W * np.float32(c), b * np.float32(c)
        elif name.startswith(("gcn_l2_", "gcn_l3_")):
            b = b * np.float32(c)
        elif name.startswith("gcn_l4_"):
            W = W * np.float32(1.0 / c)
        out[name] = (W.astype(np.float32), b.astype(np.float32))
    return out


# ---- the OU noise of the CUDA kernel (``ou_step`` in tactor_tc.cuh), restated in numpy uint64 arithmetic -------------
_M64 = 0xFFFFFFFFFFFFFFFF


def mix64(z):
    """SplitMix64's output function of state ``z`` (uint64, scalar or array; arithmetic wraps mod 2^64)"""
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def ou_noise(seed, call, stream_id, idx):
    """the standard normal the kernel draws for element ``idx`` of tensor ``stream_id`` (1 = geo, 2 = topo) in call
    ``call`` of a handle seeded with ``seed``: a SplitMix64 hash of the four, u1 and u2 formed in float32 exactly as the
    device forms them, then Box-Muller in float64"""
    idx = np.asarray(idx, dtype=np.uint64)
    with np.errstate(over="ignore"):
        key = mix64(np.uint64(int(seed) & _M64) ^ np.uint64((int(call) * 0xD1342543DE82EF95) & _M64))
        h = mix64(key + np.uint64((int(stream_id) * 0x632BE59BD9B4E019) & _M64) + idx)
    c = np.float32(2.3283064365386963e-10)
    u1 = ((h >> np.uint64(32)).astype(np.uint32).astype(np.float32) + np.float32(1.0)) * c      # (0, 1]
    u2 = (h & np.uint64(0xFFFFFFFF)).astype(np.uint32).astype(np.float32) * c
    two_u2 = (np.float32(2.0) * u2).astype(np.float64)
    return np.sqrt(-2.0 * np.log(u1.astype(np.float64))) * np.cos(np.pi * two_u2)


def ou_expected(x, mu, theta, sigma, seed, call, stream_id, idx):
    """``act``'s output for noise-free value ``x``: x + (theta (mu - x) 1e-4 + sigma n), n = ou_noise(...), in float64"""
    x = np.asarray(x, dtype=np.float64)
    n = ou_noise(seed, call, stream_id, idx)
    return x + (theta * (mu - x) * 1e-4 + sigma * n)


class OUNoise:
    """``OUNoise.gen_noise`` (truss2D_RL.py:41-48): theta*(mu-x)*dt + sigma*np.random.randn(1)"""

    def __init__(self, mu, theta, sigma, rng=None):
        self.mu, self.theta, self.sigma, self.dt = mu, theta, sigma, 0.0001
        self.rng = rng if rng is not None else np.random

    def gen_noise(self, x):
        return self.theta * (self.mu - x) * self.dt + self.sigma * self.rng.randn(1)


def act(weights, state, mu=0.1, theta=0.1, sigma=0.1, rng=None):
    """``multimodals_OneAgent.act`` for ONE environment: forward + OU noise on every entry, drawn
    row-major geo first then topo (truss2D_RL.py:341-350).  Returns float32 arrays like the reference."""
    x_n, A_n, A_s, A_ts, A_cs, x_p, A_p = state
    geo, topo = actor_forward(weights, x_n[None], A_n[None], A_s[None], A_ts[None], A_cs[None], x_p[None], A_p[None],
                              dtype=np.float32)
    geo, topo = geo[0].astype(np.float32), topo[0].astype(np.float32)
    ng, nt = OUNoise(mu, theta, sigma, rng), OUNoise(mu, theta, sigma, rng)
    for i in range(geo.shape[0]):
        for j in range(geo.shape[1]):
            geo[i, j] += ng.gen_noise(geo[i, j])[0]
    for i in range(topo.shape[0]):
        for j in range(topo.shape[1]):
            topo[i, j] += nt.gen_noise(topo[i, j])[0]
    return geo, topo
