"""CPU: the pieces of the actor oracle the GPU contract tests lean on -- the restated OU noise hash, the moments of its
normals, and the function-preserving power-of-two rescaling that moves the actor's activations across the fp16 range."""
import os

import numpy as np
import pytest

from oracle.actor_oracle import actor_forward, mix64, ou_expected, ou_noise, rescale_weights

KS = list(range(-12, 15))


def test_mix64_is_splitmix64():
    # the first output of SplitMix64 from state 0 (Vigna's reference splitmix64.c)
    assert int(mix64(0)) == 0xE220A8397B1DCDAF
    # the state advances by the golden-ratio increment: the second output is mix64 of state 0x9E3779B97F4A7C15
    assert int(mix64(0x9E3779B97F4A7C15)) == 0x6E789E6AA1B965F4
    z = np.array([0, 1, 2**63, 2**64 - 1], dtype=np.uint64)
    assert mix64(z).dtype == np.uint64 and [int(v) for v in mix64(z)] == [int(mix64(int(v))) for v in z]


def test_ou_noise_moments():
    idx = np.arange(10**6, dtype=np.uint64)
    for seed, call, stream in ((20, 0, 1), (7, 3, 2)):
        n = ou_noise(seed, call, stream, idx)
        assert np.isfinite(n).all()
        assert abs(n.mean()) < 5e-3 and abs(n.std() - 1.0) < 5e-3
        assert abs(np.mean(n ** 3)) < 2e-2 and abs(np.mean(n ** 4) - 3.0) < 5e-2
    # different keys give unrelated streams
    a, b = ou_noise(20, 0, 1, idx[:4096]), ou_noise(20, 1, 1, idx[:4096])
    c, d = ou_noise(20, 0, 2, idx[:4096]), ou_noise(21, 0, 1, idx[:4096])
    for other in (b, c, d, ou_noise(20, 0, 1, idx[1:4097])):
        assert abs(np.corrcoef(a, other)[0, 1]) < 0.05
    x = np.linspace(0, 1, 9)
    np.testing.assert_array_equal(ou_expected(x, 0.1, 0.0, 0.0, 20, 0, 1, np.arange(9)), x)
    np.testing.assert_allclose(ou_expected(x, 0.1, 0.5, 0.0, 20, 0, 1, np.arange(9)) - x, 0.5 * (0.1 - x) * 1e-4, rtol=0, atol=1e-15)


def _trained(agent):
    from mop_truss_marl_b200 import tf_checkpoint
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "actor_2000pickle_base.npz"))
    return {n: (z["agent%d/%s/kernel" % (agent, n)], z["agent%d/%s/bias" % (agent, n)]) for n in tf_checkpoint.ACTOR_LAYERS}


def _golden_inputs(family, P, seed):
    from util import load_golden
    from oracle.truss_oracle import pareto_state_data
    g = load_golden(family)
    x_n = np.concatenate([g["reset_x_n"][None], g["tr_out_x_n"]]).astype(np.float32)
    A_s = np.concatenate([g["reset_A_s"][None], g["tr_out_A_s"]]).astype(np.float32)
    A_ts = np.concatenate([g["reset_A_n_ts"][None], g["tr_out_A_n_ts"]]).astype(np.float32)
    A_cs = np.concatenate([g["reset_A_n_cs"][None], g["tr_out_A_n_cs"]]).astype(np.float32)
    B = x_n.shape[0]
    rng = np.random.RandomState(seed)
    x_p, A_p = np.zeros((B, P, 4), np.float32), np.zeros((B, P, P), np.float32)
    for b in range(B):
        n = int(rng.randint(1, P + 1))
        o1, o2 = np.sort(rng.rand(n)).astype(np.float32), np.sort(rng.rand(n))[::-1].astype(np.float32)
        x_p[b, :n], A_p[b, :n, :n] = pareto_state_data([(o1[i], o2[i]) for i in range(n)], index=int(rng.randint(0, n)))
    return x_n, g["A_n"].astype(np.float32), A_s, A_ts, A_cs, x_p, A_p


def _random_inputs(B, N, P, seed):
    rng = np.random.RandomState(seed)
    A = (rng.rand(B, N, N) < 0.3).astype(np.float32)
    A = np.maximum(A, A.transpose(0, 2, 1))
    return (rng.rand(B, N, 13).astype(np.float32), (rng.rand(N, N) * 0.3).astype(np.float32),
            (A * rng.rand(B, N, N)).astype(np.float32), (A * rng.rand(B, N, N)).astype(np.float32),
            (A * rng.rand(B, N, N)).astype(np.float32), rng.rand(B, P, 4).astype(np.float32),
            (rng.rand(B, P, P) * 0.5).astype(np.float32))


@pytest.mark.parametrize("case", ["trained1_small_bridge", "trained3_large_roof", "random"])
def test_rescale_weights_preserves_the_function(case):
    from mop_truss_marl_b200 import tf_checkpoint
    if case == "random":
        w = tf_checkpoint.random_actor_weights(seed=3)
        rng = np.random.RandomState(1)
        w = {k: (a, (rng.randn(*b.shape) * 0.05).astype(np.float32)) for k, (a, b) in w.items()}
        inp = _random_inputs(24, 16, 5, 2)
    else:
        agent, family = int(case[7]), case[9:]
        w = _trained(agent)
        inp = _golden_inputs(family, 17, agent)
    g0, t0, m0 = actor_forward(w, *inp, operand_max=True)
    e32 = []
    for k in KS:
        wk = rescale_weights(w, k)
        assert set(wk) == set(w)
        g, t, m = actor_forward(wk, *inp, operand_max=True)
        assert max(np.abs(g - g0).max(), np.abs(t - t0).max()) <= 1e-12, k
        assert m["Z"] == m0["Z"]                                  # layer 1's input does not move
        for key in ("layer2", "layer3"):                          # every split operand behind it does
            assert m[key] == pytest.approx(m0[key] * 2.0 ** k, rel=1e-9)
        g32, t32 = actor_forward(wk, *inp, dtype=np.float32)
        e32.append(max(np.abs(g32 - g).max(), np.abs(t32 - t).max()))
    # the float32 restatement does not care about the scale: its error stays flat across k
    assert max(e32) <= 1e-5 and max(e32) <= 4 * min(e32) + 1e-7, e32
