"""GPU: batched actor forward (libtfem tactor_*) against the numpy restatement in float64.

The actor has no recorded outputs in the reference (parity unpinned, SURVEY.md section 8c): the bar here
is float32-GEMM agreement with the float64 oracle of the same restated network (|delta| <= 2e-5 on the
sigmoid outputs), plus determinism and the statistics of the OU noise."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ATOL = 2e-5


def random_inputs(rng, B, N, P):
    x_n = rng.rand(B, N, 13).astype(np.float32)
    A = (rng.rand(B, N, N) < 0.3).astype(np.float32)
    A = np.maximum(A, A.transpose(0, 2, 1))
    A_s = (A * rng.rand(B, N, N)).astype(np.float32)
    A_ts = (A * rng.rand(B, N, N) * (rng.rand(B, N, N) < 0.5)).astype(np.float32)
    A_cs = (A * rng.rand(B, N, N) * (rng.rand(B, N, N) < 0.5)).astype(np.float32)
    A_n = rng.rand(N, N).astype(np.float32) * 0.3
    x_p = rng.rand(B, P, 4).astype(np.float32)
    A_p = (rng.rand(B, P, P) * 0.5).astype(np.float32)
    return x_n, A_n, A_s, A_ts, A_cs, x_p, A_p


@pytest.mark.parametrize("N,B,P", [(16, 37, 1), (16, 64, 7), (32, 9, 50), (32, 32, 3), (16, 21, 8), (16, 21, 9), (16, 12, 27), (32, 10, 16), (16, 10, 17)])
def test_forward_matches_float64_oracle(N, B, P):
    from mop_truss_marl_b200 import actor, tf_checkpoint
    from oracle.actor_oracle import actor_forward
    rng = np.random.RandomState(N + B)
    w = tf_checkpoint.random_actor_weights(seed=3)
    for k in w:                                      # non-zero biases
        w[k] = (w[k][0], (rng.randn(*w[k][1].shape) * 0.05).astype(np.float32))
    inp = random_inputs(rng, B, N, P)
    n_pf = rng.randint(1, P + 1, size=B).astype(np.int32)
    a = actor.BatchedActor(w, N, max_batch=B)
    dev = [torch.from_numpy(t).cuda() for t in inp]
    geo, topo = a.forward(*dev, n_pf=torch.from_numpy(n_pf).cuda())
    torch.cuda.synchronize()
    g64, t64 = actor_forward(w, *inp, n_pf=n_pf)
    assert geo.shape == (B, N, 2) and topo.shape == (B, N, 3)
    assert np.abs(geo.cpu().numpy() - g64).max() <= ATOL
    assert np.abs(topo.cpu().numpy() - t64).max() <= ATOL
    # determinism + n_pf=None means "all P rows"
    geo2, topo2 = a.forward(*dev, n_pf=torch.from_numpy(n_pf).cuda())
    assert torch.equal(geo, geo2) and torch.equal(topo, topo2)
    g3, t3 = a.forward(*dev)
    g64b, t64b = actor_forward(w, *inp)
    assert np.abs(g3.cpu().numpy() - g64b).max() <= ATOL and np.abs(t3.cpu().numpy() - t64b).max() <= ATOL
    # launches per forward: Pareto branch (one-row kernel, or tridiagonal kernel + dense second pass) + fused network
    assert a.launch_count() == 3 * (2 if P == 1 else 3)
    a.check()


def truss_mask(N):
    """Adjacency pattern (with self loops) of the reference's num_x x 2 trusses: chords, verticals, both diagonals."""
    nx = N // 2
    m = np.eye(N, dtype=np.float32)
    for i in range(nx):
        for j in range(nx):
            if abs(i - j) <= 1:
                m[i, j] = m[nx + i, nx + j] = m[i, nx + j] = m[nx + j, i] = 1
    return m


@pytest.mark.parametrize("N,B,P,stray", [(16, 37, 3, False), (32, 21, 2, False), (16, 19, 1, True), (32, 6, 5, True)])
def test_forward_truss_structured_adjacency(N, B, P, stray):
    """The kernel's compacted-neighbour path (rows with <= 8 entries inside A_n's pattern), and the fall-back to the
    full row when one environment has an entry outside that pattern (stray)."""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    from oracle.actor_oracle import actor_forward
    rng = np.random.RandomState(100 + N + B)
    w = tf_checkpoint.random_actor_weights(seed=5)
    for k in w:
        w[k] = (w[k][0], (rng.randn(*w[k][1].shape) * 0.05).astype(np.float32))
    inp = list(random_inputs(rng, B, N, P))
    m = truss_mask(N)
    off = m - np.eye(N, dtype=np.float32)
    inp[1] = ((rng.rand(N, N) * 0.3 + 0.05) * m).astype(np.float32)
    for i in (2, 3, 4):
        inp[i] = (rng.rand(B, N, N) * (rng.rand(B, N, N) < 0.7) * off).astype(np.float32)
    if stray:
        inp[3][B // 2, 0, N - 1] = 0.37                  # outside the pattern of A_n
        inp[2][B - 1, N - 1, 1] = 0.11
    a = actor.BatchedActor(w, N, max_batch=B)
    dev = [torch.from_numpy(np.ascontiguousarray(t)).cuda() for t in inp]
    geo, topo = a.forward(*dev)
    torch.cuda.synchronize()
    g64, t64 = actor_forward(w, *inp)
    assert np.abs(geo.cpu().numpy() - g64).max() <= ATOL
    assert np.abs(topo.cpu().numpy() - t64).max() <= ATOL
    a.check()


def test_act_noise_statistics():
    from mop_truss_marl_b200 import actor, tf_checkpoint
    rng = np.random.RandomState(0)
    N, B = 16, 2048
    w = tf_checkpoint.random_actor_weights(seed=1)
    inp = [torch.from_numpy(t).cuda() for t in random_inputs(rng, B, N, 1)]
    a = actor.BatchedActor(w, N, max_batch=B, mu=0.1, theta=0.1, sigma=0.1, seed=20)
    geo0, topo0 = a.forward(*inp)
    geo1, topo1 = a.act(*inp)
    geo2, topo2 = a.act(*inp)
    torch.cuda.synchronize()
    d = torch.cat([(geo1 - geo0).flatten(), (topo1 - topo0).flatten()]).double().cpu().numpy()
    drift = (0.1 * (0.1 - torch.cat([geo0.flatten(), topo0.flatten()]).double().cpu().numpy()) * 1e-4)
    z = (d - drift) / 0.1
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1.0) < 0.02
    assert abs(np.mean(z ** 3)) < 0.05 and abs(np.mean(z ** 4) - 3.0) < 0.1
    assert not torch.equal(geo1, geo2)               # a new call draws new noise
    assert a.update_num == 2


def test_set_weights_and_learner_round_trip():
    """tactor_set_weights on a live handle; the PyTorch learner's ActorNet (the differentiable twin used for the DDPG
    update) and the CUDA kernel agree before and after a training step."""
    from mop_truss_marl_b200 import actor, learner, tf_checkpoint
    rng = np.random.RandomState(7)
    N, B = 16, 24
    inp = random_inputs(rng, B, N, 2)
    dev = [torch.from_numpy(t).cuda() for t in inp]
    w0 = tf_checkpoint.random_actor_weights(seed=1)
    a = actor.BatchedActor(w0, N, max_batch=B)
    g0, t0 = a.forward(*dev)
    lrn = learner.MADDPGLearner(lr=1e-2, batch_size=8, device="cuda", seed=9)
    net = lrn.agents[0].actor
    a.set_weights(net.export_weights())
    g1, t1 = a.forward(*dev)
    with torch.no_grad():
        gn, tn = net(*dev)
    assert (g1 - gn).abs().max() <= ATOL and (t1 - tn).abs().max() <= ATOL
    assert (g1 - g0).abs().max() > 1e-3                  # the weights really changed
    for _ in range(12):
        s = [t if t.ndim == 2 else t[0] for t in inp]
        lrn.remember(s, [(rng.rand(N, 2).astype(np.float32), rng.rand(N, 3).astype(np.float32)) for _ in range(3)],
                     rng.randn(3).astype(np.float32), [s, s, s], 0)
    assert lrn.train()
    a.set_weights(lrn.actor_weights(0))
    g2, t2 = a.forward(*dev)
    with torch.no_grad():
        gn2, tn2 = net(*dev)
    assert (g2 - gn2).abs().max() <= ATOL and (t2 - tn2).abs().max() <= ATOL
    assert not torch.equal(g2, g1)
    a.check()


@pytest.mark.parametrize("nodes,B", [(16, 300), (16, 100), (32, 150), (16, 2400), (32, 1300), (16, 1600), (16, 1590)])
def test_last_wave_split_is_bit_identical(nodes, B, monkeypatch):
    """tiles of the last partial wave are cut into 2 or 4 row pieces, and with more work items than SMs the kernel is
    persistent (a CTA walks several items with running barrier counters); rows are independent, so the outputs must
    equal those of the plain one-CTA-per-tile launch (TACTOR_NO_SPLIT=1) bit for bit.  B = 2400 / 1300: 312 / 412 items;
    B = 300: two-way pieces of 16-node graphs are laid out half-live (one environment per 32-row group); B = 1600 / 1590:
    148 full tiles followed by 104 half-live pieces in the same CTAs (both generator instantiations in one launch), the
    last piece of 1590 partly past the batch"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    w = tf_checkpoint.random_actor_weights(seed=3)
    g = torch.Generator(device="cuda").manual_seed(1)
    r = lambda *s: torch.rand(*s, device="cuda", generator=g)   # noqa: E731
    sc = 1.0 / nodes                                             # keeps the activations O(1)
    inp = (r(B, nodes, 13), r(nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc,
           r(B, 3, 4), r(B, 3, 3) * 0.3)
    outs = []
    for no_split in ("0", "1"):
        monkeypatch.setenv("TACTOR_NO_SPLIT", no_split)
        pol = actor.BatchedActor(w, nodes, B)
        geo, topo = pol.forward(*inp)
        torch.cuda.synchronize()
        pol.check()
        outs.append((geo.clone(), topo.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert bool(torch.isfinite(outs[0][0]).all()) and 0.0 < float(outs[0][0].min()) and float(outs[0][0].max()) < 1.0


def test_fp16_range_overflow_is_reported():
    """the split tensor-core product carries activations as fp16 hi + lo: an activation beyond 65504 cannot be
    represented and must be reported (tactor_status -> TfemError), never silently returned"""
    from mop_truss_marl_b200 import actor, capi, tf_checkpoint
    nodes, B = 16, 16
    w = tf_checkpoint.random_actor_weights(seed=4)
    g = torch.Generator(device="cuda").manual_seed(5)
    r = lambda *s: torch.rand(*s, device="cuda", generator=g)   # noqa: E731
    sc = 1.0 / nodes
    adj = (r(nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc)
    pol = actor.BatchedActor(w, nodes, B)
    pol.forward(r(B, nodes, 13), *adj, r(B, 1, 4), r(B, 1, 1))
    torch.cuda.synchronize()
    pol.check()                                                  # ordinary inputs: fine
    pol2 = actor.BatchedActor(w, nodes, B)
    pol2.forward(r(B, nodes, 13) * 3e6, *adj, r(B, 1, 4), r(B, 1, 1))
    torch.cuda.synchronize()
    with pytest.raises(capi.TfemError, match="fp16 range"):
        pol2.check()


def test_tmem_store_layout_selftest():
    """the generators write the mma accumulator fragment straight into tensor memory (tcgen05.st.16x128b.x2 at lane offsets
    0 and 16): the layout the kernel assumes is checked on the device itself"""
    from mop_truss_marl_b200 import actor
    actor.selftest_tmem_layout(0)


def trained_weights(agent):
    """the reference's trained actor ``model/2000pickle_base/Agent<agent>_Actor_pickle`` from the committed fixture
    (tests/golden/make_actor_golden.py)"""
    import os
    from mop_truss_marl_b200 import tf_checkpoint
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "actor_2000pickle_base.npz"))
    return {name: (z["agent%d/%s/kernel" % (agent, name)], z["agent%d/%s/bias" % (agent, name)]) for name in tf_checkpoint.ACTOR_LAYERS}


def padded_pareto_graph(rng, B, P, front_sizes):
    """Pareto graphs as the driver feeds them: ``pareto_state_data`` of a front of n points (chain graph, normalised), zero
    rows / columns up to P (``master_DDPG_truss2D_MO.py:499-517``); the network then pools over ALL P rows"""
    from oracle.truss_oracle import pareto_state_data
    x_p = np.zeros((B, P, 4), np.float32)
    A_p = np.zeros((B, P, P), np.float32)
    for b in range(B):
        n = int(front_sizes[b])
        obj1 = np.sort(rng.rand(n)).astype(np.float32)
        obj2 = np.sort(rng.rand(n))[::-1].astype(np.float32)
        x, A = pareto_state_data([(obj1[i], obj2[i]) for i in range(n)], index=int(rng.randint(0, n)))
        x_p[b, :n], A_p[b, :n, :n] = x, A
    return x_p, A_p


@pytest.mark.parametrize("agent", [1, 2, 3])
@pytest.mark.parametrize("family,P", [("small_bridge", 1), ("small_bridge", 17), ("small_roof", 50), ("large_bridge", 50), ("large_roof", 17)])
def test_trained_checkpoint_on_golden_states(agent, family, P):
    """The trained 2000pickle_base actors (the checkpoint every test/ driver loads) on states recorded from the reference
    environment, with Pareto graphs of 1, 17 and 50 rows where the front fills only part of the rows (zero padding).  The
    fp16 hi/lo operand split must stay in range on the real weights (status 0) and agree with the float64 oracle."""
    from mop_truss_marl_b200 import actor
    from oracle.actor_oracle import actor_forward
    from util import load_golden
    g = load_golden(family)
    w = trained_weights(agent)
    rng = np.random.RandomState(100 * agent + P)
    x_n = np.concatenate([g["reset_x_n"][None], g["tr_out_x_n"]]).astype(np.float32)
    A_s = np.concatenate([g["reset_A_s"][None], g["tr_out_A_s"]]).astype(np.float32)
    A_ts = np.concatenate([g["reset_A_n_ts"][None], g["tr_out_A_n_ts"]]).astype(np.float32)
    A_cs = np.concatenate([g["reset_A_n_cs"][None], g["tr_out_A_n_cs"]]).astype(np.float32)
    B, N = x_n.shape[0], x_n.shape[1]
    sizes = rng.randint(1, P + 1, size=B)
    sizes[0] = P                                      # one full front
    x_p, A_p = padded_pareto_graph(rng, B, P, sizes)
    a = actor.BatchedActor(w, N, max_batch=B)
    dev = [torch.from_numpy(np.ascontiguousarray(t)).cuda() for t in (x_n, g["A_n"], A_s, A_ts, A_cs, x_p, A_p)]
    geo, topo = a.forward(*dev)
    a.check()                                         # tactor_status == 0: no activation left the fp16 range
    g64, t64 = actor_forward(w, x_n, g["A_n"], A_s, A_ts, A_cs, x_p, A_p)
    assert np.abs(geo.cpu().numpy() - g64).max() <= ATOL
    assert np.abs(topo.cpu().numpy() - t64).max() <= ATOL
    # both the float32 restatement (what TensorFlow computes in) and the kernel stay within 1e-5 of float64
    g32, t32 = actor_forward(w, x_n, g["A_n"], A_s, A_ts, A_cs, x_p, A_p, dtype=np.float32)
    err_kernel = max(np.abs(geo.cpu().numpy() - g64).max(), np.abs(topo.cpu().numpy() - t64).max())
    err_f32 = max(np.abs(g32 - g64).max(), np.abs(t32 - t64).max())
    assert err_kernel <= 1e-5 and err_f32 <= 1e-5, (err_kernel, err_f32)
    # optional pin against TensorFlow + spektral outputs recorded elsewhere (scripts/make_actor_golden_tf.py)
    import os
    tf_path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "actor_tf.npz")
    if os.path.exists(tf_path):
        z = np.load(tf_path)
        key = "agent%d/%s/P%d" % (agent, family, P)
        if key + "/geo" in z.files:
            gt, tt = actor_forward(w, z[key + "/x_n"], g["A_n"], z[key + "/A_s"], z[key + "/A_n_ts"], z[key + "/A_n_cs"], z[key + "/x_p"], z[key + "/A_p"])
            assert np.abs(gt - z[key + "/geo"]).max() <= 1e-5 and np.abs(tt - z[key + "/topo"]).max() <= 1e-5


@pytest.mark.parametrize("N,B,P", [(16, 70, 2), (16, 33, 16), (16, 45, 17), (32, 20, 50), (16, 64, 50)])
def test_tridiagonal_pareto_branch_is_bit_identical_to_dense(N, B, P, monkeypatch):
    """The Pareto graphs the reference builds are chains (tridiagonal A_p): pareto_tri_kernel takes them, environments with
    an entry outside the band fall back to the dense kernel.  Both give bit-identical outputs on chain graphs (padded and
    full fronts, with and without n_pf), and a batch that mixes chain and dense graphs matches the all-dense run."""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    rng = np.random.RandomState(P + B)
    w = tf_checkpoint.random_actor_weights(seed=5)
    for k in w:
        w[k] = (w[k][0], (rng.randn(*w[k][1].shape) * 0.05).astype(np.float32))
    x_n, A_n, A_s, A_ts, A_cs, _, _ = random_inputs(rng, B, N, P)
    sizes = rng.randint(1, P + 1, size=B)
    x_p, A_p = padded_pareto_graph(rng, B, P, sizes)
    dense_rows = rng.rand(B) < 0.25                        # these environments get a full (non-banded) A_p
    A_p[dense_rows] = (rng.rand(int(dense_rows.sum()), P, P) * 0.3).astype(np.float32)
    n_pf = rng.randint(1, P + 1, size=B).astype(np.int32)
    dev = [torch.from_numpy(np.ascontiguousarray(t)).cuda() for t in (x_n, A_n, A_s, A_ts, A_cs, x_p, A_p)]
    outs = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("TACTOR_PARETO_DENSE", mode)
        a = actor.BatchedActor(w, N, max_batch=B)
        o1 = a.forward(*dev)
        o2 = a.forward(*dev, n_pf=torch.from_numpy(n_pf).cuda())
        torch.cuda.synchronize()
        a.check()
        outs[mode] = [t.clone() for t in (*o1, *o2)]
    for t0, t1 in zip(outs["0"], outs["1"]):
        assert torch.equal(t0, t1)


@pytest.mark.parametrize("nodes,B", [(16, 40), (32, 12)])
def test_set_weights_device_equals_host_path(nodes, B):
    """tactor_set_weights_device rebuilds the operand images (scales, fp16 hi/lo split, core-matrix layout, layer-1 fragment
    image) with kernels: a handle updated from device tensors gives bit-identical outputs to one built from the same
    weights on the host, including weights whose scale exponent differs from the handle's previous ones"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    rng = np.random.RandomState(nodes)
    w_old = tf_checkpoint.random_actor_weights(seed=1)
    w_new = tf_checkpoint.random_actor_weights(seed=2)
    for i, k in enumerate(w_new):                     # different magnitudes per layer -> different power-of-two scales
        w_new[k] = (w_new[k][0] * np.float32(2.0 ** ((i % 5) - 2)), (rng.randn(*w_new[k][1].shape) * 0.05).astype(np.float32))
    g = torch.Generator(device="cuda").manual_seed(3)
    r = lambda *s: torch.rand(*s, device="cuda", generator=g)   # noqa: E731
    sc = 1.0 / nodes
    inp = (r(B, nodes, 13), r(nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc,
           r(B, 5, 4), r(B, 5, 5) * 0.2)
    host = actor.BatchedActor(w_new, nodes, B)
    dev = actor.BatchedActor(w_old, nodes, B)
    dev.forward(*inp)
    dev.set_weights_device({k: (torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.from_numpy(np.ascontiguousarray(b)).cuda())
                            for k, (a, b) in w_new.items()})
    o_host, o_dev = host.forward(*inp), dev.forward(*inp)
    torch.cuda.synchronize()
    host.check(); dev.check()
    assert torch.equal(o_host[0], o_dev[0]) and torch.equal(o_host[1], o_dev[1])
    with pytest.raises(ValueError):
        dev.set_weights_device({k: (torch.from_numpy(a), torch.from_numpy(b)) for k, (a, b) in w_new.items()})   # host tensors


@pytest.mark.parametrize("B,P", [(37, 1), (64, 20), (9, 7)])
def test_twelve_node_graphs_of_the_training_shapes(B, P):
    """The 6 x 2 shapes of train/code have 12 nodes: the handle pads every graph to 16 rows internally (zero features, zero
    adjacency rows / columns), divides the pooled scramble by the real node count and writes [B,12,...] outputs; checked
    against the float64 oracle run on the unpadded 12-node tensors, with the trained checkpoint"""
    from mop_truss_marl_b200 import actor
    from oracle.actor_oracle import actor_forward
    rng = np.random.RandomState(B)
    w = trained_weights(2)
    inp = random_inputs(rng, B, 12, P)
    a = actor.BatchedActor(w, 12, max_batch=B)
    dev = [torch.from_numpy(t).cuda() for t in inp]
    geo, topo = a.forward(*dev)
    a.check()
    g64, t64 = actor_forward(w, *inp)
    assert geo.shape == (B, 12, 2) and topo.shape == (B, 12, 3)
    assert np.abs(geo.cpu().numpy() - g64).max() <= ATOL and np.abs(topo.cpu().numpy() - t64).max() <= ATOL
    geo2, topo2 = a.act(*dev)                              # noise on the 12 real rows only, deterministic per (seed, call)
    assert geo2.shape == (B, 12, 2) and bool(torch.isfinite(topo2).all())


def test_training_shape_closed_loop():
    """actor + env-step on a train/code family (12 nodes, no symmetry step): a short closed loop stays healthy"""
    from mop_truss_marl_b200 import actor, batched_env
    B = 256
    env = batched_env.BatchedTrussEnv("train2_roof", B, device="cuda:0")
    env.reset()
    pol = actor.BatchedActor(trained_weights(1), env.N, B)
    x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 20], device="cuda").repeat(B, 1, 1).contiguous()
    A_p = torch.ones(B, 1, 1, device="cuda")
    for _ in range(6):
        geo, topo = pol.act(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p)
        env.step(geo, topo, (torch.rand(B, device="cuda") >= 0.5).to(torch.uint8))
    torch.cuda.synchronize()
    pol.check()
    assert int(env.status.abs().max()) == 0 and bool(torch.isfinite(env.point).all())
