"""GPU: the actor kernel's contract beyond test_gpu_actor.py.

* accuracy across activation scales: the fp16 hi/lo split either agrees with float64 or reports through tactor_status,
  wherever the activations sit (DESIGN.md section 3.3);
* the OU noise element by element against its numpy restatement (oracle.actor_oracle.ou_noise), on direct calls and
  through the host-resident rollout (direct, capturing and replayed steps);
* whole production batches of env-produced states against float64;
* layout invariants bit for bit: permutation of the environments, prefixes of one handle, nothing read or written past
  row B."""
import json
import os

import numpy as np
import pytest

from test_gpu_actor import padded_pareto_graph, random_inputs, trained_weights

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ATOL = 2e-5
F16_MAX = 65504.0
# the kernel carries the mix operands X and Y = A X of layer 2 times 64, those of layer 3 times 8 (DESIGN.md section 3.3):
# they must stay below 65504 / 64 and 65504 / 8
PRESCALE = {"layer2": 64.0, "layer3": 8.0}


def record(name, data):
    """the measured errors of this file, per case (the numbers DESIGN.md quotes): printed, and merged into
    $ACTOR_CONTRACT_JSON when that variable names a file"""
    print(name, json.dumps(data))
    path = os.environ.get("ACTOR_CONTRACT_JSON")
    if not path:
        return
    try:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        old = json.load(open(path)) if os.path.exists(path) else {}
        old[name] = data
        json.dump(old, open(path, "w"), indent=1)
    except OSError:
        pass


def _dev(arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _err(geo, topo, g64, t64):
    return max(float(np.abs(geo - g64).max()), float(np.abs(topo - t64).max()))


def _raises(pol):
    from mop_truss_marl_b200 import capi
    try:
        pol.check()
        return False
    except capi.TfemError as e:
        assert "fp16 range" in str(e), e
        return True


# ================================================= accuracy across activation scales ====================================
KS = [-12, -10, -8, -6, -4, -2, 0, 2, 4, 8, 12, 14]


def _golden_case(family, P, agent):
    from util import load_golden
    g = load_golden(family)
    x_n = np.concatenate([g["reset_x_n"][None], g["tr_out_x_n"]]).astype(np.float32)
    A_s = np.concatenate([g["reset_A_s"][None], g["tr_out_A_s"]]).astype(np.float32)
    A_ts = np.concatenate([g["reset_A_n_ts"][None], g["tr_out_A_n_ts"]]).astype(np.float32)
    A_cs = np.concatenate([g["reset_A_n_cs"][None], g["tr_out_A_n_cs"]]).astype(np.float32)
    rng = np.random.RandomState(100 * agent + P)
    B = x_n.shape[0]
    sizes = rng.randint(1, P + 1, size=B)
    sizes[0] = P
    x_p, A_p = padded_pareto_graph(rng, B, P, sizes)
    return (x_n, g["A_n"].astype(np.float32), A_s, A_ts, A_cs, x_p, A_p)


SCALE_CASES = [("trained%d" % a, fam, P) for a in (1, 2, 3) for fam in ("small_bridge", "large_roof") for P in (1, 17)]
SCALE_CASES += [("random", "random16", 7), ("random", "random32", 3)]
# the lower edge of the window cannot be reported, only placed: random 32-node weights on dense random graphs already sit at
# 1.7e-5 at k = 0, and at k <= -10 most of their layer-3 operands fall below the window (measured 2.3e-5 / 3.3e-5 at
# k = -10 / -12, DESIGN.md section 3.3), so that case sweeps from k = -8
LOWEST_K = {"random32": -8}


@pytest.mark.parametrize("weights,inputs,P", SCALE_CASES)
def test_accuracy_across_activation_scales(weights, inputs, P):
    """rescale_weights(w, k) moves every activation between layer 1 and the heads by 2^k without changing the function.
    For every k the kernel either reports (check() raises) -- exactly when the float64 forward's largest split operand
    leaves the fp16 window -- or agrees with float64 to 2e-5: never a silent wrong answer."""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    from oracle.actor_oracle import actor_forward, rescale_weights
    if weights == "random":
        rng = np.random.RandomState(11)
        w = tf_checkpoint.random_actor_weights(seed=3)
        w = {k: (a, (rng.randn(*b.shape) * 0.05).astype(np.float32)) for k, (a, b) in w.items()}
        N = int(inputs[6:])
        inp = random_inputs(rng, 48, N, P)
    else:
        w = trained_weights(int(weights[7:]))
        inp = _golden_case(inputs, P, int(weights[7:]))
    B, N = inp[0].shape[0], inp[0].shape[1]
    dev = _dev(inp)
    pol = actor.BatchedActor(w, N, max_batch=B)
    rows, failures = [], []
    for k in [k for k in KS if k >= LOWEST_K.get(inputs, KS[0])]:
        wk = rescale_weights(w, k)
        pol.set_weights(wk)
        geo, topo = pol.forward(*dev)
        raised = _raises(pol)
        g64, t64, m = actor_forward(wk, *inp, operand_max=True)
        g32, t32 = actor_forward(wk, *inp, dtype=np.float32)
        err32 = _err(g32, t32, g64, t64)
        worst = max(m["Z"], m["layer2"] * PRESCALE["layer2"], m["layer3"] * PRESCALE["layer3"]) / F16_MAX
        assert abs(worst - 1.0) > 0.01, "grid point %d sits within 1 %% of the fp16 limit: undecided" % k
        expect_raise = worst > 1.0
        err = None if raised else _err(geo.cpu().numpy(), topo.cpu().numpy(), g64, t64)
        rows.append({"k": k, "operand_max": m, "window_use": worst, "raised": raised, "expect_raise": expect_raise,
                     "err": err, "err_f32": err32, "err/err_f32": None if err is None else err / err32})
        if raised != expect_raise or (err is not None and err > ATOL):
            failures.append(rows[-1])
    record("scale_%s_%s_P%d" % (weights, inputs, P), rows)
    assert not failures, failures
    assert any(r["err"] is not None for r in rows) and any(r["raised"] for r in rows)   # both sides of the window


# ================================================= OU noise, element by element ========================================
def _noise_close(got, x, mu, theta, sigma, seed, call, stream, clip=False):
    """got (kernel act) against ou_expected(x = the noise-free value): 4 float32 ulps of the output plus 2e-6 sigma |n|"""
    from oracle.actor_oracle import ou_expected, ou_noise
    got = np.asarray(got, np.float64).ravel()
    x = np.asarray(x, np.float64).ravel()
    idx = np.arange(x.size, dtype=np.uint64)
    want = ou_expected(x, mu, theta, sigma, seed, call, stream, idx)
    n = ou_noise(seed, call, stream, idx)
    if clip:
        want = np.clip(want, 0.0, 1.0)
    tol = 4 * np.spacing(np.abs(got).astype(np.float32)).astype(np.float64) + 2e-6 * sigma * np.abs(n)
    bad = np.abs(got - want) > tol
    return int(bad.sum()), float(np.abs(got - want).max())


def _assert_noise(out, ref, mu, theta, sigma, seed, call, what, clip=False):
    for hd, (got, x) in enumerate(zip(out, ref)):
        nbad, worst = _noise_close(got.cpu().numpy() if torch.is_tensor(got) else got,
                                   x.cpu().numpy() if torch.is_tensor(x) else x, mu, theta, sigma, seed, call, hd + 1, clip)
        assert nbad == 0, (what, "geo" if hd == 0 else "topo", nbad, worst)


@pytest.mark.parametrize("N,B", [(16, 4096), (32, 8192), (12, 1500)])
def test_act_noise_element_by_element(N, B):
    """act = forward + theta (mu - x) 1e-4 + sigma n(seed, call, tensor, element), element = the flat index of the output
    ([B, N, 2] / [B, N, 3], real rows only for the padded 12-node graphs); consecutive calls draw calls 0, 1, ...; a call
    with sigma = theta = 0 is forward and draws no call index; sigma = 0 leaves the drift alone; n_pf keys the same way"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    rng = np.random.RandomState(N + B)
    w = tf_checkpoint.random_actor_weights(seed=9)
    P = 5
    inp = list(random_inputs(rng, B, N, P))
    for i in (1, 2, 3, 4):
        inp[i] = (inp[i] / N).astype(np.float32)               # keeps the outputs away from saturated 0 / 1
    dev = _dev(inp)
    n_pf = torch.from_numpy(rng.randint(1, P + 1, size=B).astype(np.int32)).cuda()
    mu, theta, sigma = 0.1, 0.15, 0.2
    a = actor.BatchedActor(w, N, max_batch=B, mu=mu, theta=theta, sigma=sigma, seed=20)
    x0 = [t.clone() for t in a.forward(*dev)]
    _assert_noise(a.act(*dev), x0, mu, theta, sigma, 20, 0, "call 0")
    _assert_noise(a.act(*dev), x0, mu, theta, sigma, 20, 1, "call 1")
    a.seed = 0xFEEDFACECAFEBEEF                                # a second seed, next call index
    _assert_noise(a.act(*dev), x0, mu, theta, sigma, a.seed, 2, "seed 2, call 2")
    a.sigma, a.theta = 0.0, 0.0                                # plain forward; no call index drawn
    o = a.act(*dev)
    assert torch.equal(o[0], x0[0]) and torch.equal(o[1], x0[1])
    a.sigma, a.theta = sigma, theta
    _assert_noise(a.act(*dev), x0, mu, theta, sigma, a.seed, 3, "call 3 after a noise-free call")
    a.sigma = 0.0                                              # drift only (draws call 4)
    _assert_noise(a.act(*dev), x0, mu, theta, 0.0, a.seed, 4, "drift only")
    a.sigma = sigma
    xp = [t.clone() for t in a.forward(*dev, n_pf=n_pf)]
    _assert_noise(a.act(*dev, n_pf=n_pf), xp, mu, theta, sigma, a.seed, 5, "n_pf, call 5")
    a.check()


def _parent_forward(twin, env, parent, x_p, A_p, lo, hi):
    """the noise-free actions of one piece of the host parent, from the twin handle"""
    d = lambda t: t[lo:hi].contiguous().to(env.device)          # noqa: E731
    g, t = twin.forward(d(parent["x_n"]), env.A_n, d(parent["A_s"]), d(parent["A_n_ts"]), d(parent["A_n_cs"]), d(x_p), d(A_p))
    return g.cpu().numpy(), t.cpu().numpy()


@pytest.mark.parametrize("agents", [1, 3])
def test_rollout_noise_keys(agents):
    """HostRollout (one agent, step) and step_agents (three actors) over 6 steps with two alternating buffer sets: steps 1, 2
    are issued directly, step 3 (4) captures a CUDA graph for its buffer set and runs it, steps 5, 6 replay.  Every step
    reserves one call index per piece: piece j of step s (0-based) draws call pieces * s + j of its actor, with element
    indices counted from the piece's first environment.  Children's actions are compared after the env step's in-place
    clip to [0, 1] (truss2D_ENV.py:379-391)."""
    from mop_truss_marl_b200 import actor, batched_env, tf_checkpoint
    from mop_truss_marl_b200.host_pipeline import STATE_IN, HostRollout
    B = 600
    env = batched_env.BatchedTrussEnv("small_bridge", B)
    env.reset()
    params = [dict(mu=0.1, theta=0.1 + 0.05 * k, sigma=0.1 + 0.05 * k, seed=100 + 7 * k) for k in range(agents)]
    weights = [tf_checkpoint.random_actor_weights(seed=30 + k) for k in range(agents)]
    pols = [actor.BatchedActor(weights[k], env.N, B, **params[k]) for k in range(agents)]
    twins = [actor.BatchedActor(weights[k], env.N, B, sigma=0.0, theta=0.0) for k in range(agents)]
    roll = HostRollout(env, pols if agents > 1 else pols[0], pieces=3)
    assert len(roll.ranges) == 3 and roll.ranges[-1] == (448, 600)
    parents = [roll.alloc_host(), roll.alloc_host()]
    outs = [roll.alloc_host_children() for _ in range(2)] if agents > 1 else None
    for k in STATE_IN:
        parents[0][k].copy_(getattr(env, k))
    roll.fill_compact(parents[0])
    g = torch.Generator().manual_seed(5)
    P = 3
    x_p = torch.rand(B, P, 4, generator=g).pin_memory()
    A_p = (torch.rand(B, P, P, generator=g) * 0.5).pin_memory()
    coins = [(torch.rand(B, generator=g) >= 0.5).to(torch.uint8).pin_memory() for _ in range(agents)]
    for s in range(6):
        src = parents[s & 1]
        ref = [[_parent_forward(twins[k], env, src, x_p, A_p, lo, hi) for lo, hi in roll.ranges] for k in range(agents)]
        if agents == 1:
            dst = parents[1 - (s & 1)]
            roll.step(src, coins[0], x_p, A_p, dst)
            children = [dst]
        else:
            children = outs[s & 1]
            roll.step_agents(src, coins, x_p, A_p, children)
        for k in range(agents):
            p = params[k]
            for j, (lo, hi) in enumerate(roll.ranges):
                got = (children[k]["a_geo"][lo:hi].numpy(), children[k]["a_topo"][lo:hi].numpy())
                _assert_noise(got, ref[k][j], p["mu"], p["theta"], p["sigma"], p["seed"], 3 * s + j,
                              ("step", s + 1, "agent", k, "piece", j), clip=True)
        if agents > 1:
            nxt = parents[1 - (s & 1)]
            for name in nxt:
                nxt[name].copy_(children[s % agents][name])
    for p in pols:
        p.check()


# ================================================= production batches against float64 ==================================
def _closed_loop_states(family, B, seed):
    """reset + 3 closed-loop act / step of the trained agent 1: env-produced states of the production batch"""
    from mop_truss_marl_b200 import actor, batched_env
    env = batched_env.BatchedTrussEnv(family, B, device="cuda:0")
    env.reset()
    pol = actor.BatchedActor(trained_weights(1), env.N, B, seed=seed)
    x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50], device="cuda").repeat(B, 1, 1).contiguous()
    A_p = torch.ones(B, 1, 1, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(3):
        geo, topo = pol.act(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p)
        env.step(geo, topo, (torch.rand(B, device="cuda", generator=g) >= 0.5).to(torch.uint8))
    torch.cuda.synchronize()
    pol.check()
    assert int(env.status.abs().max()) == 0
    return env


def _pareto_inputs(B, seed, rows=50):
    """pareto.state_data of random fronts of 1..50 points (chain graphs, zero padding to 50 rows); a quarter of the
    environments get a dense A_p instead (the dense Pareto kernel behind the tridiagonal one)"""
    from mop_truss_marl_b200 import pareto
    g = torch.Generator(device="cuda").manual_seed(seed)
    pts = torch.rand(B, rows, 4, device="cuda", generator=g)
    pts[:, :, 0] = torch.sort(pts[:, :, 0], dim=1).values
    pts[:, :, 1] = torch.sort(pts[:, :, 1], dim=1, descending=True).values
    pts = pts.contiguous()
    front_len = torch.randint(1, rows + 1, (B,), device="cuda", generator=g, dtype=torch.int32)
    front_len[0] = rows
    index = (torch.rand(B, device="cuda", generator=g) * front_len.float()).to(torch.int32).clamp_max(front_len - 1)
    x_p, A_p = pareto.state_data(pts, front_len=front_len, index=index.contiguous(), rows=rows)
    dense = torch.rand(B, device="cuda", generator=g) < 0.25
    A_p[dense] = torch.rand(int(dense.sum()), rows, rows, device="cuda", generator=g) * 0.3
    n_pf = torch.randint(1, rows + 1, (B,), device="cuda", generator=g, dtype=torch.int32)
    return x_p.contiguous(), A_p.contiguous(), n_pf


PRODUCTION = [("small_bridge", 4096), ("large_bridge", 8192), ("large_roof", 4096), ("train2_roof", 4096)]


@pytest.mark.parametrize("family,B", PRODUCTION)
def test_production_batch_against_float64(family, B):
    """every environment of a production batch of env-produced states (fronts of up to 50 rows, chain and dense A_p in
    one batch, with and without n_pf) against the float64 oracle, 512 environments at a time: status 0, error <= 2e-5 and
    at most 8 times the float32 restatement's error on the same environments"""
    from mop_truss_marl_b200 import actor
    from oracle.actor_oracle import actor_forward
    env = _closed_loop_states(family, B, seed=B + len(family))
    x_p, A_p, n_pf = _pareto_inputs(B, seed=B)
    w = trained_weights(1)
    pol = actor.BatchedActor(w, env.N, B)
    state = (env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p)
    outs = {"all rows": [t.cpu().numpy() for t in pol.forward(*state)],
            "n_pf": [t.cpu().numpy() for t in pol.forward(*state, n_pf=n_pf)]}
    pol.check()
    host = [t.cpu().numpy() for t in state]
    npf_h = n_pf.cpu().numpy()
    summary = {}
    for name, (geo, topo) in outs.items():
        worst, worst_ratio, worst32 = 0.0, 0.0, 0.0
        for lo in range(0, B, 512):
            hi = min(B, lo + 512)
            args = [host[0][lo:hi], host[1]] + [h[lo:hi] for h in host[2:]]
            npf = npf_h[lo:hi] if name == "n_pf" else None
            g64, t64 = actor_forward(w, *args, n_pf=npf)
            g32, t32 = actor_forward(w, *args, n_pf=npf, dtype=np.float32)
            err = _err(geo[lo:hi], topo[lo:hi], g64, t64)
            err32 = _err(g32, t32, g64, t64)
            worst, worst32, worst_ratio = max(worst, err), max(worst32, err32), max(worst_ratio, err / err32)
            assert err <= ATOL and err <= 8 * err32, (name, lo, err, err32)
        summary[name] = {"max err": worst, "max err_f32": worst32, "max err/err_f32": worst_ratio}
    record("production_%s_%d" % (family, B), summary)


# ================================================= layout invariants (bit for bit) =====================================
def _random_state(B, N, P, seed, extra=0):
    """device inputs of B environments (+ extra rows of allocation behind them), activations O(1)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.rand(*s, device="cuda", generator=g)   # noqa: E731
    sc = 1.0 / N
    Bx = B + extra
    return [r(Bx, N, 13), r(N, N) * sc, r(Bx, N, N) * sc, r(Bx, N, N) * sc, r(Bx, N, N) * sc, r(Bx, P, 4), r(Bx, P, P) * 0.3]


@pytest.mark.parametrize("N,B", [(16, 4096), (32, 8192)])
def test_permutation_of_environments(N, B):
    """rows are independent: permuting the environments permutes the outputs, bit for bit (every environment lands in a
    different tile, row group, piece and CTA)"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    inp = _random_state(B, N, 3, seed=N)
    pol = actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=3), N, B)
    geo, topo = pol.forward(*inp)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(N)).cuda()
    pi = [t if t.dim() == 2 else t[perm].contiguous() for t in inp]
    geo_p, topo_p = pol.forward(*pi)
    torch.cuda.synchronize()
    pol.check()
    assert torch.equal(geo_p, geo[perm]) and torch.equal(topo_p, topo[perm])


@pytest.mark.parametrize("N,sizes", [(16, [1, 9, 109, 300, 1184, 1185, 1590, 4095, 4096]), (32, [1, 3, 592, 593, 1300, 8191, 8192])])
def test_prefixes_of_one_handle(N, sizes):
    """one handle created for the largest batch, called on the first B' environments: every call equals the first B' rows
    of the full call.  16 nodes: 4-way pieces (9, 109), half-live 2-way pieces (300, 1590), exactly one wave of 148 tiles
    (1184), one tile more (1185), persistence with split pieces (1590, 4095, 4096); 32 nodes likewise"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    Bmax = max(sizes)
    inp = _random_state(Bmax, N, 3, seed=7 + N)
    pol = actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=4), N, Bmax)
    geo, topo = [t.clone() for t in pol.forward(*inp)]
    for b in sizes:
        sub = [t if t.dim() == 2 else t[:b] for t in inp]
        g, t = pol.forward(*sub)
        torch.cuda.synchronize()
        assert torch.equal(g, geo[:b]) and torch.equal(t, topo[:b]), b
    pol.check()


@pytest.mark.parametrize("N,B", [(16, 4093), (32, 8190), (16, 1590)])
def test_nothing_read_or_written_past_the_batch(N, B):
    """the inputs are the first B environments of allocations of B + 8 whose tail is NaN (n_pf: a huge count), the outputs
    views of larger buffers filled with a sentinel: the result is that of clean inputs bit for bit, status 0, and the
    tail of every output buffer is untouched"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    P, extra = 3, 8
    clean = _random_state(B, N, P, seed=B)
    dirty = []
    for t in clean:
        if t.dim() == 2:
            dirty.append(t)
            continue
        d = torch.full((B + extra,) + tuple(t.shape[1:]), float("nan"), device="cuda")
        d[:B] = t
        dirty.append(d)
    n_pf_full = torch.full((B + extra,), 1 << 30, dtype=torch.int32, device="cuda")
    n_pf_full[:B] = torch.randint(1, P + 1, (B,), generator=torch.Generator().manual_seed(B), dtype=torch.int32).cuda()
    pol = actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=6), N, B)
    for npf in (None, n_pf_full):
        ref = [t.clone() for t in pol.forward(*clean, n_pf=None if npf is None else npf[:B].clone())]
        pol.check()
        sentinel = -7.25
        geo_buf = torch.full((B + extra, N, 2), sentinel, device="cuda")
        topo_buf = torch.full((B + extra, N, 3), sentinel, device="cuda")
        out = (geo_buf[:B], topo_buf[:B])
        pol.forward(*[t if t.dim() == 2 else t[:B] for t in dirty], n_pf=None if npf is None else npf[:B], out=out)
        torch.cuda.synchronize()
        pol.check()                                            # no NaN of the tails reached the kernel's operands
        assert torch.equal(out[0], ref[0]) and torch.equal(out[1], ref[1])
        assert bool((geo_buf[B:] == sentinel).all()) and bool((topo_buf[B:] == sentinel).all())
