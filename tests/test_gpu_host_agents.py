"""GPU: HostRollout over a list of actors / trollout_step_agents_host -- the driver's inner step (every agent acts on the
same parent and steps its own child) in one call, the parent uploaded once.  Child k must be bit for bit what a
one-agent HostRollout of actor k gives on the same parent with coin k, OU noise included, on the direct path and on
the replayed CUDA graph."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _bits(t):
    return t.contiguous().view(torch.uint8)


def _assert_same(got: dict, want: dict, what):
    assert set(got) == set(want), what
    for k in want:
        assert torch.equal(_bits(got[k]), _bits(want[k])), (what, k)


def _alloc(roll, kind):
    """kind: "compact" (raw tables + their live columns; the columns go up), "full" (raw tables only), "slim"
    (alloc_host(raw_tables=False): the columns only, both directions)"""
    return roll.alloc_host(compact=kind != "full", raw_tables=kind != "slim")


def _fill_parent(buf, env):
    from mop_truss_marl_b200.host_pipeline import STATE_IN
    for k in STATE_IN:
        if k in buf:
            buf[k].copy_(getattr(env, k))
    if "node_y" in buf:
        buf["node_y"].copy_(env.nN_x_n[:, :, 1])
        buf["element_section"].copy_(env.nN_x_e[:, :, 0])
    torch.cuda.synchronize()


def _agents(env, K, **kw):
    """K actors with different weights, seeds and noise parameters; the same call twice gives twins"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    return [actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=30 + k), env.N, env.B, device=env.device,
                               **dict(dict(seed=100 + k, theta=0.1 + 0.05 * k, sigma=0.1 + 0.05 * k), **kw))
            for k in range(K)]


def _pareto(B, P=2, n_pf=False):
    g = torch.Generator().manual_seed(7)
    x_p = torch.rand(B, P, 4, generator=g).pin_memory()
    A_p = torch.rand(B, P, P, generator=g).pin_memory()
    npf = torch.randint(1, P + 1, (B,), generator=g, dtype=torch.int32).pin_memory() if n_pf else None
    return x_p, A_p, npf


@pytest.mark.parametrize("family,B,pieces,kind,env_var", [
    ("small_bridge", 77, [32, 45], "compact", None),
    ("large_roof", 70, 2, "full", None),
    ("train0_roof", 100, [64, 36], "slim", None),                 # the 12-node actor (padded to 16 nodes inside)
    ("small_bridge", 150, 3, "compact", ("TROLLOUT_NO_GRAPH", "1")),
    ("train0_roof", 90, 2, "compact", ("TROLLOUT_ZEROCOPY", "0")),
    ("large_bridge", 130, "auto", "slim", None),
])
def test_children_equal_single_agent_rollouts(family, B, pieces, kind, env_var, monkeypatch):
    """three agents, five consecutive steps with OU noise on: step 1 is enqueued directly, step 2 captured, steps 3-5
    replayed (unless TROLLOUT_NO_GRAPH=1).  The coins and the next parent (one of the children) are copied into the
    same host buffers every step, so that the buffer set repeats.  Every output of every child equals the one-agent
    rollout of its twin actor, and the launch counters of the two arms agree."""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import HostRollout
    if env_var:
        monkeypatch.setenv(*env_var)
    K = 3
    env_m, env_s = batched_env.BatchedTrussEnv(family, B), batched_env.BatchedTrussEnv(family, B)
    env_m.reset(); env_s.reset()
    pol_m, pol_s = _agents(env_m, K), _agents(env_s, K)
    multi = HostRollout(env_m, pol_m, pieces=pieces)
    singles = [HostRollout(env_s, pol_s[k], pieces=pieces) for k in range(K)]
    assert multi.ranges == singles[0].ranges and multi.ranges[-1][1] == B
    parent = _alloc(multi, kind)
    _fill_parent(parent, env_m)
    outs = multi.alloc_host_children(compact=kind != "full", raw_tables=kind != "slim")
    assert len(outs) == K
    ref = [_alloc(singles[k], kind) for k in range(K)]
    x_p, A_p, n_pf = _pareto(B, n_pf=(kind == "full"))
    rng = np.random.RandomState(4)
    coins = [torch.empty(B, dtype=torch.uint8).pin_memory() for _ in range(K)]
    for it in range(5):
        for c in coins:
            c.copy_(torch.from_numpy((rng.rand(B) >= 0.5).astype(np.uint8)))
        multi.step_agents(parent, coins, x_p, A_p, outs, n_pf_host=n_pf)
        for k in range(K):
            singles[k].step(parent, coins[k], x_p, A_p, ref[k], n_pf_host=n_pf)
            _assert_same(outs[k], ref[k], (it, k))
        assert not torch.equal(outs[0]["a_geo"], outs[1]["a_geo"])       # the agents really differ
        for k in parent:
            parent[k].copy_(outs[it % K][k])
    for k in range(K):
        assert pol_m[k].launch_count() == pol_s[k].launch_count() and pol_m[k].update_num == pol_s[k].update_num == 5
        pol_m[k].check()
    assert env_m.launch_count() == env_s.launch_count()
    up_m, down_m = multi.bytes_per_step(compact=kind != "full", raw_tables=kind != "slim")
    up_s, down_s = singles[0].bytes_per_step(compact=kind != "full", raw_tables=kind != "slim")
    assert up_m == up_s + (K - 1) * B and down_m == K * down_s               # parent up once, every child down


def test_children_equal_resident_parent_path():
    """the resident path's "three agents act on the same parent" (BatchedTrussEnv.step(parent=...), bench.py --train)
    gives the same children, over several fed-back steps (noise off: the resident act draws one call per step, the
    rollout one per piece)"""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import HostRollout, STATE_IN, STATE_OUT
    family, B, K = "small_bridge", 96, 3
    par = batched_env.BatchedTrussEnv(family, B)
    par.reset()
    kids = [batched_env.BatchedTrussEnv(family, B) for _ in range(K)]
    pol = _agents(par, K, sigma=0.0, theta=0.0)
    roll = HostRollout(par, pol, pieces=2)
    parent = roll.alloc_host()
    _fill_parent(parent, par)
    outs = roll.alloc_host_children()
    x_p, A_p, _ = _pareto(B)
    x_p_d, A_p_d = x_p.to(par.device), A_p.to(par.device)
    g = torch.Generator().manual_seed(2)
    for it in range(4):
        coins = [(torch.rand(B, generator=g) >= 0.5).to(torch.uint8).pin_memory() for _ in range(K)]
        roll.step_agents(parent, coins, x_p, A_p, outs)
        for k in range(K):
            a_geo, a_topo = pol[k].act(par.x_n, par.A_n, par.A_s, par.A_n_ts, par.A_n_cs, x_p_d, A_p_d)
            kids[k].step(a_geo, a_topo, coins[k].to(par.device), parent=par)
            torch.cuda.synchronize()
            for name in STATE_OUT:
                assert torch.equal(outs[k][name], getattr(kids[k], name).cpu()), (it, k, name)
            assert torch.equal(outs[k]["a_geo"], a_geo.cpu()) and torch.equal(outs[k]["a_topo"], a_topo.cpu())
        nxt = it % K
        for name in STATE_IN:
            getattr(par, name).copy_(getattr(kids[nxt], name))
        for name in parent:
            parent[name].copy_(outs[nxt][name])
        torch.cuda.synchronize()


def test_one_agent_list_equals_trollout_create(monkeypatch):
    """trollout_create_agents with one actor is trollout_create: the same bits over direct and replayed steps"""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import HostRollout
    B = 200
    env = batched_env.BatchedTrussEnv("small_bridge", B)
    env.reset()
    a, b = _agents(env, 1), _agents(env, 1)
    r_one, r_list = HostRollout(env, a[0], pieces=3), HostRollout(env, b, pieces=3)
    bufs = [[r.alloc_host(), r.alloc_host()] for r in (r_one, r_list)]
    for bb in bufs:
        _fill_parent(bb[0], env)
    x_p, A_p, _ = _pareto(B)
    coin = (torch.rand(B, generator=torch.Generator().manual_seed(3)) >= 0.5).to(torch.uint8).pin_memory()
    for it in range(5):
        src, dst = it & 1, 1 - (it & 1)
        r_one.step(bufs[0][src], coin, x_p, A_p, bufs[0][dst])
        r_list.step_agents(bufs[1][src], [coin], x_p, A_p, [bufs[1][dst]])
        _assert_same(bufs[1][dst], bufs[0][dst], it)
    assert a[0].launch_count() == b[0].launch_count()
    assert r_one.bytes_per_step() == r_list.bytes_per_step()
    r_one.step(bufs[0][1], coin, x_p, A_p, bufs[0][0])              # a one-actor list also takes step()
    r_list.step(bufs[1][1], coin, x_p, A_p, bufs[1][0])
    _assert_same(bufs[1][0], bufs[0][0], "step")


def test_refusals():
    from mop_truss_marl_b200 import actor, batched_env, capi, tf_checkpoint
    from mop_truss_marl_b200.host_pipeline import HostRollout, _IO, _lib
    B = 64
    env = batched_env.BatchedTrussEnv("small_bridge", B)
    env.reset()
    pols = _agents(env, 4)
    with pytest.raises(capi.TfemError, match="n_agents must be in 1..3, got 0"):
        HostRollout(env, [])
    with pytest.raises(capi.TfemError, match="n_agents must be in 1..3, got 4"):
        HostRollout(env, pols)
    with pytest.raises(capi.TfemError, match="distinct actor handles"):
        HostRollout(env, [pols[0], pols[1], pols[0]])
    other = actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=1), 32, B)        # a large-mesh actor
    with pytest.raises(ValueError, match="16 nodes"):
        HostRollout(env, [pols[0], other])
    roll = HostRollout(env, pols[:3], pieces=2)
    parent = roll.alloc_host()
    _fill_parent(parent, env)
    outs = roll.alloc_host_children()
    x_p, A_p, _ = _pareto(B)
    coins = [None] * 3
    with pytest.raises(ValueError, match="runs 3 actors: step it with step_agents"):
        roll.step(parent, None, x_p, A_p, outs[0])
    rc = _lib.trollout_step_host(roll._h, B, C.byref(_IO()), 0.1, 0.1, 0.1, 1)     # refused before any buffer is read
    assert rc == -1 and b"trollout_step_agents_host" in _lib.trollout_last_error()
    with pytest.raises(ValueError, match="one coin"):
        roll.step_agents(parent, coins, x_p, A_p, outs[:2])
    del outs[2]["point"]
    with pytest.raises(ValueError, match="lacks 'point'"):
        roll.step_agents(parent, coins, x_p, A_p, outs)
    outs[2] = roll.alloc_host()
    roll.step_agents(parent, coins, x_p, A_p, outs)                                   # usable after the refusals
    assert [p.update_num for p in pols[:3]] == [1, 1, 1]
