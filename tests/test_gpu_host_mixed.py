"""GPU: MixedHostRollout / trollout_step_host_mixed / trollout_step_agents_host_mixed -- the host-resident rollout over a
mixed-family batch (batched_env.MixedTrussEnv).  Every environment of every child must be bit for bit what the resident
mixed path (MixedTrussEnv + BatchedActor) and what a single-family HostRollout of its own family compute, on the direct
path and on the replayed CUDA graph, and the graph must read the family ids when it is replayed."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SMALL, LARGE = ("small_bridge", "small_roof"), ("large_bridge", "large_roof")


def _train():
    from mop_truss_marl_b200.families import TRAIN_FAMILIES
    return TRAIN_FAMILIES


def _bits(t):
    return t.contiguous().view(torch.uint8)


def _assert_same(got: dict, want: dict, what):
    assert set(got) == set(want), what
    for k in want:
        assert torch.equal(_bits(got[k]), _bits(want[k])), (what, k)


def _random_ids(rng, F, B):
    ids = rng.randint(0, F, size=B).astype(np.uint8)
    ids[:F] = np.arange(F)                    # every family present
    rng.shuffle(ids)
    return ids


def _mixed_env(families, ids):
    from mop_truss_marl_b200 import batched_env
    env = batched_env.MixedTrussEnv(families, len(ids))
    env.reset(torch.from_numpy(np.asarray(ids, np.uint8)).to(env.device))
    return env


def _alloc(roll, kind):
    """kind: "compact" (raw tables + their live columns; the columns go up), "full" (raw tables only), "slim"
    (alloc_host(raw_tables=False): the columns only, both directions)"""
    return roll.alloc_host(compact=kind != "full", raw_tables=kind != "slim")


def _fill_parent(buf, env, rows=None):
    """the host state tuple of `env` (a MixedTrussEnv: with its family ids), or of its environments `rows`"""
    from mop_truss_marl_b200.host_pipeline import STATE_IN
    src = {k: getattr(env, k) for k in STATE_IN}
    src["node_y"], src["element_section"] = env.nN_x_n[:, :, 1], env.nN_x_e[:, :, 0]
    if hasattr(env, "family_ids"):
        src["family"] = env.family_ids
    for k in buf:
        if k in src:
            buf[k].copy_(src[k] if rows is None else src[k][rows])
    torch.cuda.synchronize()


def _actors(env, K, **kw):
    """K actors with different weights, seeds and noise parameters; the same call twice gives twins"""
    from mop_truss_marl_b200 import actor, tf_checkpoint
    return [actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=50 + k), env.N, env.B, device=env.device,
                               **dict(dict(seed=300 + k, theta=0.1 + 0.05 * k, sigma=0.1 + 0.05 * k), **kw))
            for k in range(K)]


def _pareto(B, P=2, n_pf=False):
    g = torch.Generator().manual_seed(7)
    x_p = torch.rand(B, P, 4, generator=g).pin_memory()
    A_p = torch.rand(B, P, P, generator=g).pin_memory()
    npf = torch.randint(1, P + 1, (B,), generator=g, dtype=torch.int32).pin_memory() if n_pf else None
    return x_p, A_p, npf


def _resident_child(par, kid, pol, coin, x_p, A_p, n_pf=None):
    """the resident mixed path: `pol` acts on the parent batch `par`, `kid` becomes its child (parent=)"""
    dev = par.device
    a_geo, a_topo = pol.act(par.x_n, par.A_n, par.A_s, par.A_n_ts, par.A_n_cs, x_p.to(dev), A_p.to(dev),
                            None if n_pf is None else n_pf.to(dev))
    kid.step(a_geo, a_topo, coin.to(dev), parent=par)
    torch.cuda.synchronize()
    return a_geo, a_topo


def _resident_outputs(kid, a_geo, a_topo, keys):
    src = {"a_geo": a_geo, "a_topo": a_topo, "family": kid.family_ids, "node_y": kid.nN_x_n[:, :, 1],
           "element_section": kid.nN_x_e[:, :, 0]}
    return {k: (src[k] if k in src else getattr(kid, k)).cpu() for k in keys}


@pytest.mark.parametrize("which,B,pieces,kind", [
    ("train", 300, [64, 236], "compact"),
    ("small", 77, 3, "full"),
    ("large", 70, 2, "compact"),
    ("train", 1500, "auto", "slim"),
])
def test_one_agent_equals_resident_mixed_path(which, B, pieces, kind):
    """noise off, six ping-pong steps between two buffer sets (two direct, two captured, two replayed): every output of
    the host rollout equals the resident MixedTrussEnv stepped by a twin actor, the family ids passed on included"""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import MixedHostRollout
    families = {"train": _train(), "small": SMALL, "large": LARGE}[which]
    ids = _random_ids(np.random.RandomState(B), len(families), B)
    env = _mixed_env(families, ids)
    res = _mixed_env(families, ids)
    kid = batched_env.MixedTrussEnv(families, B)
    pol, pol_r = _actors(env, 1, sigma=0.0, theta=0.0)[0], _actors(env, 1, sigma=0.0, theta=0.0)[0]
    roll = MixedHostRollout(env, pol, pieces=pieces)
    assert roll.ranges[-1][1] == B
    bufs = [_alloc(roll, kind), _alloc(roll, kind)]
    _fill_parent(bufs[0], env)
    x_p, A_p, n_pf = _pareto(B, n_pf=(kind == "full"))
    g = torch.Generator().manual_seed(5)
    for it in range(6):
        src, dst = bufs[it & 1], bufs[1 - (it & 1)]
        coin = (torch.rand(B, generator=g) >= 0.5).to(torch.uint8).pin_memory()
        roll.step(src, coin, x_p, A_p, dst, n_pf_host=n_pf)
        a_geo, a_topo = _resident_child(res, kid, pol_r, coin, x_p, A_p, n_pf)
        _assert_same(dst, _resident_outputs(kid, a_geo, a_topo, dst), it)
        for name in ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "move_range"):
            getattr(res, name).copy_(getattr(kid, name))
    assert int(kid.status.abs().max()) == 0 and pol.update_num == 6
    pol.check()


@pytest.mark.parametrize("env_var", [None, ("TROLLOUT_NO_GRAPH", "1"), ("TROLLOUT_ZEROCOPY", "0")])
def test_three_agents_equal_one_agent_rollouts(env_var, monkeypatch):
    """three agents over the ten train families, five fed-back steps with OU noise on (direct, captured, then
    replayed unless TROLLOUT_NO_GRAPH=1): every child equals the one-agent MixedHostRollout of its twin actor, and the
    launch counters and update_num of the two arms agree"""
    from mop_truss_marl_b200.host_pipeline import MixedHostRollout
    if env_var:
        monkeypatch.setenv(*env_var)
    K, B = 3, 230
    ids = _random_ids(np.random.RandomState(3), 10, B)
    env_m, env_s = _mixed_env(_train(), ids), _mixed_env(_train(), ids)
    pol_m, pol_s = _actors(env_m, K), _actors(env_s, K)
    multi = MixedHostRollout(env_m, pol_m, pieces=3)
    singles = [MixedHostRollout(env_s, pol_s[k], pieces=3) for k in range(K)]
    parent = multi.alloc_host()
    _fill_parent(parent, env_m)
    outs = multi.alloc_host_children()
    assert all("family" in o for o in outs)
    ref = [singles[k].alloc_host() for k in range(K)]
    x_p, A_p, _ = _pareto(B)
    rng = np.random.RandomState(4)
    coins = [torch.empty(B, dtype=torch.uint8).pin_memory() for _ in range(K)]
    for it in range(5):
        for c in coins:
            c.copy_(torch.from_numpy((rng.rand(B) >= 0.5).astype(np.uint8)))
        multi.step_agents(parent, coins, x_p, A_p, outs)
        for k in range(K):
            singles[k].step(parent, coins[k], x_p, A_p, ref[k])
            _assert_same(outs[k], ref[k], (it, k))
            assert torch.equal(outs[k]["family"], torch.from_numpy(ids))
        assert not torch.equal(outs[0]["a_geo"], outs[1]["a_geo"])       # the agents really differ
        for k in parent:
            parent[k].copy_(outs[it % K][k])
    for k in range(K):
        assert pol_m[k].launch_count() == pol_s[k].launch_count() and pol_m[k].update_num == pol_s[k].update_num == 5
        pol_m[k].check()
    assert env_m.launch_count() == env_s.launch_count()


def test_every_environment_equals_its_single_family_rollout():
    """noise off, three agents, two fed-back steps: environment b of every child of the mixed rollout equals what a
    single-family HostRollout of family ids[b] gives on the sub-batch of that family (in batch order)"""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import HostRollout, MixedHostRollout
    K, B = 3, 256
    ids = _random_ids(np.random.RandomState(8), 10, B)
    env = _mixed_env(_train(), ids)
    pol, pol_f = _actors(env, K, sigma=0.0, theta=0.0), _actors(env, K, sigma=0.0, theta=0.0)
    mix = MixedHostRollout(env, pol, pieces=2)
    parent, outs = mix.alloc_host(), mix.alloc_host_children()
    _fill_parent(parent, env)
    per = []
    for f, name in enumerate(_train()):
        rows = torch.from_numpy(np.nonzero(ids == f)[0])
        r = HostRollout(batched_env.BatchedTrussEnv(name, len(rows)), pol_f, pieces=1)
        p = r.alloc_host()
        _fill_parent(p, env, rows.to(env.device))
        per.append((rows, r, p, r.alloc_host_children()))
    x_p, A_p, _ = _pareto(B)
    g = torch.Generator().manual_seed(6)
    for it in range(2):
        coins = [(torch.rand(B, generator=g) >= 0.5).to(torch.uint8).pin_memory() for _ in range(K)]
        mix.step_agents(parent, coins, x_p, A_p, outs)
        for rows, r, p, o in per:
            r.step_agents(p, [c[rows].contiguous() for c in coins], x_p[rows].contiguous(), A_p[rows].contiguous(), o)
            for k in range(K):
                for name in o[k]:
                    assert torch.equal(_bits(outs[k][name][rows]), _bits(o[k][name])), (it, r.env.spec.name, k, name)
            for name in p:
                p[name].copy_(o[1][name])
        for name in parent:
            parent[name].copy_(outs[1][name])
    assert int(outs[0]["status"].abs().max()) == 0


@pytest.mark.parametrize("zerocopy", ["1", "0"])
def test_ids_are_read_at_every_replay(zerocopy, monkeypatch):
    """the same buffers every step: step 1 direct, step 2 captured, steps 3-4 replayed.  Before step 4 some ids are
    rewritten in the same pinned buffer; the replayed step follows them (the mapped-memory transfer kernel, or with
    TROLLOUT_ZEROCOPY=0 the captured memcpy node, reads them at replay), checked against the resident path"""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import MixedHostRollout
    monkeypatch.setenv("TROLLOUT_ZEROCOPY", zerocopy)
    B = 200
    rng = np.random.RandomState(12)
    ids = _random_ids(rng, 10, B)
    env = _mixed_env(_train(), ids)
    res = _mixed_env(_train(), ids)
    kid = batched_env.MixedTrussEnv(_train(), B)
    pol, pol_r = _actors(env, 1, sigma=0.0, theta=0.0)[0], _actors(env, 1, sigma=0.0, theta=0.0)[0]
    roll = MixedHostRollout(env, pol, pieces=[64, 136])
    parent, out = roll.alloc_host(), roll.alloc_host()
    _fill_parent(parent, env)
    x_p, A_p, _ = _pareto(B)
    coin = (torch.rand(B, generator=torch.Generator().manual_seed(1)) >= 0.5).to(torch.uint8).pin_memory()
    moved = torch.from_numpy(rng.choice(B, 40, replace=False))
    for it in range(4):
        if it == 3:
            before = out["point"].clone()
            new = (parent["family"][moved].long() + 1 + torch.from_numpy(rng.randint(0, 9, 40))) % 10
            parent["family"][moved] = new.to(torch.uint8)                 # in place: same buffer, same graph
            res.family_ids.copy_(parent["family"])
        roll.step(parent, coin, x_p, A_p, out)
        a_geo, a_topo = _resident_child(res, kid, pol_r, coin, x_p, A_p)
        _assert_same(out, _resident_outputs(kid, a_geo, a_topo, out), it)
    assert torch.equal(out["family"], parent["family"])
    assert not torch.equal(out["point"][moved], before[moved])             # the new families really changed the step


def test_bad_family_ids():
    """ids >= F set TFEM_STATUS_BAD_FAMILY in those environments' host status; every other environment is bit for
    bit the resident path with the same ids (direct, captured and replayed steps)"""
    from mop_truss_marl_b200 import batched_env, capi
    from mop_truss_marl_b200.host_pipeline import MixedHostRollout
    B = 160
    rng = np.random.RandomState(13)
    ids = _random_ids(rng, 10, B)
    env = _mixed_env(_train(), ids)
    res = _mixed_env(_train(), ids)
    kid = batched_env.MixedTrussEnv(_train(), B)
    pol, pol_r = _actors(env, 1, sigma=0.0, theta=0.0)[0], _actors(env, 1, sigma=0.0, theta=0.0)[0]
    roll = MixedHostRollout(env, pol, pieces=2)
    parent, out = roll.alloc_host(), roll.alloc_host()
    _fill_parent(parent, env)
    bad = torch.tensor([0, 31, 32, 100, 159])
    parent["family"][bad] = torch.tensor([10, 255, 16, 200, 11], dtype=torch.uint8)
    res.family_ids.copy_(parent["family"])
    good = torch.from_numpy(np.setdiff1d(np.arange(B), bad.numpy()))
    x_p, A_p, _ = _pareto(B)
    coin = (torch.rand(B, generator=torch.Generator().manual_seed(2)) >= 0.5).to(torch.uint8).pin_memory()
    for it in range(3):
        roll.step(parent, coin, x_p, A_p, out)
        a_geo, a_topo = _resident_child(res, kid, pol_r, coin, x_p, A_p)
        want = _resident_outputs(kid, a_geo, a_topo, out)
        assert (out["status"][bad] == capi.STATUS_BAD_FAMILY).all() and (out["status"][good] == 0).all(), it
        for k in out:
            assert torch.equal(_bits(out[k][good]), _bits(want[k][good])), (it, k)


def test_refusals():
    from mop_truss_marl_b200 import batched_env, capi
    from mop_truss_marl_b200.host_pipeline import HostRollout, MixedHostRollout, _AgentsIO, _IO, _lib
    B = 64
    ids = _random_ids(np.random.RandomState(1), 10, B)
    mix = _mixed_env(_train(), ids)
    pols = _actors(mix, 3)
    with pytest.raises(capi.TfemError, match="several families.*MixedHostRollout"):
        HostRollout(mix, pols[0])
    one, three = MixedHostRollout(mix, pols[0], pieces=2), MixedHostRollout(mix, pols, pieces=2)
    f3 = (C.c_float * 3)(0.1, 0.1, 0.1)
    s3 = (C.c_uint64 * 3)(1, 2, 3)
    # the plain calls on a rollout over ten families, refused before any buffer is read
    assert _lib.trollout_step_host(one._h, B, C.byref(_IO()), 0.1, 0.1, 0.1, 1) == -1
    assert b"trollout_step_host_mixed" in _lib.trollout_last_error()
    assert _lib.trollout_step_agents_host(three._h, B, C.byref(_AgentsIO()), f3, f3, f3, s3) == -1
    assert b"trollout_step_agents_host_mixed" in _lib.trollout_last_error()
    # NULL and misaligned ids
    fam = torch.zeros(B + 16, dtype=torch.uint8).pin_memory()
    assert _lib.trollout_step_host_mixed(one._h, B, None, C.byref(_IO()), 0.1, 0.1, 0.1, 1) == -1
    assert _lib.trollout_step_agents_host_mixed(three._h, B, None, C.byref(_AgentsIO()), f3, f3, f3, s3) == -1
    assert _lib.trollout_step_host_mixed(one._h, B, fam.data_ptr() + 1, C.byref(_IO()), 0.1, 0.1, 0.1, 1) == -4
    assert b"16-byte aligned" in _lib.trollout_last_error()
    # the _mixed calls on a rollout over a tfem_create handle
    env = batched_env.BatchedTrussEnv("train0_roof", B)
    env.reset()
    plain = HostRollout(env, _actors(env, 1)[0], pieces=2)
    assert _lib.trollout_step_host_mixed(plain._h, B, fam.data_ptr(), C.byref(_IO()), 0.1, 0.1, 0.1, 1) == -1
    assert b"tfem_create_mixed" in _lib.trollout_last_error()
    with pytest.raises(ValueError, match="MixedTrussEnv"):
        MixedHostRollout(env, _actors(env, 1)[0])
    # a state tuple without the ids
    parent, out = one.alloc_host(), one.alloc_host()
    _fill_parent(parent, mix)
    x_p, A_p, _ = _pareto(B)
    no_ids = {k: v for k, v in parent.items() if k != "family"}
    with pytest.raises(ValueError, match="lacks 'family'"):
        one.step(no_ids, None, x_p, A_p, out)
    with pytest.raises(ValueError, match="lacks 'family'"):
        three.step_agents(no_ids, [None] * 3, x_p, A_p, three.alloc_host_children())
    assert pols[0].update_num == 0
    one.step(parent, None, x_p, A_p, out)                                      # usable after the refusals
    assert pols[0].update_num == 1 and int(out["status"].abs().max()) == 0


def test_one_family_mixed_env_through_both_kinds_of_step():
    """a one-family MixedTrussEnv steps through the plain HostRollout bit for bit as a BatchedTrussEnv of that family;
    the plain and the _mixed call on one rollout over it, with the same buffers, give the same bits (each kind of step
    is captured and replayed as its own graph)"""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import HostRollout, MixedHostRollout, _IO, _check, _lib
    B = 96
    single = batched_env.BatchedTrussEnv("train2_bridge", B)
    single.reset()
    mix1 = _mixed_env(("train2_bridge",), np.zeros(B, np.uint8))
    r_single = HostRollout(single, _actors(single, 1)[0], pieces=2)
    r_plain = HostRollout(mix1, _actors(mix1, 1)[0], pieces=2)
    pol = _actors(mix1, 1, sigma=0.0, theta=0.0)[0]
    r_both = MixedHostRollout(mix1, pol, pieces=2)
    bufs = {r: [r.alloc_host(), r.alloc_host()] for r in (r_single, r_plain)}
    for r, env in ((r_single, single), (r_plain, mix1)):
        _fill_parent(bufs[r][0], env)
    parent, out = r_both.alloc_host(), r_both.alloc_host()
    _fill_parent(parent, mix1)
    x_p, A_p, _ = _pareto(B)
    coin = (torch.rand(B, generator=torch.Generator().manual_seed(4)) >= 0.5).to(torch.uint8).pin_memory()
    for it in range(4):
        src, dst = it & 1, 1 - (it & 1)
        for r in (r_single, r_plain):
            r.step(bufs[r][src], coin, x_p, A_p, bufs[r][dst])
        _assert_same(bufs[r_plain][dst], bufs[r_single][dst], it)
        io = _IO()
        r_both._parent(io, parent, x_p, A_p, None)
        r_both._child(io, out, coin)
        _check(_lib.trollout_step_host(r_both._h, B, C.byref(io), pol.mu, pol.theta, pol.sigma, pol.seed))
        plain = {k: v.clone() for k, v in out.items() if k != "family"}
        r_both.step(parent, coin, x_p, A_p, out)
        _assert_same({k: v for k, v in out.items() if k != "family"}, plain, ("mixed vs plain", it))


@pytest.mark.parametrize("agents", [1, 3])
def test_bytes_per_step(agents):
    """a ten-family rollout uploads the family id on top of what a one-family rollout of the same dimensions moves"""
    from mop_truss_marl_b200.host_pipeline import MixedHostRollout
    B = 128
    ten = _mixed_env(_train(), _random_ids(np.random.RandomState(2), 10, B))
    one = _mixed_env(_train()[:1], np.zeros(B, np.uint8))
    r10 = MixedHostRollout(ten, _actors(ten, agents), pieces=2)
    r1 = MixedHostRollout(one, _actors(one, agents), pieces=2)
    for compact in (True, False):
        up10, down10 = r10.bytes_per_step(compact=compact)
        up1, down1 = r1.bytes_per_step(compact=compact)
        assert up10 == up1 + B and down10 == down1
