"""GPU: families of the chord lengths num_x = 3..16 beyond the reference's 6, 8 and 16, with train/code's ENV (no symmetry
step), and the actor on their 2 num_x node graphs (padded to the 16- or 32-node build).  The families are built here
(test_chord_lengths_cpu.spec_pair) and registered under their own names for the duration of a test only, so that the
helpers of test_gpu_parity.py, test_gpu_train_families.py, test_gpu_mixed.py and the actor tests run on them unchanged.

* every new num_x, bridge and roof: reset, random walks (uniform, small, saturated) against the Python and C oracles
  with the bars of DESIGN.md section 4, adversarial transitions, solve_only and read_genes;
* whole 4096-environment batches of an odd and an even num_x against the C oracle; the dense DMMA solve of an odd num_x;
* mixed batches of num_x 10 and 15 bit for bit against single-family batches, bad ids included, and the family limit;
* the actor on every newly accepted node count with the trained 2000pickle_base agents, its OU noise and its last-wave
  split; the host-resident three-agent step on an odd num_x; the drop-in modules on a 10 x 2 truss."""
import numpy as np
import pytest

from test_chord_lengths_cpu import spec_pair

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NEW_CHORDS = (3, 4, 5, 7, 9, 10, 11, 12, 13, 14, 15)
NEW_NODES = tuple(2 * n for n in NEW_CHORDS)          # every newly accepted actor node count: 6, 8, 10, 14, 18, 20, ..., 30
TYPES = ("bridge", "roof")
WALKS = ("uniform", "small_actions", "saturated")


@pytest.fixture
def register(monkeypatch):
    """register(num_x, truss_type, **spec_args) -> the name under which the library and the oracle know the family"""
    import oracle.truss_oracle as orc_mod
    from mop_truss_marl_b200 import families

    def reg(num_x, truss_type, **kw):
        lib, orc = spec_pair(num_x, truss_type, **kw)
        monkeypatch.setitem(families.FAMILIES, lib.name, lib)
        monkeypatch.setitem(orc_mod.FAMILIES, orc.name, orc)
        return lib.name
    return reg


@pytest.fixture(scope="module")
def envmod():
    from mop_truss_marl_b200 import batched_env
    return batched_env


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ================================================= env-step against the oracles =========================================
@pytest.mark.parametrize("truss_type", TYPES)
@pytest.mark.parametrize("num_x", NEW_CHORDS)
def test_constants_and_reset_vs_oracle(envmod, register, num_x, truss_type):
    from test_gpu_parity import cpu
    from test_gpu_train_families import oracle, reset_checks
    name = register(num_x, truss_type)
    o = oracle(name)
    env = envmod.BatchedTrussEnv(name, 3)
    assert np.array_equal(cpu(env.A_n), o.A_n) and np.array_equal(cpu(env.mask), o.mask)
    assert np.array_equal(cpu(env.nC_e), o.nC_e)
    assert np.array_equal(env.int_obj, np.array([o.int_obj1, o.int_obj2], dtype=np.float32))
    env.reset()
    torch.cuda.synchronize()
    for i in range(3):
        reset_checks(env, i, name)


@pytest.mark.parametrize("walk", WALKS)
@pytest.mark.parametrize("truss_type", TYPES)
@pytest.mark.parametrize("num_x", NEW_CHORDS)
def test_walk_vs_oracles(envmod, register, num_x, truss_type, walk):
    """three steps of one walk, every environment against the C oracle and (inside the flat 1e-9) the Python oracle
    (test_gpu_train_families.step_and_check): transition and move range bit-exact, FP64 fields within the flat 1e-9 --
    for the saturated walk, whose heights reach d_min, within 20 eps cond(K) of the extended-precision solve and no
    further from it than the oracle --, float32 tensors and point within 2 ulp, flags exact"""
    from test_gpu_train_families import population_rule, report, step_and_check
    name = register(num_x, truss_type)
    B, N = 32, 2 * num_x
    rng = np.random.RandomState(num_x * 10 + WALKS.index(walk) + 3 * TYPES.index(truss_type))
    env = envmod.BatchedTrussEnv(name, B)
    env.reset()
    ids = np.zeros(B, np.uint8)
    up = rng.rand(B, N) < 0.5
    stats, failed, r_errs = {}, [], []
    for s in range(3):
        if walk == "uniform":
            geo, topo = rng.rand(B, N, 2), rng.rand(B, N, 3)
        elif walk == "small_actions":
            geo, topo = 0.1 * rng.rand(B, N, 2), 0.1 * rng.rand(B, N, 3)
        else:                                        # every node held at its saturated direction, sections at random
            geo = np.where(up[..., None], np.float32([1, 0]), np.float32([0, 1]))
            topo = (rng.rand(B, N, 3) < 0.5)
        coin = (rng.rand(B) >= 0.5).astype(np.uint8)
        failed += step_and_check(env, [name], ids, dev(geo.astype(np.float32)), dev(topo.astype(np.float32)), dev(coin),
                                 "%s %s step %d" % (name, walk, s), stats, None if walk == "saturated" else 0, r_errs)
    report(walk, stats)
    if walk == "saturated":
        failed += population_rule(r_errs)
    assert not failed, "; ".join(failed)


@pytest.mark.parametrize("truss_type", TYPES)
@pytest.mark.parametrize("num_x", NEW_CHORDS)
def test_adversarial_transition_vs_oracle(envmod, register, num_x, truss_type):
    import test_gpu_parity
    test_gpu_parity.test_adversarial_transition_vs_oracle(envmod, register(num_x, truss_type))


@pytest.mark.parametrize("truss_type", TYPES)
@pytest.mark.parametrize("num_x", NEW_CHORDS)
def test_solve_only_vs_oracle(envmod, register, num_x, truss_type):
    import test_gpu_parity
    test_gpu_parity.test_solve_only_vs_oracle(envmod, register(num_x, truss_type))


@pytest.mark.parametrize("truss_type", TYPES)
@pytest.mark.parametrize("num_x", NEW_CHORDS)
def test_read_genes_vs_oracle(num_x, truss_type):
    """GeneEvaluator of a spec (max_height = span_y, the generator's y_max) against oracle/genes_oracle.py"""
    from mop_truss_marl_b200.genes import GeneEvaluator
    from oracle import genes_oracle
    from oracle.truss_oracle import TrussOracle
    from test_gpu_genes import ALL, fp64_tol
    from util import assert_f32_close, nrm
    lib, orc = spec_pair(num_x, truss_type)
    o = TrussOracle(orc)
    rng = np.random.RandomState(num_x)
    B = 48
    genes = rng.rand(B, o.mesh.N + o.mesh.E)
    genes[::3, :o.mesh.N] *= 0.05
    genes[1::4, o.mesh.N:] = np.round(genes[1::4, o.mesh.N:] * 8) / 8
    ev = GeneEvaluator(lib)
    assert ev.max_height == lib.span_y[0]
    ev.read_genes(genes, fields=ALL)
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in ev.out.items()}
    assert int(np.abs(out["status"]).max()) == 0
    for b in range(B):
        want = genes_oracle.read_genes(o, genes[b], max_height=ev.max_height)
        assert np.array_equal(out["y"][b], want["y"]) and np.array_equal(out["section"][b], want["section"]), b
        tol = fp64_tol(o, want["y"], want["section"])
        for k in ("d", "axial", "ratio"):
            assert nrm(out[k][b], want[k]) <= tol, (b, k, tol)
        assert abs(out["U"][b] - want["U"]) <= tol * abs(want["U"])
        assert_f32_close("point", out["point"][b], want["point"])
        assert nrm(out["point64"][b], want["point64"]) <= tol


@pytest.mark.parametrize("num_x,truss_type", [(11, "bridge"), (12, "roof")])
def test_full_batch_against_c_oracle(envmod, register, num_x, truss_type):
    import test_gpu_parity
    test_gpu_parity.test_full_batch_against_c_oracle(envmod, register(num_x, truss_type), 4096)


def test_dense_dmma_solve_vs_oracle_and_banded(envmod, register):
    import test_gpu_parity
    test_gpu_parity.test_dense_dmma_solve_vs_oracle_and_banded(envmod, register(13, "bridge"))


# ================================================= mixed batches =========================================================
def mixed_specs(num_x):
    """three families of one num_x: a bridge, a roof with other spans and targets, a bridge of another height"""
    import dataclasses
    bridge, _ = spec_pair(num_x, "bridge")
    roof, _ = spec_pair(num_x, "roof", span_y=4.0)
    roof = dataclasses.replace(roof, span_x=tuple(5.0 for _ in roof.span_x), tar_y=tuple(2.0 for _ in roof.tar_y))
    tall, _ = spec_pair(num_x, "bridge", span_y=6.0, loady=-75000.0)
    tall = dataclasses.replace(tall, name=tall.name + "_tall")
    return [bridge, roof, tall]


@pytest.mark.parametrize("num_x", [10, 15])
def test_mixed_batch_bit_identical(num_x):
    from mop_truss_marl_b200 import capi
    from test_gpu_mixed import Twin, walk
    rng = np.random.RandomState(num_x)
    B = 160
    ids = rng.randint(0, 3, size=B).astype(np.uint8)
    ids[:3] = np.arange(3)
    bad = rng.rand(B) < 0.05
    bad[5] = True
    ids[bad] = rng.choice(np.array([3, 17, 255], np.uint8), size=int(bad.sum()))
    tw = Twin(mixed_specs(num_x), ids)
    tw.reset()
    tw.compare("reset")
    walk(tw, rng)
    st = tw.mix.status.cpu().numpy()
    assert (st[~bad] == 0).all() and (st[bad] == capi.STATUS_BAD_FAMILY).all()


@pytest.mark.parametrize("num_x", [10, 15])
def test_mixed_family_limit_reported(num_x):
    """16 families do not fit the shared memory of one CTA at two CTAs per SM: refused with the limit in the text; the
    limit itself is accepted and one more is refused"""
    import dataclasses
    import re
    from mop_truss_marl_b200 import batched_env, capi
    base = mixed_specs(num_x)[0]
    variants = [dataclasses.replace(base, name="%s_v%d" % (base.name, k), loady=base.loady * (1 + 0.1 * k)) for k in range(16)]
    with pytest.raises(capi.TfemError, match=r"at most \d+ families") as e:
        batched_env.MixedTrussEnv(variants, 8)
    k = int(re.search(r"at most (\d+) families", str(e.value)).group(1))
    print("num_x = %d: at most %d families" % (num_x, k))
    assert 1 <= k < 16
    batched_env.MixedTrussEnv(variants[:k], 8)
    with pytest.raises(capi.TfemError, match="at most %d families" % k):
        batched_env.MixedTrussEnv(variants[:k + 1], 8)


# ================================================= actor =================================================================
ATOL = 2e-5


def env_states(num_x, truss_type, B):
    """reset plus two random steps of a family of num_x: the graph tensors the actor reads in play"""
    from mop_truss_marl_b200 import batched_env
    lib, _ = spec_pair(num_x, truss_type)
    env = batched_env.BatchedTrussEnv(lib, B)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(num_x)
    keys = ("x_n", "A_s", "A_n_ts", "A_n_cs")
    states = [[getattr(env, k).cpu().numpy().copy() for k in keys]]
    for s in range(2):
        env.step(torch.rand(B, env.N, 2, device="cuda", generator=g) * (0.5 + 0.5 * s),
                 torch.rand(B, env.N, 3, device="cuda", generator=g),
                 (torch.rand(B, device="cuda", generator=g) >= 0.5).to(torch.uint8))
        torch.cuda.synchronize()
        assert int(env.status.abs().max()) == 0
        states.append([getattr(env, k).cpu().numpy().copy() for k in keys])
    cat = [np.concatenate([st[i] for st in states]).astype(np.float32) for i in range(len(keys))]
    return cat[0], env.A_n.cpu().numpy().astype(np.float32), cat[1], cat[2], cat[3]


@pytest.mark.parametrize("agent", [1, 2, 3])
@pytest.mark.parametrize("nodes", NEW_NODES)
def test_trained_agents_on_random_graphs(nodes, agent):
    from mop_truss_marl_b200 import actor
    from oracle.actor_oracle import actor_forward
    from test_gpu_actor import trained_weights
    rng = np.random.RandomState(100 * agent + nodes)
    B, P = 40, (1, 17, 50)[agent - 1]
    r = lambda *s: rng.rand(*s).astype(np.float32)          # noqa: E731
    sc = np.float32(1.0 / nodes)                             # dense adjacency scaled by 1 / N: activations O(1)
    inp = [r(B, nodes, 13), r(nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc, r(B, nodes, nodes) * sc,
           r(B, P, 4), r(B, P, P) * np.float32(0.3)]
    n_pf = rng.randint(1, P + 1, size=B).astype(np.int32)
    a = actor.BatchedActor(trained_weights(agent), nodes, max_batch=B)
    geo, topo = a.forward(*[dev(t) for t in inp], n_pf=dev(n_pf))
    a.check()
    g64, t64 = actor_forward(trained_weights(agent), *inp, n_pf=n_pf)
    assert geo.shape == (B, nodes, 2) and topo.shape == (B, nodes, 3)
    assert np.abs(geo.cpu().numpy() - g64).max() <= ATOL and np.abs(topo.cpu().numpy() - t64).max() <= ATOL


@pytest.mark.parametrize("agent", [1, 2, 3])
@pytest.mark.parametrize("nodes", NEW_NODES)
def test_trained_agents_on_env_states(nodes, agent):
    """states the env-step produced for a family of nodes / 2 columns, with Pareto graphs of 1 to 50 rows zero-padded to
    P = 50 (test_gpu_actor.padded_pareto_graph)"""
    from mop_truss_marl_b200 import actor
    from oracle.actor_oracle import actor_forward
    from test_gpu_actor import padded_pareto_graph, trained_weights
    rng = np.random.RandomState(7 * agent + nodes)
    x_n, A_n, A_s, A_ts, A_cs = env_states(nodes // 2, TYPES[agent % 2], 8)
    B, P = x_n.shape[0], 50
    sizes = rng.randint(1, P + 1, size=B)
    sizes[0], sizes[1] = P, 1
    x_p, A_p = padded_pareto_graph(rng, B, P, sizes)
    w = trained_weights(agent)
    a = actor.BatchedActor(w, nodes, max_batch=B)
    geo, topo = a.forward(*[dev(t) for t in (x_n, A_n, A_s, A_ts, A_cs, x_p, A_p)])
    a.check()
    g64, t64 = actor_forward(w, x_n, A_n, A_s, A_ts, A_cs, x_p, A_p)
    assert np.abs(geo.cpu().numpy() - g64).max() <= ATOL and np.abs(topo.cpu().numpy() - t64).max() <= ATOL


@pytest.mark.parametrize("N,B", [(10, 1500), (24, 1200)])
def test_act_noise_element_by_element(N, B):
    """one count padded to the 16-node build, one to the 32-node build: the noise of output element i is drawn for i of
    the unpadded [B, N, 2] / [B, N, 3] tensors"""
    import test_gpu_actor_contract
    test_gpu_actor_contract.test_act_noise_element_by_element(N, B)


@pytest.mark.parametrize("nodes,B", [(14, 300), (14, 1600), (30, 150), (30, 1300)])
def test_last_wave_split_is_bit_identical(nodes, B, monkeypatch):
    import test_gpu_actor
    test_gpu_actor.test_last_wave_split_is_bit_identical(nodes, B, monkeypatch)


# ================================================= host-resident rollout =================================================
def test_rollout_agents_equal_resident_path():
    """HostRollout(env, [pol0, pol1, pol2]).step_agents on a 7 x 2 bridge against the resident path (the three agents act
    on the same parent, BatchedTrussEnv.step(parent=...)): step 1 direct, step 2 captured, steps 3-4 replayed"""
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.host_pipeline import HostRollout, STATE_IN, STATE_OUT
    from test_gpu_host_agents import _agents, _fill_parent, _pareto
    lib, _ = spec_pair(7, "bridge")
    B, K = 96, 3
    par = batched_env.BatchedTrussEnv(lib, B)
    par.reset()
    kids = [batched_env.BatchedTrussEnv(lib, B) for _ in range(K)]
    pol = _agents(par, K, sigma=0.0, theta=0.0)
    roll = HostRollout(par, pol, pieces=2)
    parent = roll.alloc_host()
    _fill_parent(parent, par)
    outs = roll.alloc_host_children()
    x_p, A_p, _ = _pareto(B)
    x_p_d, A_p_d = x_p.to(par.device), A_p.to(par.device)
    g = torch.Generator().manual_seed(3)
    for it in range(4):
        coins = [(torch.rand(B, generator=g) >= 0.5).to(torch.uint8).pin_memory() for _ in range(K)]
        roll.step_agents(parent, coins, x_p, A_p, outs)
        for k in range(K):
            a_geo, a_topo = pol[k].act(par.x_n, par.A_n, par.A_s, par.A_n_ts, par.A_n_cs, x_p_d, A_p_d)
            kids[k].step(a_geo, a_topo, coins[k].to(par.device), parent=par)
            torch.cuda.synchronize()
            assert int(kids[k].status.abs().max()) == 0
            for name in STATE_OUT:
                assert torch.equal(outs[k][name], getattr(kids[k], name).cpu()), (it, k, name)
            assert torch.equal(outs[k]["a_geo"], a_geo.cpu()) and torch.equal(outs[k]["a_topo"], a_topo.cpu())
        nxt = it % K
        for name in STATE_IN:
            getattr(par, name).copy_(getattr(kids[nxt], name))
        for name in parent:
            parent[name].copy_(outs[nxt][name])
        torch.cuda.synchronize()
    for p in pol:
        p.check()


# ================================================= drop-in modules =======================================================
def test_dropin_ten_column_truss():
    """gen_model(10, 2, ...) + Game_research04 + MADDPG.agents[k].act, as the reference driver calls them with a 10 x 2
    truss (train/code's ENV: no symmetry step): the reset state and four steps against the oracle"""
    import random
    from mop_truss_marl_b200 import compat
    from oracle.truss_oracle import TrussOracle
    from test_gpu_compat import quiet
    from util import assert_f32_close
    compat.install()
    import truss2D_ENV as ENV
    import truss2D_GEN as GEN
    import truss2D_RL as RL
    lib, orc = spec_pair(10, "bridge")
    o = TrussOracle(orc)
    gm = quiet(GEN.gen_model, 10, 2, list(lib.span_x), list(lib.span_y), list(lib.tar_y), lib.dmin, 0, lib.loady, "bridge", 1, None)
    game = quiet(ENV.Game_research04, 500, gm, 3)
    st = game._game_get_1_state()
    want = o.reset()
    for k, idx in (("x_n", 0), ("A_s", 2), ("A_n_ts", 3), ("A_n_cs", 4), ("nN_x_n", 8), ("nN_x_e", 9)):
        assert_f32_close("reset " + k, st[idx], want[k])
    assert np.array_equal(st[1], o.A_n) and np.array_equal(st[10], o.nC_e)
    mu = [[0.1, 0.1], [0.1, 0.1, 0.1]]
    maddpg = RL.MADDPG(1e-7, 1, 0.95, 0.99, 200, 200, 1000, 3, [2, 3], mu, mu, mu)
    m = gm.model
    x_p, A_p = st[6], st[7]
    orig = random.random
    try:
        for s in range(4):
            geo, topo = maddpg.agents[s % 3].act(st[0], st[1], st[2], st[3], st[4], x_p, A_p)
            assert geo.shape == (20, 2) and topo.shape == (20, 3)
            up = np.array([np.float32(n.max_up) for n in m.nodes])
            down = np.array([np.float32(n.max_down) for n in m.nodes])
            coin = s % 2 == 0
            random.random = (lambda: 0.75) if coin else (lambda: 0.25)
            set_node, set_elem = np.array(st[8], np.float32), np.array(st[9], np.float32)
            want = o.step(set_node, set_elem, up, down, geo.copy(), topo.copy(), coin)
            point, S = game._game_modify(st[8], st[9], st[10], [geo, topo])
            assert_f32_close("step %d point" % s, np.array(point, dtype=np.float32), want["point"])
            for k, idx in (("x_n", 0), ("A_s", 2), ("A_n_ts", 3), ("A_n_cs", 4), ("nN_x_n", 8), ("nN_x_e", 9)):
                assert_f32_close("step %d %s" % (s, k), S[idx], want[k])
            assert [float(n.coord[1]) for n in m.nodes] == want["y"].tolist()
            assert [e.section_no for e in m.elements] == want["section"].tolist()
            st = S
    finally:
        random.random = orig
