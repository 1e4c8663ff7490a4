"""GPU: the env-step kernel on the ten 6 x 2 training families (families.TRAIN_FAMILIES), the NX = 6 instantiation that the
training driver's mixed batches (MixedTrussEnv, MixedHostRollout) run on.

* constants and reset of every family, through single-family handles and one mixed handle, against the oracle and the
  reference's recorded reset;
* the transitions recorded from the reference (tests/golden/twins_train.npz, twins_adversarial.npz) through the kernel;
* a saturated walk (heights driven to d_min / y_max) against the C oracle and the extended-precision solve;
* a whole production mixed batch, every environment against the C oracle (grouped by family) and the Python oracle, with
  random and then trained-actor actions.  B = 4096 is more than the resident warps at 2 CTAs per SM, so warps step a
  second environment, of another family, after their first;
* B = 16384 mixed batches (several environments per warp at any occupancy) bit for bit against single-family batches, in
  id layouts that change the family between the environments of a warp, keep it, or put a bad id before a good one.

Random walks, adversarial transitions and solve_only of every training family, and the size-independent properties at
B = 16384, are in test_gpu_parity.py.  Since the five shapes of one truss type share every table but the targets
(test_train_families_cpu.py), a kernel that read another shape's tables would differ only in the target column of x_n /
nN_x_n and in point / point64 (obj2 = sum |target - y|: train1 and train2 share int_obj2 and the sum of their targets, so
between those two point differs only once a height is below a target): the production-batch test compares those fields
against the oracle of each environment's own family."""
import functools
import json

import numpy as np
import pytest

from mop_truss_marl_b200.families import TRAIN_FAMILIES
from test_gpu_mixed import Twin, assert_bits
from test_gpu_parity import compare_env, cpu, load_state
from test_oracle_twins import TRAIN_RUNS, twins
from util import F32_FIELDS, FP64_TOL, nrm, ulp_diff

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

WALKS = ("uniform", "small_actions", "saturated")
EPS = np.finfo(np.float64).eps


@functools.lru_cache(maxsize=None)
def oracle(name):
    from oracle.truss_oracle import TrussOracle
    return TrussOracle(name)


@functools.lru_cache(maxsize=None)
def c_oracle(name):
    from oracle.c_oracle import COracle
    return COracle(name)


def cond_of(name, y, section):
    return float(np.linalg.cond(oracle(name).solve_only(y, section)["K"]))


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ================================================= constants and reset ==================================================
def reset_checks(env, i, name):
    o = oracle(name)
    want = o.reset()
    compare_env(env, i, want, point=want["point"], tag="%s reset[%d]" % (name, i))
    assert nrm(cpu(env.point64[i]), want["point64"]) <= FP64_TOL, name
    if name in TRAIN_RUNS:                                  # the reset the reference recorded
        g, p = twins("twins_train"), name + "/reset_"
        rec = {k[len(p):]: g[k] for k in g.files if k.startswith(p)}
        compare_env(env, i, rec, point=rec["point"], tag="%s recorded reset[%d]" % (name, i))


@pytest.mark.parametrize("name", TRAIN_FAMILIES)
def test_constants_and_reset_vs_oracle(name):
    from mop_truss_marl_b200 import batched_env
    o = oracle(name)
    env = batched_env.BatchedTrussEnv(name, 3)
    assert np.array_equal(cpu(env.A_n), o.A_n) and np.array_equal(cpu(env.mask), o.mask)
    assert np.array_equal(cpu(env.nC_e), o.nC_e)
    assert np.array_equal(env.int_obj, np.array([o.int_obj1, o.int_obj2], dtype=np.float32))
    env.reset()
    torch.cuda.synchronize()
    for i in range(3):
        reset_checks(env, i, name)


def test_mixed_reset_vs_oracle():
    from mop_truss_marl_b200 import batched_env
    rng = np.random.RandomState(3)
    ids = np.concatenate([np.arange(10), rng.randint(0, 10, size=27)]).astype(np.uint8)
    rng.shuffle(ids)
    mix = batched_env.MixedTrussEnv(TRAIN_FAMILIES, len(ids))
    o0 = oracle(TRAIN_FAMILIES[0])
    assert np.array_equal(cpu(mix.A_n), o0.A_n) and np.array_equal(cpu(mix.nC_e), o0.nC_e)
    assert np.array_equal(mix.int_obj, np.array([[oracle(n).int_obj1, oracle(n).int_obj2] for n in TRAIN_FAMILIES], np.float32))
    mix.reset(dev(ids))
    torch.cuda.synchronize()
    for i, f in enumerate(ids):
        reset_checks(mix, i, TRAIN_FAMILIES[f])


# ================================================= recorded transitions =================================================
@pytest.mark.parametrize("run", TRAIN_RUNS)
@pytest.mark.parametrize("walk", WALKS)
def test_recorded_walks_through_the_kernel(run, walk):
    from mop_truss_marl_b200 import batched_env
    g, p = twins("twins_train"), "%s/%s/" % (run, walk)
    T = len(g[p + "in_coin"])
    env = batched_env.BatchedTrussEnv(run, T)
    load_state(env, g[p + "in_set_node"], g[p + "in_set_element"], g[p + "in_max_up"], g[p + "in_max_down"])
    a_geo, a_topo = dev(g[p + "in_a_geo"]), dev(g[p + "in_a_topo"])
    env.step(a_geo, a_topo, dev(g[p + "in_coin"].astype(np.uint8)))
    torch.cuda.synchronize()
    assert np.array_equal(cpu(a_geo), g[p + "out_a_geo"]) and np.array_equal(cpu(a_topo), g[p + "out_a_topo"])
    for i in range(T):
        want = {k[len(p + "out_"):]: g[k][i] for k in g.files if k.startswith(p + "out_")}
        compare_env(env, i, want, point=want["point"], cond=cond_of(run, want["y"], want["section"]), tag="%s %s[%d]" % (run, walk, i))


@pytest.mark.parametrize("run", TRAIN_RUNS)
def test_recorded_adversarial_through_the_kernel(run):
    from mop_truss_marl_b200 import batched_env
    from util import assert_f32_close
    g, p = twins("twins_adversarial"), run + "/"
    T = len(g[p + "in_coin"])
    env = batched_env.BatchedTrussEnv(run, T)
    load_state(env, g[p + "in_set_node"], g[p + "in_set_element"], g[p + "in_max_up"], g[p + "in_max_down"])
    a_geo, a_topo = dev(g[p + "in_a_geo"]), dev(g[p + "in_a_topo"])
    env.step(a_geo, a_topo, dev(g[p + "in_coin"].astype(np.uint8)))
    torch.cuda.synchronize()
    assert np.array_equal(cpu(a_geo), g[p + "out_a_geo"], equal_nan=True) and np.array_equal(cpu(a_topo), g[p + "out_a_topo"])
    for i in range(T):
        tag = "%s adversarial[%d]" % (run, i)
        assert np.array_equal(cpu(env.y[i]), g[p + "out_y"][i]), tag
        assert np.array_equal(cpu(env.nN_x_e[i])[:, 0].astype(np.int32), g[p + "out_section"][i]), tag
        mr = cpu(env.move_range[i])
        assert np.array_equal(mr[:, 0], g[p + "out_max_up"][i]) and np.array_equal(mr[:, 1], g[p + "out_max_down"][i]), tag
        if g[p + "well"][i]:                                # cond(K) < 1e6: the FEM and the observation tensors too
            assert int(env.status[i]) == 0, tag
            assert nrm(cpu(env.d[i]), g[p + "out_d"][i]) <= FP64_TOL, tag
            for k in ("x_n", "nN_x_n", "nN_x_e"):
                assert_f32_close(tag + " " + k, cpu(getattr(env, k)[i]), g[p + "out_" + k][i])


# ================================================= whole batches against the oracles ===================================
def c_oracle_batch(families, ids, inp):
    """the C oracle's step of every environment with the tables of its own family, in batch order"""
    B = len(ids)
    want = {"a_geo": inp["a_geo"].copy(), "a_topo": inp["a_topo"].copy()}
    for f, name in enumerate(families):
        rows = np.nonzero(ids == f)[0]
        if not len(rows):
            continue
        ag, at = want["a_geo"][rows], want["a_topo"][rows]                    # fancy indexing: contiguous copies
        out = c_oracle(name).step(inp["set_node"][rows], inp["set_elem"][rows], ag, at, inp["coin"][rows], inp["stale"][rows])
        want["a_geo"][rows], want["a_topo"][rows] = ag, at                  # clipped in place
        for k, v in out.items():
            if k not in want:
                want[k] = np.empty((B,) + v.shape[1:], v.dtype)
            want[k][rows] = v
    return want


PY_FIELDS = F32_FIELDS + ("reactions", "point64")


def py_oracle_batch(families, ids, inp, rows):
    """the Python oracle's observation tensors, reactions and point64 for the environments ``rows``"""
    out = {k: [] for k in PY_FIELDS}
    for b in rows:
        w = oracle(families[ids[b]]).step(inp["set_node"][b], inp["set_elem"][b], inp["stale"][b, :, 0], inp["stale"][b, :, 1],
                                          inp["a_geo"][b].copy(), inp["a_topo"][b].copy(), bool(inp["coin"][b]))
        for k in PY_FIELDS:
            out[k].append(w[k])
    return {k: np.stack(v) for k, v in out.items()}


def step_and_check(env, families, ids, a_geo, a_topo, coin, tag, stats, max_outside, r_errs):
    """Steps ``env`` (whose family ids are ``ids``) once and checks every environment.  Returns the names of the fields
    that failed.

    * C oracle, every environment: clipped actions, heights (float64 bits), weak flags, sections, move range bit-exact;
      d / axial / ratio / U counted against the flat 1e-9, and every environment's displacements within 20 eps cond(K)
      of the extended-precision solve (their errors in units of eps cond(K), the kernel's and the oracle's, are appended
      to ``r_errs`` for population_rule); the compression flags where the member force is not a rounding-level zero;
      point within 2 ulp.
    * Python oracle, every environment inside the flat 1e-9 with no rounding-level member force: the float32 observation
      tensors within 2 ulp and their 0 / 1 columns exact, reactions and point64 within 1e-9."""
    from oracle import exact_fem
    B = len(ids)
    inp = {"set_node": cpu(env.nN_x_n).copy(), "set_elem": cpu(env.nN_x_e).copy(), "stale": cpu(env.move_range).copy(),
           "a_geo": cpu(a_geo).copy(), "a_topo": cpu(a_topo).copy(), "coin": cpu(coin).copy()}
    want = c_oracle_batch(families, ids, inp)
    env.step(a_geo, a_topo, coin)
    torch.cuda.synchronize()
    failed = []

    def expect(ok, what):
        if not ok:
            failed.append(what)

    expect(int(np.abs(cpu(env.status)).max()) == 0 and int(want["status"].max()) == 0, "status")
    expect(np.array_equal(cpu(a_geo), want["a_geo"]) and np.array_equal(cpu(a_topo), want["a_topo"]), "clipped actions")
    expect(np.array_equal(cpu(env.y), want["y"]), "y")
    expect(np.array_equal(cpu(env.y_weak), want["weak"]), "weak flags")
    expect(np.array_equal(cpu(env.nN_x_e)[:, :, 0].astype(np.int32), want["section"]), "section")
    expect(np.array_equal(cpu(env.move_range), want["move_range"]), "move range")
    # FP64 against the C oracle, counted; against the exact displacements, every environment
    got = {k: cpu(getattr(env, k)) for k in ("d", "axial", "ratio", "U")}
    errs = {k: np.abs(got[k] - want[k]).max(axis=1) / np.abs(want[k]).max(axis=1) for k in ("d", "axial", "ratio")}
    errs["U"] = np.abs(got["U"] - want["U"]) / np.abs(want["U"])
    worst = np.maximum.reduce([errs[k] for k in errs])
    outside = worst > FP64_TOL
    expect(worst.max() <= 1e-6, "FP64 beyond 1e-6")
    e_gpu, e_orc, cond = np.empty(B), np.empty(B), np.empty(B)
    for f, name in enumerate(families):
        rows = np.nonzero(ids == f)[0]
        if len(rows):
            mesh = oracle(name).mesh
            d_exact = exact_fem.exact_displacements(mesh, want["y"][rows], want["section"][rows])
            e_gpu[rows] = exact_fem.rel_err(got["d"][rows], d_exact)
            e_orc[rows] = exact_fem.rel_err(want["d"][rows], d_exact)
            cond[rows] = exact_fem.cond2(mesh, want["y"][rows], want["section"][rows])
    expect((e_gpu <= np.maximum(20 * EPS * cond, 1e-13)).all(), "d beyond 20 eps cond from the exact solve")
    r_errs.append((e_gpu / (EPS * cond), e_orc / (EPS * cond)))
    if max_outside is not None:
        expect(outside.sum() <= max_outside, "environments outside the flat 1e-9")
    expect(not outside.any() or cond[outside].min() > 1e5, "a well-conditioned environment outside the flat 1e-9")
    ax = want["axial"]
    clear = np.abs(ax) > 1e-7 * np.abs(ax).max(axis=1, keepdims=True)
    mism = cpu(env.nN_x_e)[:, :, 4].astype(np.int32) != want["iscompress"]
    expect(not (mism & clear).any(), "iscompress")
    u_point = ulp_diff(cpu(env.point), want["point"]).max(axis=1)
    expect(u_point.max() <= 2, "point")
    # the Python oracle: observation tensors, reactions, point64
    rows = np.nonzero(~outside & clear.all(axis=1))[0]
    pw = py_oracle_batch(families, ids, inp, rows)
    u = {k: ulp_diff(cpu(getattr(env, k))[rows], pw[k]).reshape(len(rows), -1).max(axis=1) for k in F32_FIELDS}
    for k in F32_FIELDS:
        expect(u[k].max() <= 2, k)
    for k, cols in (("nN_x_n", [11]), ("nN_x_e", [0, 3, 4, 6, 13, 20])):
        expect(np.array_equal(cpu(getattr(env, k))[rows][:, :, cols], pw[k][:, :, cols]), k + " flags")
    expect(np.array_equal(cpu(env.x_n)[rows][:, :, 12] > 0.5, pw["x_n"][:, :, 12] > 0.5), "x_n flags")
    e_py = {}
    for k in ("reactions", "point64"):
        g_k = cpu(getattr(env, k))[rows]
        e_py[k] = np.abs(g_k - pw[k]).max(axis=1) / np.abs(pw[k]).max(axis=1)
        expect(e_py[k].max() <= FP64_TOL, k)
    # per family, the largest errors of this step merged into ``stats``
    pos = np.full(B, -1)
    pos[rows] = np.arange(len(rows))
    for f, name in enumerate(families):
        sel = np.nonzero(ids == f)[0]
        if not len(sel):
            continue
        sel_py = pos[sel][pos[sel] >= 0]
        s = stats.setdefault(name, {"env-steps": 0, "outside flat 1e-9": 0, "python-checked env-steps": 0})
        s["env-steps"] += int(len(sel))
        s["outside flat 1e-9"] += int(outside[sel].sum())
        s["python-checked env-steps"] += int(len(sel_py))
        new = {"max cond(K)": cond[sel].max(), "max kernel error vs exact": e_gpu[sel].max(),
               "max oracle error vs exact": e_orc[sel].max(), "point ulp": u_point[sel].max()}
        new.update({"%s vs C oracle" % k: errs[k][sel].max() for k in errs})
        if len(sel_py):
            new.update({"%s ulp" % k: u[k][sel_py].max() for k in F32_FIELDS})
            new.update({"%s vs Python oracle" % k: e_py[k][sel_py].max() for k in e_py})
        for k, v in new.items():
            s[k] = max(s.get(k, 0), float(v))
    return ["%s: %s" % (tag, f) for f in failed]


def population_rule(r_errs):
    """As a population the kernel's displacement errors, in units of eps cond(K), are no larger than the oracle's (the
    rule of test_gpu_parity.test_ill_conditioned_solves_vs_extended_precision), pooled over a whole walk: per step, a few
    hundred environments make the maximum a noisy statistic.  (A LAPACK Cholesky solve of the saturated walk's
    geometries is up to 1.85 times LU's maximum on single steps, 1.04 times over the walk.)"""
    r_gpu, r_orc = np.concatenate([g for g, _ in r_errs]), np.concatenate([o for _, o in r_errs])
    stats = {"max": [float(r_gpu.max()), float(r_orc.max())], "median": [float(np.median(r_gpu)), float(np.median(r_orc))]}
    print("error / (eps cond(K)), kernel and oracle:", json.dumps(stats))
    failed = []
    if r_gpu.max() > 2 * r_orc.max():
        failed.append("d further from the exact solve than the oracle (max)")
    if np.median(r_gpu) > 2 * np.median(r_orc):
        failed.append("d further from the exact solve than the oracle (median)")
    return failed


def report(title, stats):
    print()
    for name in sorted(stats):
        print(title, name, json.dumps({k: (v if isinstance(v, int) else float("%.3g" % v)) for k, v in stats[name].items()}))


def test_saturated_walk_vs_oracle_and_exact_solve():
    """Actions held at 0 or 1 for ten steps drive the heights towards d_min (0.2 m) or y_max: every environment of all ten
    families against the C and Python oracles, and its displacements against the extended-precision solve (where cond(K)
    grows, the flat 1e-9 is not asked; the kernel must stay within 20 eps cond of the exact solve and be no further from
    it than the oracle).  The largest cond(K) reached is printed per family."""
    from mop_truss_marl_b200 import batched_env
    rng = np.random.RandomState(17)
    B, N = 640, 12
    ids = (np.arange(B) % 10).astype(np.uint8)
    rng.shuffle(ids)
    mix = batched_env.MixedTrussEnv(TRAIN_FAMILIES, B)
    mix.reset(dev(ids))
    # per environment: every node up, every node down, or each node its own saturated direction, fixed for the walk
    kind = rng.randint(0, 3, size=B)
    up = np.where(kind[:, None] == 0, True, np.where(kind[:, None] == 1, False, rng.rand(B, N) < 0.5))
    geo = np.where(up[..., None], np.float32([1, 0]), np.float32([0, 1])).astype(np.float32)
    stats, failed, r_errs = {}, [], []
    for s in range(10):
        topo = (rng.rand(B, N, 3) < 0.5).astype(np.float32)
        coin = (rng.rand(B) >= 0.5).astype(np.uint8)
        failed += step_and_check(mix, TRAIN_FAMILIES, ids, dev(geo), dev(topo), dev(coin), "saturated step %d" % s, stats, None,
                                 r_errs)
    report("saturated walk", stats)
    failed += population_rule(r_errs)
    assert not failed, "; ".join(failed)


def test_production_mixed_batch_vs_oracles():
    """MixedTrussEnv(TRAIN_FAMILIES, 4096) with seeded random ids: reset, three steps of out-of-range, ordinary and small
    random actions, then two steps of the trained actor (agent 1 of the 2000pickle_base checkpoint, with noise).  Every
    environment of every step is checked (step_and_check); the per-family largest errors are printed."""
    from mop_truss_marl_b200 import actor, batched_env
    from test_gpu_actor import trained_weights
    B, N = 4096, 12
    ids = np.random.RandomState(2024).randint(0, 10, size=B).astype(np.uint8)
    mix = batched_env.MixedTrussEnv(TRAIN_FAMILIES, B)
    mix.reset(dev(ids))
    g = torch.Generator(device="cuda").manual_seed(7)
    pol = actor.BatchedActor(trained_weights(1), N, B)
    x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50], device="cuda").repeat(B, 1, 1).contiguous()
    A_p = torch.ones(B, 1, 1, device="cuda")
    stats, failed, r_errs = {}, [], []
    for s in range(5):
        if s < 3:
            scale = (1.3, 0.6, 0.25)[s]                      # out-of-range, ordinary and small actions
            a_geo = (torch.rand(B, N, 2, device="cuda", generator=g) * scale - 0.05).contiguous()
            a_topo = (torch.rand(B, N, 3, device="cuda", generator=g) * 1.2 - 0.1).contiguous()
        else:
            a_geo, a_topo = pol.act(mix.x_n, mix.A_n, mix.A_s, mix.A_n_ts, mix.A_n_cs, x_p, A_p)
        coin = (torch.rand(B, device="cuda", generator=g) >= 0.5).to(torch.uint8)
        failed += step_and_check(mix, TRAIN_FAMILIES, ids, a_geo, a_topo, coin, "step %d" % s, stats, B // 50, r_errs)
    pol.check()
    report("production batch", stats)
    failed += population_rule(r_errs)
    assert not failed, "; ".join(failed)


# ================================================= several environments per warp =======================================
LAYOUTS = ("random", "alternating", "runs", "bad_ids")


@pytest.mark.parametrize("layout", LAYOUTS)
def test_several_environments_per_warp_bit_identical(layout):
    """B = 16384 (at least three environments per warp at up to 4 CTAs per SM): the mixed batch bit for bit against
    single-family batches of the same environments.  Warp w steps w, w + W, w + 2W, ... for W resident warps; the layouts
    need no W: random ids; b % 10 (W = 2368 is no multiple of 10, so the shape changes between a warp's environments;
    W being even, the truss type, and with it the constant pool columns, does not);
    runs of 1024 environments of one family; random ids with 3 % bad ids, so that warps step a good environment right
    after a bad one (which gets TFEM_STATUS_BAD_FAMILY, leaves its actions unclipped and its outputs unwritten)."""
    from mop_truss_marl_b200 import capi
    B, N = 16384, 12
    rng = np.random.RandomState(LAYOUTS.index(layout) + 40)
    b = np.arange(B)
    ids = {"random": rng.randint(0, 10, size=B), "alternating": b % 10, "runs": (b // 1024) % 10,
           "bad_ids": rng.randint(0, 10, size=B)}[layout].astype(np.uint8)
    bad = np.zeros(B, bool)
    if layout == "bad_ids":
        bad = rng.rand(B) < 0.03
        ids[bad] = rng.choice(np.array([10, 17, 255], np.uint8), size=int(bad.sum()))
    tw = Twin(TRAIN_FAMILIES, ids)
    tw.reset()
    tw.compare("reset")
    bad_rows, good_rows = dev(np.nonzero(bad)[0]), dev(np.nonzero(~bad)[0])
    for s in range(3):
        if s == 0:
            a_geo, a_topo = rng.rand(B, N, 2), rng.rand(B, N, 3)
        elif s == 1:
            a_geo, a_topo = 0.3 * rng.rand(B, N, 2), 0.3 * rng.rand(B, N, 3)
        else:
            a_geo, a_topo = rng.randn(B, N, 2), rng.randn(B, N, 3)
        a_geo, a_topo = dev(a_geo.astype(np.float32)), dev(a_topo.astype(np.float32))
        raw = (a_geo.clone(), a_topo.clone())
        tw.step(a_geo, a_topo, dev((rng.rand(B) >= 0.5).astype(np.uint8)))
        tw.compare("%s step %d" % (layout, s))
        st = tw.mix.status
        assert int(st[good_rows].abs().max()) == 0
        if bad.any():
            assert bool((st[bad_rows] == capi.STATUS_BAD_FAMILY).all())
            assert_bits(a_geo[bad_rows], raw[0][bad_rows], "bad-id a_geo")
            assert_bits(a_topo[bad_rows], raw[1][bad_rows], "bad-id a_topo")
