"""GPU parity tests: the CUDA path, called through the C ABI, against the golden vectors recorded from the
reference and against the CPU oracle on seeded random inputs (SURVEY.md section 8c).

  bit-exact ... post-transition heights, sections, move range, in-place clipped actions, 0/1 flags
  1e-9 ....... d, axial force, stress ratio, U, reactions (normwise, FEM-coerced float64 reference)
  2 ulp ...... float32 observation tensors and the objective point
"""
import ctypes as C
import os

import numpy as np
import pytest

from mop_truss_marl_b200.families import SYM_NONE, TRAIN_FAMILIES
from util import FAMILY_NAMES, F32_FIELDS, FP64_TOL, assert_f32_close, load_golden, nrm

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def envmod():
    from mop_truss_marl_b200 import batched_env
    return batched_env


def make_env(envmod, name, B):
    return envmod.BatchedTrussEnv(name, B, device="cuda:0")


def cpu(t):
    return t.detach().cpu().numpy()


def load_state(env, set_node, set_element, max_up, max_down):
    env.nN_x_n.copy_(torch.from_numpy(np.ascontiguousarray(set_node)))
    env.nN_x_e.copy_(torch.from_numpy(np.ascontiguousarray(set_element)))
    env.move_range.copy_(torch.from_numpy(np.stack([max_up, max_down], axis=-1).astype(np.float32)))


def fp64_tol(cond=None):
    """1e-9 (north_star) over the conditioning range the reference reaches in normal play (cond(K) <= 1e6,
    SURVEY.md section 0); beyond that the reference's own LU result is only good to ~eps*cond, so the
    tolerance grows linearly with cond (saturated golden walks reach cond 1.9e8)."""
    if cond is None or cond <= 1e6:
        return FP64_TOL
    return FP64_TOL * cond / 1e6


def compare_env(env, i, want, point=None, tag="", cond=None):
    """want: dict with the oracle/golden fields of ONE environment"""
    raw_n, raw_e = cpu(env.nN_x_n[i]), cpu(env.nN_x_e[i])
    # bit-exact
    assert np.array_equal(raw_n[:, 1], want["y"].astype(np.float32)), tag + " y"
    assert np.array_equal(cpu(env.y[i]), want["y"]), tag + " y (float64 bits)"
    assert np.array_equal(cpu(env.y_weak[i]).astype(bool), want["y_weak"]), tag + " weak flags"
    assert np.array_equal(raw_e[:, 0].astype(np.int32), want["section"]), tag + " section"
    mr = cpu(env.move_range[i])
    assert np.array_equal(mr[:, 0], want["max_up"]) and np.array_equal(mr[:, 1], want["max_down"]), tag + " move range"
    assert np.array_equal(raw_e[:, 4].astype(np.int32), want["iscompress"]), tag + " iscompress"
    assert int(env.status[i]) == 0
    # float64
    for k in ("d", "axial", "ratio", "reactions"):
        e = nrm(cpu(getattr(env, k)[i]), want[k])
        assert e <= fp64_tol(cond), "%s %s: %.3e (cond %s)" % (tag, k, e, cond)
    assert abs(float(env.U[i]) - float(want["U"])) <= fp64_tol(cond) * abs(float(want["U"])), tag + " U"
    # float32 tensors
    for k in F32_FIELDS:
        assert_f32_close(tag + " " + k, cpu(getattr(env, k)[i]), want[k])
    for k, cols in (("nN_x_n", [11]), ("nN_x_e", [0, 3, 4, 6, 13, 20])):
        assert np.array_equal(cpu(getattr(env, k)[i])[:, cols], want[k][:, cols]), tag + " flags " + k
    assert np.array_equal(cpu(env.x_n[i])[:, 12] > 0.5, want["x_n"][:, 12] > 0.5)
    if point is not None:
        assert_f32_close(tag + " point", cpu(env.point[i]), point)


@pytest.mark.parametrize("name", FAMILY_NAMES)
def test_constants_and_reset_vs_golden(envmod, name):
    g = load_golden(name)
    env = make_env(envmod, name, 3)
    assert np.array_equal(cpu(env.A_n), g["A_n"]) and np.array_equal(cpu(env.mask), g["mask"])
    assert np.array_equal(cpu(env.nC_e), g["nC_e"])
    env.reset()
    torch.cuda.synchronize()
    want = {k[len("reset_"):]: v for k, v in g.items() if k.startswith("reset_")}
    for i in range(3):
        compare_env(env, i, want, tag="reset[%d]" % i)


@pytest.mark.parametrize("name", FAMILY_NAMES)
def test_transitions_vs_golden(envmod, name):
    g = load_golden(name)
    T = g["tr_mode"].shape[0]
    env = make_env(envmod, name, T)
    load_state(env, g["tr_in_set_node"], g["tr_in_set_element"], g["tr_in_max_up"], g["tr_in_max_down"])
    a_geo = torch.from_numpy(g["tr_in_a_geo"].copy()).cuda()
    a_topo = torch.from_numpy(g["tr_in_a_topo"].copy()).cuda()
    coin = torch.from_numpy(g["tr_in_coin"].copy()).cuda()
    env.step(a_geo, a_topo, coin)
    torch.cuda.synchronize()
    assert np.array_equal(cpu(a_geo), g["tr_out_a_geo"]) and np.array_equal(cpu(a_topo), g["tr_out_a_topo"])
    from oracle.truss_oracle import TrussOracle
    o = TrussOracle(name)
    for i in range(T):
        want = {k[len("tr_out_"):]: v[i] for k, v in g.items() if k.startswith("tr_out_")}
        cond = float(np.linalg.cond(o.solve_only(want["y"], want["section"])["K"]))
        compare_env(env, i, want, point=g["tr_out_point"][i], cond=cond,
                    tag="%s tr[%d] mode %d" % (name, i, g["tr_mode"][i]))


@pytest.mark.parametrize("name", FAMILY_NAMES + TRAIN_FAMILIES)
def test_random_walk_vs_oracle(envmod, name):
    """every environment feeds its own state back; the oracle follows each one (the four test/ families and the ten
    6 x 2 train/code families: 12 nodes, mixed spans, no symmetry step)"""
    from oracle.truss_oracle import TrussOracle
    o = TrussOracle(name)
    B = 48 if o.mesh.N <= 16 else 16
    steps = 4
    env = make_env(envmod, name, B)
    env.reset()
    rng = np.random.RandomState(7)
    N = o.mesh.N
    for s in range(steps):
        scale = 1.0 if s % 2 == 0 else 0.3
        a_geo = (rng.rand(B, N, 2) * scale).astype(np.float32)
        a_topo = (rng.rand(B, N, 3) * np.array([scale, scale, 1.0])).astype(np.float32)
        if s == 2:
            a_geo = (rng.randn(B, N, 2) + 0.5).astype(np.float32)
        coin = (rng.rand(B) >= 0.5).astype(np.uint8)
        set_node, set_elem, mr = cpu(env.nN_x_n).copy(), cpu(env.nN_x_e).copy(), cpu(env.move_range).copy()
        tg, tt, tc = torch.from_numpy(a_geo.copy()).cuda(), torch.from_numpy(a_topo.copy()).cuda(), torch.from_numpy(coin).cuda()
        env.step(tg, tt, tc)
        torch.cuda.synchronize()
        for i in range(B):
            ag, at = a_geo[i].copy(), a_topo[i].copy()
            want = o.step(set_node[i], set_elem[i], mr[i, :, 0], mr[i, :, 1], ag, at, bool(coin[i]))
            assert np.array_equal(cpu(tg[i]), ag) and np.array_equal(cpu(tt[i]), at)
            compare_env(env, i, want, point=want["point"], tag="%s step %d env %d" % (name, s, i))
            assert nrm(cpu(env.point64[i]), want["point64"]) <= FP64_TOL


@pytest.mark.parametrize("name", FAMILY_NAMES + TRAIN_FAMILIES)
def test_adversarial_transition_vs_oracle(envmod, name):
    """ties, exact 0/1, out-of-range, inf / NaN geometry actions and absurd stale move ranges: the
    post-transition heights (float64 bits + weak flags), sections, clipped actions and new move range must be
    bit-exact; the FEM is compared only where the oracle can solve the resulting geometry"""
    from oracle.truss_oracle import TrussOracle
    from util import adversarial_actions, adversarial_move_range
    o = TrussOracle(name)
    N = o.mesh.N
    B = 64 if N == 16 else 24
    rng = np.random.RandomState(3)
    env = make_env(envmod, name, B)
    env.reset()
    for s in range(3):
        acts = [adversarial_actions(rng, N) for _ in range(B)]
        a_geo = np.stack([a for a, _ in acts]); a_topo = np.stack([t for _, t in acts])
        mrs = [adversarial_move_range(rng, N) for _ in range(B)]
        mr = np.stack([np.stack([u, d], axis=-1) for u, d in mrs]).astype(np.float32)
        coin = (rng.rand(B) >= 0.5).astype(np.uint8)
        env.move_range.copy_(torch.from_numpy(mr))
        set_node, set_elem = cpu(env.nN_x_n).copy(), cpu(env.nN_x_e).copy()
        tg, tt = torch.from_numpy(a_geo.copy()).cuda(), torch.from_numpy(a_topo.copy()).cuda()
        env.step(tg, tt, torch.from_numpy(coin).cuda())
        torch.cuda.synchronize()
        bad = 0
        for i in range(B):
            ag, at = a_geo[i].copy(), a_topo[i].copy()
            try:
                want = o.step(set_node[i], set_elem[i], mr[i, :, 0], mr[i, :, 1], ag, at, bool(coin[i]))
            except Exception:
                # the oracle (like the reference) cannot solve this geometry; the transition is still checked below
                want = None
            assert np.array_equal(cpu(tg[i]), ag, equal_nan=True) and np.array_equal(cpu(tt[i]), at)
            if want is None:
                bad += 1
                assert int(env.status[i]) != 0
                continue
            assert np.array_equal(cpu(env.y[i]), want["y"]), (name, s, i)
            assert np.array_equal(cpu(env.y_weak[i]).astype(bool), want["y_weak"])
            assert np.array_equal(cpu(env.nN_x_e[i])[:, 0].astype(np.int32), want["section"])
            got_mr = cpu(env.move_range[i])
            assert np.array_equal(got_mr[:, 0], want["max_up"]) and np.array_equal(got_mr[:, 1], want["max_down"])
            if np.isfinite(want["d"]).all() and np.linalg.cond(o.solve_only(want["y"], want["section"])["K"]) < 1e6:
                assert int(env.status[i]) == 0
                assert nrm(cpu(env.d[i]), want["d"]) <= FP64_TOL
                assert_f32_close("x_n", cpu(env.x_n[i]), want["x_n"])
                assert_f32_close("nN_x_e", cpu(env.nN_x_e[i]), want["nN_x_e"])
        assert bad < B
        # continue the walk from a sane state so later steps exercise new corners
        env.reset() if s == 1 else None


@pytest.mark.parametrize("name", ["small_bridge", "large_roof"])
def test_step_host_equals_step(envmod, name):
    g = load_golden(name)
    T = g["tr_mode"].shape[0]
    env = make_env(envmod, name, T)
    load_state(env, g["tr_in_set_node"], g["tr_in_set_element"], g["tr_in_max_up"], g["tr_in_max_down"])
    a_geo = torch.from_numpy(g["tr_in_a_geo"].copy()).cuda(); a_topo = torch.from_numpy(g["tr_in_a_topo"].copy()).cuda()
    env.step(a_geo, a_topo, torch.from_numpy(g["tr_in_coin"].copy()).cuda())
    torch.cuda.synchronize()
    mr = np.stack([g["tr_in_max_up"], g["tr_in_max_down"]], axis=-1).astype(np.float32)
    hg, ht = g["tr_in_a_geo"].copy(), g["tr_in_a_topo"].copy()
    out = envmod.step_host(env.handle, g["tr_in_set_node"].copy(), g["tr_in_set_element"].copy(), mr, hg, ht,
                           g["tr_in_coin"].copy())
    for k in F32_FIELDS + ("point", "point64", "d", "axial", "ratio", "U", "reactions", "status", "y", "y_weak"):
        assert np.array_equal(out[k], cpu(getattr(env, k))), k
    assert np.array_equal(mr, cpu(env.move_range)) and np.array_equal(hg, cpu(a_geo)) and np.array_equal(ht, cpu(a_topo))


@pytest.mark.parametrize("name", ("small_roof", "large_bridge") + TRAIN_FAMILIES)
def test_solve_only_vs_oracle(envmod, name):
    from oracle.truss_oracle import TrussOracle
    o = TrussOracle(name)
    m = o.mesh
    rng = np.random.RandomState(11)
    B = 64
    y = np.zeros((B, m.N))
    y[:, m.N // 2:] = 1.0 + rng.rand(B, m.N // 2) * (m.y_max - 1.0)
    y[:, 1:m.N // 2 - 1] = rng.rand(B, m.N // 2 - 2) * 0.6
    sec = rng.randint(0, 5, size=(B, m.E)).astype(np.int32)
    env = make_env(envmod, name, 1)
    out = env.solve_only(torch.from_numpy(y).cuda(), torch.from_numpy(sec).cuda())
    torch.cuda.synchronize()
    for i in range(B):
        want = o.solve_only(y[i], sec[i])
        assert int(out["status"][i]) == 0
        for k in ("d", "axial", "ratio", "reactions"):
            assert nrm(cpu(out[k][i]), want[k]) <= FP64_TOL, (k, i)
        assert abs(float(out["U"][i]) - want["U"]) <= FP64_TOL * abs(want["U"])


@pytest.mark.parametrize("name", ["large_bridge", "large_roof", "small_bridge"])
def test_dense_dmma_solve_vs_oracle_and_banded(envmod, name):
    """the north_star's dense blocked Cholesky with DMMA trailing updates (tfem_solve_dense_dmma) against the oracle
    and against the banded production solve, on the same geometries"""
    from oracle.truss_oracle import TrussOracle
    o = TrussOracle(name)
    m = o.mesh
    rng = np.random.RandomState(12)
    B = 200
    y = np.zeros((B, m.N))
    y[:, m.N // 2:] = 1.0 + rng.rand(B, m.N // 2) * (m.y_max - 1.0)
    y[:, 1:m.N // 2 - 1] = rng.rand(B, m.N // 2 - 2) * 0.6
    sec = rng.randint(0, 5, size=(B, m.E)).astype(np.int32)
    env = make_env(envmod, name, 1)
    yt, st = torch.from_numpy(y).cuda(), torch.from_numpy(sec).cuda()
    d, status = env.solve_dense_dmma(yt, st)
    banded = env.solve_only(yt, st)
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0
    for i in range(B):
        assert nrm(cpu(d[i]), cpu(banded["d"][i])) <= FP64_TOL, i
    for i in range(0, B, 25):
        assert nrm(cpu(d[i]), o.solve_only(y[i], sec[i])["d"]) <= FP64_TOL, i


def test_degenerate_geometry_sets_status(envmod):
    """zero-length vertical: the reference divides by zero (python float) / raises; we flag the env"""
    from oracle.truss_oracle import TrussOracle
    o = TrussOracle("small_bridge")
    m = o.mesh
    y = np.array([0.0] * 8 + [4.0] * 8)[None].repeat(2, 0)
    y[1, 8 + 3] = 0.0                                   # top node 3 on top of bottom node 3
    sec = np.full((2, m.E), 4, dtype=np.int32)
    env = make_env(envmod, "small_bridge", 1)
    out = env.solve_only(torch.from_numpy(y).cuda(), torch.from_numpy(sec).cuda())
    torch.cuda.synchronize()
    assert int(out["status"][0]) == 0 and int(out["status"][1]) != 0
    with pytest.raises((ZeroDivisionError, FloatingPointError, Exception)):
        o.solve_only(y[1], sec[1])


@pytest.mark.parametrize("name,B", [("small_bridge", 4096), ("small_roof", 16384), ("large_bridge", 8192),
                                    ("train0_roof", 16384), ("train3_bridge", 16384)])
def test_full_size_properties(envmod, name, B):
    """BASELINE.json batch sizes: size-independent properties of the solved batch"""
    env = make_env(envmod, name, B)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    N, E = env.N, env.E
    for s in range(3):
        a_geo = torch.rand(B, N, 2, device="cuda", generator=g) * 0.5
        a_topo = torch.rand(B, N, 3, device="cuda", generator=g)
        coin = (torch.rand(B, device="cuda", generator=g) >= 0.5).to(torch.uint8)
        env.step(a_geo, a_topo, coin)
    torch.cuda.synchronize()
    assert int(env.status.abs().max()) == 0
    P = torch.from_numpy(env.handle.table("loadvec")).cuda()
    # (1) strain energy = half the work of the loads
    work = 0.5 * (env.d @ P)
    assert float(((env.U - work).abs() / work.abs()).max()) <= 1e-9
    # (2) reactions balance the applied load
    tnsc = env.handle.table("tnsc"); ndof = env.ndof
    res_ids = [(i, a) for i in range(N) for a in range(2) if tnsc[i, a] > ndof]
    ry = sum(env.reactions[:, tnsc[i, a] - 1 - ndof] for i, a in res_ids if a == 1)
    rx = sum(env.reactions[:, tnsc[i, a] - 1 - ndof] for i, a in res_ids if a == 0)
    assert float(((ry + P.sum()).abs() / P.sum().abs()).max()) <= 1e-9
    assert float((rx.abs() / P.sum().abs()).max()) <= 1e-9
    # (3) the symmetry pass leaves mirror-symmetric geometry and sections -> mirror-symmetric deflections (the training
    # shapes have mixed spans and no symmetry pass)
    nx = N // 2
    y = env.nN_x_n[:, :, 1]
    if env.spec.symmetry != SYM_NONE:
        assert torch.equal(y[:, nx:], y[:, nx:].flip(1)) and torch.equal(y[:, :nx], y[:, :nx].flip(1))
        dy = env.nN_x_n[:, :, 10].double()
        assert float(((dy[:, :nx] - dy[:, :nx].flip(1)).abs().max() / dy.abs().max())) <= 1e-6
    # (4) re-solving the emitted geometry reproduces d bit-exactly (idempotence of the FEM stage)
    sec = env.nN_x_e[:, :, 0].to(torch.int32).contiguous()
    again = env.solve_only(y.double().contiguous(), sec)
    assert torch.equal(again["d"], env.d) and torch.equal(again["axial"], env.axial)
    # (5) sharding invariance: the second half of the batch alone gives the same bits
    half = make_env(envmod, name, B // 2)
    half.reset()
    g2 = torch.Generator(device="cuda").manual_seed(0)
    for s in range(3):
        a_geo = torch.rand(B, N, 2, device="cuda", generator=g2) * 0.5
        a_topo = torch.rand(B, N, 3, device="cuda", generator=g2)
        coin = (torch.rand(B, device="cuda", generator=g2) >= 0.5).to(torch.uint8)
        half.step(a_geo[B // 2:].contiguous(), a_topo[B // 2:].contiguous(), coin[B // 2:].contiguous())
    torch.cuda.synchronize()
    for k in F32_FIELDS + ("point", "d", "axial", "ratio", "U"):
        assert torch.equal(getattr(half, k), getattr(env, k)[B // 2:]), k


def record_parity_counts(name, counts):
    """gpurun_out/r2_parity_counts.json (copied to profiles/ for the record): per family and step, how many environments
    of the full batch sit outside the flat 1e-9 and what the extended-precision solve says about them"""
    import json
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "r2_parity_counts.json")
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        data = json.load(open(path)) if os.path.exists(path) else {}
        data[name] = counts
        json.dump(data, open(path, "w"), indent=1)
    except OSError:
        pass


@pytest.mark.parametrize("name", FAMILY_NAMES)
def test_ill_conditioned_solves_vs_extended_precision(envmod, name):
    """The golden transitions (geometries the REFERENCE visited, cond(K) up to 1.9e8 on the saturated walks; tr_out_d is
    what its own float64 LU returned) solved by the kernel and, in extended precision, by oracle/exact_fem.py: wherever the
    kernel is more than 1e-9 from the reference it is because the REFERENCE is that far from the exact displacements --
    the kernel itself obeys the same eps * cond bound and is as close to the truth as the reference is."""
    from oracle import exact_fem
    from oracle.truss_oracle import FAMILIES, build_mesh
    g = load_golden(name)
    m = build_mesh(FAMILIES[name])
    y, sec, d_ref = g["tr_out_y"], g["tr_out_section"].astype(np.int32), g["tr_out_d"]
    env = make_env(envmod, name, len(y))
    out = env.solve_only(torch.from_numpy(np.ascontiguousarray(y)).cuda(), torch.from_numpy(np.ascontiguousarray(sec)).cuda())
    torch.cuda.synchronize()
    assert int(out["status"].abs().max()) == 0
    d_gpu = cpu(out["d"])
    d_exact = exact_fem.exact_displacements(m, y, sec)
    cond = exact_fem.cond2(m, y, sec)
    e_gpu, e_ref = exact_fem.rel_err(d_gpu, d_exact), exact_fem.rel_err(d_ref, d_exact)
    eps = np.finfo(np.float64).eps
    assert (e_gpu <= np.maximum(20 * eps * cond, 1e-13)).all(), float((e_gpu / (eps * cond)).max())
    assert e_gpu[cond <= 1e6].max() <= 1e-10                          # a decade inside the flat tolerance in normal play
    hard = cond > 1e6
    # case by case either solver can be the luckier one; as a population the kernel's error measured in units of eps * cond
    # is no larger than the reference's
    r_gpu, r_ref = e_gpu / (eps * cond), e_ref / (eps * cond)
    assert r_gpu.max() <= 2 * r_ref.max() and np.median(r_gpu[hard]) <= 2 * np.median(r_ref[hard]) + 1e-3
    gpu_vs_ref = np.abs(d_gpu - d_ref).max(axis=1) / np.abs(d_ref).max(axis=1)
    assert (gpu_vs_ref <= e_gpu + e_ref + 1e-15).all()                  # triangle inequality: the whole difference is explained
    assert (gpu_vs_ref[cond <= 1e6] <= FP64_TOL).all()
    record_parity_counts("golden_" + name, {
        "cases": int(len(y)), "cond>1e6": int(hard.sum()), "max cond": float(cond.max()),
        "kernel vs reference: outside flat 1e-9": int((gpu_vs_ref > FP64_TOL).sum()),
        "max kernel error vs exact": float(e_gpu.max()), "max reference error vs exact": float(e_ref.max()),
        "cond>1e6: kernel closer to exact than the reference": int((e_gpu[hard] <= e_ref[hard]).sum()),
        "max error / (eps cond): kernel": float((e_gpu / (eps * cond)).max()),
        "max error / (eps cond): reference": float((e_ref / (eps * cond)).max())})


def test_empty_batch_and_bad_args(envmod):
    env = make_env(envmod, "small_bridge", 4)
    env.reset()
    with pytest.raises(ValueError):
        env.step(torch.zeros(4, 16, 2), torch.zeros(4, 16, 3))          # CPU tensors
    with pytest.raises(ValueError):
        env.step(torch.zeros(3, 16, 2, device="cuda"), torch.zeros(4, 16, 3, device="cuda"))
    from mop_truss_marl_b200 import capi
    sin, sout = capi.StepIn(), capi.StepOut()
    assert capi.lib.tfem_step(env.handle.ptr, 0, C.byref(sin), C.byref(sout), None) == 0   # B = 0 is a no-op
    assert capi.lib.tfem_step(env.handle.ptr, 4, C.byref(sin), C.byref(sout), None) == -1  # missing inputs


@pytest.mark.parametrize("name,B", [("small_bridge", 4096), ("small_roof", 16384), ("large_bridge", 8192), ("large_roof", 4096)])
def test_full_batch_against_c_oracle(envmod, name, B):
    """EVERY environment of a BASELINE.json-sized batch against the C restatement of the oracle (oracle/truss_oracle.c,
    pinned by tests/test_c_oracle.py): three env steps from reset, each step's inputs taken from the GPU state"""
    from oracle.c_oracle import COracle
    from util import ulp_diff
    from oracle import exact_fem
    from oracle.truss_oracle import FAMILIES, build_mesh
    co = COracle(name)
    mesh = build_mesh(FAMILIES[name])
    env = make_env(envmod, name, B)
    env.reset()
    N, E, nx = env.N, env.E, env.N // 2
    g = torch.Generator(device="cuda").manual_seed(7)
    rng_np = np.random.RandomState(11)
    counts = {"family": name, "envs": B, "steps": []}
    for s in range(3):
        scale = (1.3, 0.6, 0.25)[s]                                   # out-of-range, ordinary and small actions
        a_geo = (torch.rand(B, N, 2, device="cuda", generator=g) * scale - 0.05).contiguous()
        a_topo = (torch.rand(B, N, 3, device="cuda", generator=g) * 1.2 - 0.1).contiguous()
        coin = (torch.rand(B, device="cuda", generator=g) >= 0.5).to(torch.uint8)
        set_node, set_elem, stale = cpu(env.nN_x_n).copy(), cpu(env.nN_x_e).copy(), cpu(env.move_range).copy()
        ag, at = cpu(a_geo).copy(), cpu(a_topo).copy()
        want = co.step(set_node, set_elem, ag, at, cpu(coin), stale)
        env.step(a_geo, a_topo, coin)
        torch.cuda.synchronize()
        tag = "%s step %d" % (name, s)
        assert int(env.status.abs().max()) == 0 and int(want["status"].max()) == 0, tag
        # bit-exact: clipped actions, heights (float64 bit patterns), weak flags, sections, move range
        assert np.array_equal(cpu(a_geo), ag) and np.array_equal(cpu(a_topo), at), tag + " clip"
        assert np.array_equal(cpu(env.y), want["y"]), tag + " y"
        assert np.array_equal(cpu(env.y_weak), want["weak"]), tag + " weak"
        assert np.array_equal(cpu(env.nN_x_e)[:, :, 0].astype(np.int32), want["section"]), tag + " section"
        assert np.array_equal(cpu(env.move_range), want["move_range"]), tag + " move range"
        # FP64: flat 1e-9 normwise against the oracle (north_star) is COUNTED per environment.  The environments outside it
        # are the ill-conditioned ones (d_min-deep trusses, cond(K) up to 1e8), where the oracle's LU -- the reference's --
        # is itself eps * cond away from the exact displacements: for every one of them the exact displacements are formed
        # in extended precision (oracle/exact_fem.py) and the kernel must be as close to them as the oracle is.
        errs = {}
        for k in ("d", "axial", "ratio"):
            got = cpu(getattr(env, k))
            errs[k] = np.abs(got - want[k]).max(axis=1) / np.abs(want[k]).max(axis=1)
            assert errs[k].max() <= 1e-6, "%s %s %.3e" % (tag, k, errs[k].max())
        errs["U"] = np.abs(cpu(env.U) - want["U"]) / np.abs(want["U"])
        assert errs["U"].max() <= 1e-6, tag + " U"
        worst = np.maximum.reduce([errs[k] for k in ("d", "axial", "ratio", "U")])
        outside = np.nonzero(worst > FP64_TOL)[0]
        sample = np.concatenate([outside, rng_np.choice(B, size=min(B, 256), replace=False)])
        d_exact = exact_fem.exact_displacements(mesh, want["y"][sample], want["section"][sample])
        e_gpu = exact_fem.rel_err(cpu(env.d)[sample], d_exact)
        e_orc = exact_fem.rel_err(want["d"][sample], d_exact)
        cond = exact_fem.cond2(mesh, want["y"][sample], want["section"][sample])
        bound = 20 * np.finfo(np.float64).eps * cond
        assert (e_gpu <= np.maximum(bound, 1e-13)).all(), "%s: kernel beyond 20 eps cond (%.2e)" % (tag, (e_gpu / bound).max())
        r_gpu, r_orc = e_gpu / (np.finfo(np.float64).eps * cond), e_orc / (np.finfo(np.float64).eps * cond)
        assert r_gpu.max() <= 2 * r_orc.max(), "%s: kernel further from the exact solve than the oracle (%.2f vs %.2f eps cond)" % (
            tag, r_gpu.max(), r_orc.max())
        no = len(outside)
        assert no <= B // 50, "%s: %d of %d environments outside the flat 1e-9" % (tag, no, B)      # measured: none
        if no:
            assert cond[:no].min() > 1e5, "%s: an environment outside 1e-9 is not ill-conditioned (cond %.1e)" % (tag, cond[:no].min())
        # flags: compression flag; a mismatch is only legitimate where the member force is a rounding-level zero
        ax = want["axial"]
        flags_gpu = cpu(env.nN_x_e)[:, :, 4].astype(np.int32)
        mism = flags_gpu != want["iscompress"]
        clear = np.abs(ax) > 1e-7 * np.abs(ax).max(axis=1, keepdims=True)
        assert not (mism & clear).any(), tag + " iscompress"
        counts["steps"].append({
            "step": s, "envs": B, "outside_flat_1e-9": int(no), "fraction_inside_flat_1e-9": float(1.0 - no / B),
            "max_err_vs_oracle": {k: float(errs[k].max()) for k in errs},
            "outside: min cond(K)": float(cond[:no].min()) if no else None,
            "outside: max kernel error vs exact": float(e_gpu[:no].max()) if no else None,
            "outside: max oracle error vs exact": float(e_orc[:no].max()) if no else None,
            "outside: kernel closer to exact than the oracle": int((e_gpu[:no] <= e_orc[:no]).sum()) if no else None,
            "sample(256): max kernel error vs exact": float(e_gpu[no:].max()), "sample(256): max oracle error vs exact": float(e_orc[no:].max()),
            "iscompress flags": int(mism.size), "iscompress mismatches (all at rounding-level zero forces)": int(mism.sum())})
        # objective point: <= 2 ulp(float32)
        assert ulp_diff(cpu(env.point), want["point"]).max() <= 2, tag + " point"
    record_parity_counts(name, counts)
