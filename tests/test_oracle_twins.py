"""CPU: the cases of the comparisons with the original project's modules (tests/test_oracle_vs_reference.py and the
reference legs of tests/test_pareto_oracle.py) that the vectors recorded from the reference do not hold, replayed through
the oracle against the outputs recorded by tests/golden/make_oracle_twins.py, with the tolerances of those comparisons;
and the textbook example of test_kat_example_3_8 through the oracle's own solver."""
import os
import types

import numpy as np
import pytest

from oracle import pareto_oracle, truss_oracle
from oracle.truss_oracle import TrussOracle, pareto_state_data
from test_oracle_golden import check
from util import FP64_TOL, GOLDEN_DIR, assert_f32_close, nrm

TRAIN_RUNS = ("train0_roof", "train3_bridge")
ALL_RUNS = ("small_bridge", "small_roof", "large_bridge", "large_roof") + TRAIN_RUNS


def twins(name):
    return np.load(os.path.join(GOLDEN_DIR, name + ".npz"))


def replay(o, g, prefix, i):
    a_geo, a_topo = g[prefix + "in_a_geo"][i].copy(), g[prefix + "in_a_topo"][i].copy()
    out = o.step(g[prefix + "in_set_node"][i], g[prefix + "in_set_element"][i], g[prefix + "in_max_up"][i],
                 g[prefix + "in_max_down"][i], a_geo, a_topo, bool(g[prefix + "in_coin"][i]))
    assert np.array_equal(a_geo, g[prefix + "out_a_geo"][i], equal_nan=True)          # clipped in place
    assert np.array_equal(a_topo, g[prefix + "out_a_topo"][i])
    return out


@pytest.mark.parametrize("run", TRAIN_RUNS)
def test_train_shape_tables(run):
    g, o = twins("twins_train"), TrussOracle(run)
    m, p = o.mesh, run + "/"
    for k, v in (("conn", m.conn), ("tnsc", m.tnsc), ("res", m.res), ("top", m.top), ("pair", m.pair), ("x", m.x),
                 ("loaded", m.loaded), ("has_loady", m.has_loady), ("P", m.P), ("ndof", m.ndof),
                 ("limits", [m.y_max, m.y_min, m.d_min, m.max_deformation]), ("sym_src", [m.sym_src_false, m.sym_src_true]),
                 ("sym_elem_pairs", np.array(m.sym_elem_pairs).reshape(-1, 2)), ("A_n", o.A_n), ("mask", o.mask),
                 ("nC_e", o.nC_e), ("int_obj", [o.int_obj1, o.int_obj2])):
        assert np.array_equal(np.array(v), g[p + k]), k
    assert np.array_equal(np.array([np.nan if t is None else t for t in m.target_top]), g[p + "target"], equal_nan=True)


@pytest.mark.parametrize("run", TRAIN_RUNS)
@pytest.mark.parametrize("mode", ["uniform", "small_actions", "saturated"])
def test_train_shape_reset_and_walk(run, mode):
    g, o = twins("twins_train"), TrussOracle(run)
    check(o.reset(), g, run + "/reset_")
    p = "%s/%s/" % (run, mode)
    assert len(g[p + "in_coin"]) > 0
    for i in range(len(g[p + "in_coin"])):
        out = replay(o, g, p, i)
        check(out, g, p + "out_", i)
        assert_f32_close("point", out["point"], g[p + "out_point"][i])


@pytest.mark.parametrize("run", ALL_RUNS)
def test_adversarial_walk_recorded(run):
    g, o, p = twins("twins_adversarial"), TrussOracle(run), run + "/"
    assert len(g[p + "in_coin"]) > 0
    for i in range(len(g[p + "in_coin"])):
        out = replay(o, g, p, i)
        for k in ("y", "section", "max_up", "max_down"):
            assert np.array_equal(out[k], g[p + "out_" + k][i]), k
        if g[p + "well"][i]:                          # cond(K) < 1e6: the FEM and observation fields too
            assert nrm(out["d"], g[p + "out_d"][i]) <= FP64_TOL
            for k in ("x_n", "nN_x_n", "nN_x_e"):
                assert_f32_close(k, out[k], g[p + "out_" + k][i])


def test_pareto_state_data_recorded():
    g = twins("twins_pareto")
    keys = sorted(k[:-1] for k in g.files if k.startswith("psd") and k.endswith("_x"))
    assert len(keys) == 8
    for key in keys:
        max_front, n = (int(v) for v in key[3:-1].split("_n"))
        x, A = pareto_state_data(g[key + "pf"], n // 2, max_front=max_front)
        assert np.array_equal(x, g[key + "x"]) and np.array_equal(A, g[key + "A"], equal_nan=True), key


def test_thinning_of_large_fronts_recorded():
    """fronts of more than MAX_FRONT = 50 members thinned with an explicit draw (utils.simple_cull's random.sample)"""
    g = twins("twins_pareto")
    keys = sorted(k[:-3] for k in g.files if k.startswith("thin") and k.endswith("pts"))
    assert len(keys) == 5
    for key in keys:
        front, *stats = pareto_oracle.front_stats(g[key + "pts"], thin_pick=[int(v) for v in g[key + "pick"]])
        assert len(front) == 50 and np.array_equal(np.array(front), g[key + "front"]), key
        assert np.allclose(stats, g[key + "stats"], rtol=1e-12, atol=1e-14), key
        hv = [pareto_oracle.hypervolume(front, (0.9, 0.95)), pareto_oracle.hypervolume(front)]
        assert np.abs(np.array(hv) - g[key + "hv"]).max() <= 1e-12, key


def test_kat_example_3_8_oracle_solver(monkeypatch):
    """the textbook example kept as a comment in the reference's FEM_2Dtruss.py:474-558 (three bars meeting at one loaded
    node, inches and kips), solved by the oracle's direct-stiffness solve"""
    monkeypatch.setattr(truss_oracle, "SECTION_TABLE", np.array([[8e4], [6e4], [8e4]]))   # areas 8, 6, 8 after the 1e-4
    monkeypatch.setattr(truss_oracle, "YOUNG", 29000.0)
    m = types.SimpleNamespace(N=4, E=3, ndof=2, x=[0, 12 * 12, 24 * 12, 12 * 12], conn=[[0, 3], [1, 3], [2, 3]],
                              tnsc=[[3, 4], [5, 6], [7, 8], [1, 2]], P=[150, -300])
    fem = truss_oracle.fem_solve(m, [0.0, 0.0, 0.0, 16.0 * 12], [0, 1, 2])
    assert np.allclose(fem["K"], [[696, 0], [0, 2143.5833333333335]], rtol=1e-12)
    assert np.allclose(fem["d"], [0.21551724137931033, -0.13995257162850366], rtol=1e-12)
    assert np.allclose(fem["axial"], [-16.770011273957138, 126.83201803833144, 233.22998872604282], rtol=1e-12)
