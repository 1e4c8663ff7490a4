"""CPU: the C restatement of the oracle (oracle/truss_oracle.c, whole batches, OpenMP) against the golden transitions
recorded from the reference itself and against the pinned Python oracle."""
import numpy as np
import pytest

from oracle.c_oracle import COracle
from oracle.truss_oracle import TrussOracle
from util import FAMILY_NAMES, FP64_TOL, load_golden, nrm


@pytest.fixture(scope="module", params=FAMILY_NAMES)
def fam(request):
    return request.param, load_golden(request.param), COracle(request.param, threads=4)


def test_golden_transitions(fam):
    name, g, co = fam
    T = g["tr_mode"].shape[0]
    a_geo, a_topo = g["tr_in_a_geo"].copy(), g["tr_in_a_topo"].copy()
    stale = np.ascontiguousarray(np.stack([g["tr_in_max_up"], g["tr_in_max_down"]], axis=-1).astype(np.float32))
    out = co.step(np.ascontiguousarray(g["tr_in_set_node"]), np.ascontiguousarray(g["tr_in_set_element"]), a_geo, a_topo,
                  g["tr_in_coin"].astype(np.uint8), stale)
    # float32 / weak-scalar transition, move range, flags, objective point: bit-exact
    assert np.array_equal(a_geo, g["tr_out_a_geo"]) and np.array_equal(a_topo, g["tr_out_a_topo"])      # clipped in place
    assert np.array_equal(out["y"], g["tr_out_y"]) and np.array_equal(out["weak"].astype(bool), g["tr_out_y_weak"])
    assert np.array_equal(out["section"], g["tr_out_section"])
    assert np.array_equal(out["move_range"][:, :, 0], g["tr_out_max_up"])
    assert np.array_equal(out["move_range"][:, :, 1], g["tr_out_max_down"])
    assert np.array_equal(out["iscompress"], g["tr_out_iscompress"])
    assert np.array_equal(out["point"], g["tr_out_point"])
    assert int(out["status"].max()) == 0
    # FP64 fields: 1e-9 for cond(K) <= 1e6, growing linearly beyond (the rule of tests/test_gpu_parity.py::fp64_tol)
    py = TrussOracle(name)
    for i in range(T):
        cond = float(np.linalg.cond(py.solve_only(g["tr_out_y"][i], g["tr_out_section"][i])["K"]))
        tol = FP64_TOL * max(1.0, cond / 1e6)
        for k in ("d", "axial", "ratio"):
            assert nrm(out[k][i], g["tr_out_" + k][i]) <= tol, (i, k, cond)
        assert abs(out["U"][i] - float(g["tr_out_U"][i])) <= tol * abs(float(g["tr_out_U"][i]))


def test_reset_geometry_and_solve_entry(fam):
    name, g, co = fam
    out = co.solve(g["reset_y"][None], g["reset_section"][None])
    assert nrm(out["d"][0], g["reset_d"]) <= 1e-12 and nrm(out["axial"][0], g["reset_axial"]) <= 1e-12
    assert abs(out["U"][0] - float(g["reset_U"])) <= 1e-12 * float(g["reset_U"])
    assert np.array_equal(out["point"][0, :2], np.ones(2, dtype=np.float32))     # obj / int_obj at the generated geometry


def test_random_walk_vs_python_oracle_and_thread_invariance(fam):
    name, g, co = fam
    random_walk_vs_python_oracle(name, co)


def random_walk_vs_python_oracle(name, co):
    """three steps of 24 environments from reset: bit-exact against the Python oracle, and for one thread or many"""
    py = co.py
    N, E = py.mesh.N, py.mesh.E
    rng = np.random.RandomState(3)
    B = 24
    st = py.reset()
    set_node = np.repeat(st["nN_x_n"][None], B, axis=0).astype(np.float32)
    set_elem = np.repeat(st["nN_x_e"][None], B, axis=0).astype(np.float32)
    stale = np.repeat(np.stack([st["max_up"], st["max_down"]], axis=-1)[None], B, axis=0).astype(np.float32)
    single = COracle(name, threads=1)
    for step in range(3):
        a_geo = (rng.rand(B, N, 2) * 1.2 - 0.1).astype(np.float32)
        a_topo = (rng.rand(B, N, 3) * 1.2 - 0.1).astype(np.float32)
        coin = (rng.rand(B) >= 0.5).astype(np.uint8)
        ag1, at1 = a_geo.copy(), a_topo.copy()
        out = co.step(set_node, set_elem, ag1, at1, coin, stale)
        ag2, at2 = a_geo.copy(), a_topo.copy()
        out1 = single.step(set_node, set_elem, ag2, at2, coin, stale)
        for k in out:
            assert np.array_equal(out[k], out1[k]), k                      # the thread count does not change a bit
        nxt_node, nxt_elem = set_node.copy(), set_elem.copy()
        for b in range(B):
            ag, at = a_geo[b].copy(), a_topo[b].copy()
            want = py.step(set_node[b], set_elem[b], stale[b, :, 0], stale[b, :, 1], ag, at, bool(coin[b]))
            assert np.array_equal(ag, ag1[b]) and np.array_equal(at, at1[b])
            assert np.array_equal(out["y"][b], want["y"]) and np.array_equal(out["weak"][b].astype(bool), want["y_weak"])
            assert np.array_equal(out["section"][b], want["section"])
            assert np.array_equal(out["move_range"][b, :, 0], want["max_up"])
            assert np.array_equal(out["move_range"][b, :, 1], want["max_down"])
            assert np.array_equal(out["point"][b], want["point"])
            assert nrm(out["d"][b], want["d"]) <= 1e-9
            nxt_node[b], nxt_elem[b] = want["nN_x_n"], want["nN_x_e"]
        set_node, set_elem, stale = nxt_node, nxt_elem, out["move_range"].copy()
