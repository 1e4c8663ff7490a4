"""CPU: the oracles on the ten 6 x 2 training families (families.TRAIN_FAMILIES), the batch the training driver steps.

* The C restatement of the oracle against the transitions recorded from the reference for train0_roof and train3_bridge
  (tests/golden/twins_train.npz, twins_adversarial.npz), and against the Python oracle on random walks of every family.
* The reference pins the oracle for train0_roof and train3_bridge only.  Every other training family has the tables of
  the pinned family of its truss type except the targets (and int_obj2, which is formed from them), so one oracle step
  from a shared state differs between shapes only in the target column of x_n / nN_x_n and in point / point64.  A kernel
  that read the wrong shape's tables would therefore show only in those fields: the GPU tests check them directly."""
import numpy as np
import pytest

from oracle.c_oracle import COracle
from oracle.truss_oracle import TrussOracle
from test_c_oracle import random_walk_vs_python_oracle
from test_oracle_twins import TRAIN_RUNS, twins
from util import F32_FIELDS, FP64_TOL, nrm

from mop_truss_marl_b200.families import TRAIN_FAMILIES

WALKS = ("uniform", "small_actions", "saturated")
PINNED = {"roof": "train0_roof", "bridge": "train3_bridge"}          # the families the reference recorded
TARGET_COL = 9                                                       # target * top / (y + 1e-6) in x_n and nN_x_n


def stale_range(g, p):
    return np.ascontiguousarray(np.stack([g[p + "in_max_up"], g[p + "in_max_down"]], axis=-1).astype(np.float32))


@pytest.mark.parametrize("run", TRAIN_RUNS)
@pytest.mark.parametrize("walk", WALKS)
def test_c_oracle_vs_recorded_train_walks(run, walk):
    g, p = twins("twins_train"), "%s/%s/" % (run, walk)
    co, py = COracle(run, threads=4), TrussOracle(run)
    a_geo, a_topo = g[p + "in_a_geo"].copy(), g[p + "in_a_topo"].copy()
    out = co.step(np.ascontiguousarray(g[p + "in_set_node"]), np.ascontiguousarray(g[p + "in_set_element"]), a_geo, a_topo,
                  g[p + "in_coin"].astype(np.uint8), stale_range(g, p))
    # transition, clipped actions, move range, flags and the objective point: bit-exact
    assert np.array_equal(a_geo, g[p + "out_a_geo"]) and np.array_equal(a_topo, g[p + "out_a_topo"])
    assert np.array_equal(out["y"], g[p + "out_y"]) and np.array_equal(out["weak"].astype(bool), g[p + "out_y_weak"])
    assert np.array_equal(out["section"], g[p + "out_section"])
    assert np.array_equal(out["move_range"][:, :, 0], g[p + "out_max_up"])
    assert np.array_equal(out["move_range"][:, :, 1], g[p + "out_max_down"])
    assert np.array_equal(out["iscompress"], g[p + "out_iscompress"])
    assert np.array_equal(out["point"], g[p + "out_point"])
    assert int(out["status"].max()) == 0
    # FP64 fields: 1e-9 up to cond(K) = 1e6, growing linearly beyond (test_gpu_parity.fp64_tol)
    for i in range(len(out["y"])):
        cond = float(np.linalg.cond(py.solve_only(g[p + "out_y"][i], g[p + "out_section"][i])["K"]))
        tol = FP64_TOL * max(1.0, cond / 1e6)
        for k in ("d", "axial", "ratio"):
            assert nrm(out[k][i], g[p + "out_" + k][i]) <= tol, (i, k, cond)
        assert abs(out["U"][i] - float(g[p + "out_U"][i])) <= tol * abs(float(g[p + "out_U"][i]))


@pytest.mark.parametrize("run", TRAIN_RUNS)
def test_c_oracle_vs_recorded_adversarial(run):
    """ties, exact 0 / 1, out-of-range and non-finite actions, absurd stale move ranges (twins_adversarial.npz)"""
    g, p = twins("twins_adversarial"), run + "/"
    a_geo, a_topo = g[p + "in_a_geo"].copy(), g[p + "in_a_topo"].copy()
    out = COracle(run, threads=4).step(np.ascontiguousarray(g[p + "in_set_node"]), np.ascontiguousarray(g[p + "in_set_element"]),
                                       a_geo, a_topo, g[p + "in_coin"].astype(np.uint8), stale_range(g, p))
    assert np.array_equal(a_geo, g[p + "out_a_geo"], equal_nan=True) and np.array_equal(a_topo, g[p + "out_a_topo"])
    assert np.array_equal(out["y"], g[p + "out_y"]) and np.array_equal(out["section"], g[p + "out_section"])
    assert np.array_equal(out["move_range"][:, :, 0], g[p + "out_max_up"])
    assert np.array_equal(out["move_range"][:, :, 1], g[p + "out_max_down"])
    for i in np.nonzero(g[p + "well"])[0]:                             # cond(K) < 1e6: the FEM too
        assert int(out["status"][i]) == 0
        assert nrm(out["d"][i], g[p + "out_d"][i]) <= FP64_TOL


@pytest.mark.parametrize("name", TRAIN_FAMILIES)
def test_c_oracle_random_walk_vs_python_oracle(name):
    random_walk_vs_python_oracle(name, COracle(name, threads=4))


MESH_TABLES = ("conn", "tnsc", "res", "top", "pair", "x", "loaded", "has_loady", "P", "ndof")


def tables(o):
    m = o.mesh
    t = {k: np.array(getattr(m, k)) for k in MESH_TABLES}
    t.update(limits=np.array([m.y_max, m.y_min, m.d_min, m.max_deformation]),
             sym_src=np.array([m.sym_src_false, m.sym_src_true]), sym_elem_pairs=np.array(m.sym_elem_pairs).reshape(-1, 2),
             A_n=o.A_n, mask=o.mask, nC_e=o.nC_e, int_obj1=np.array(o.int_obj1))
    return t


@pytest.mark.parametrize("name", TRAIN_FAMILIES)
def test_train_family_tables_are_the_pinned_ones(name):
    """every table of a training family but its targets equals what the reference recorded for the pinned family of the
    same truss type; int_obj1 (the volume of the generated geometry) too, int_obj2 is formed from the targets"""
    o = TrussOracle(name)
    pinned = PINNED[o.spec.truss_type]
    g, p = twins("twins_train"), pinned + "/"
    for k, v in tables(o).items():
        want = g[p + "int_obj"][0] if k == "int_obj1" else g[p + k]
        assert np.array_equal(v, want), (name, k)
    targets = np.array([np.nan if t is None else t for t in o.mesh.target_top])
    assert np.array_equal(np.isnan(targets), np.isnan(g[p + "target"]))
    assert np.array_equal(targets[6:], np.array(o.spec.tar_y, dtype=np.float64))


def test_shapes_differ_only_in_the_target_fields():
    """From one state and one action, the five shapes of a truss type give bit-identical heights, sections, move ranges,
    FEM fields, A_s / A_n_ts / A_n_cs and nN_x_e; x_n and nN_x_n differ in the target column only, and point / point64
    in the target distance (obj2).  train1 and train2 share int_obj2 (as do train3 and train4), so a swap of those two
    is visible in the target column alone."""
    rng = np.random.RandomState(5)
    N = 12
    int_obj2 = {}
    for tt in ("roof", "bridge"):
        names = [n for n in TRAIN_FAMILIES if n.endswith(tt)]
        oracles = [TrussOracle(n) for n in names]
        for o in oracles:
            int_obj2[o.spec.name] = o.int_obj2
        st = oracles[0].reset()
        node, elem = st["nN_x_n"], st["nN_x_e"]
        up, down = st["max_up"], st["max_down"]
        for step in range(6):
            a_geo = rng.rand(N, 2).astype(np.float32)
            a_topo = rng.rand(N, 3).astype(np.float32)
            coin = bool(rng.rand() < 0.5)
            outs = [o.step(node, elem, up, down, a_geo.copy(), a_topo.copy(), coin) for o in oracles]
            ref = outs[0]
            for o, out in zip(oracles[1:], outs[1:]):
                tag = "%s vs %s step %d" % (o.spec.name, names[0], step)
                for k in ("y", "y_weak", "section", "max_up", "max_down", "d", "axial", "ratio", "U", "reactions", "iscompress",
                          "length") + tuple(f for f in F32_FIELDS if f not in ("x_n", "nN_x_n")):
                    assert np.array_equal(out[k], ref[k]), (tag, k)
                for k in ("x_n", "nN_x_n"):
                    other = [c for c in range(out[k].shape[1]) if c != TARGET_COL]
                    assert np.array_equal(out[k][:, other], ref[k][:, other]), (tag, k)
                    assert not np.array_equal(out[k][:, TARGET_COL], ref[k][:, TARGET_COL]), (tag, k)
                assert np.array_equal(out["point"][[0, 2, 3]], ref["point"][[0, 2, 3]]), tag
                assert np.array_equal(out["point64"][[0, 2, 3]], ref["point64"][[0, 2, 3]]), tag
            node, elem, up, down = ref["nN_x_n"], ref["nN_x_e"], ref["max_up"], ref["max_down"]
    assert int_obj2["train1_roof"] == int_obj2["train2_roof"] and int_obj2["train3_bridge"] == int_obj2["train4_bridge"]
    assert len(set(int_obj2[n] for n in TRAIN_FAMILIES if n.endswith("roof"))) == 3
