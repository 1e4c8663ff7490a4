"""Writes tests/golden/twins_{train,adversarial,pareto}.npz: the cases of tests/test_oracle_vs_reference.py and of the
reference legs of tests/test_pareto_oracle.py that the vectors recorded from the reference (make_golden.py,
make_golden_pareto.py) do not hold, with the seeds and loops of those tests:

  * twins_train.npz ....... the two train/code shapes (train0_roof, train3_bridge): static tables, reset state, and the
                            uniform / small_actions / saturated walks of test_random_walk
  * twins_adversarial.npz . test_adversarial_walk on all six runs (ties, exact bounds, inf / NaN geometry actions,
                            absurd stale move ranges)
  * twins_pareto.npz ...... test_pareto_state_data (MAX_FRONT 50 of test/*/code and 20 of train/code) and the thinning of
                            fronts above MAX_FRONT of test_thinning_of_large_fronts_matches_reference

Those tests import the unmodified reference modules, which are not part of the repository.  The outputs here are
recorded from the CPU oracle (oracle/truss_oracle.py, oracle/pareto_oracle.py), which has not changed since commit
0f4d1e1, whose tests pinned it against the reference on exactly these cases (bit-exact geometry and flags, FEM fields
within 1e-9, float32 tensors within 2 ulp).  tests/test_oracle_twins.py replays every recorded case through the oracle
with the tolerances of the original comparison, so a later change to the oracle that would have broken the pin fails.

    python tests/golden/make_oracle_twins.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import pareto_oracle                                    # noqa: E402
from oracle.truss_oracle import SingularStiffness, TrussOracle, pareto_state_data   # noqa: E402
from util import adversarial_actions, adversarial_move_range       # noqa: E402

TRAIN_RUNS = ("train0_roof", "train3_bridge")
ALL_RUNS = ("small_bridge", "small_roof", "large_bridge", "large_roof") + TRAIN_RUNS
WALK_OUT = ("y", "section", "y_weak", "max_up", "max_down", "iscompress", "d", "axial", "ratio", "length", "reactions", "U",
            "x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "point")
ADV_OUT = ("y", "section", "max_up", "max_down", "d", "x_n", "nN_x_n", "nN_x_e")
# every step of every walk is taken; only a fixed share is stored, so that the files stay small
WALK_KEEP, ADV_KEEP, THIN_KEEP = 24, 6, 5


def record(rec, prefix, set_node, set_elem, up, down, a_geo, a_topo, coin, out, clipped, keys):
    for k, v in (("set_node", set_node), ("set_element", set_elem), ("max_up", up), ("max_down", down), ("a_geo", a_geo),
                 ("a_topo", a_topo), ("coin", coin)):
        rec.setdefault(prefix + "in_" + k, []).append(np.array(v))
    rec.setdefault(prefix + "out_a_geo", []).append(clipped[0])
    rec.setdefault(prefix + "out_a_topo", []).append(clipped[1])
    for k in keys:
        rec.setdefault(prefix + "out_" + k, []).append(np.array(out[k]))


def walk(o, mode, rec, prefix):
    """test_random_walk driven by the oracle: three children from one parent, the stale move range of the last child;
    every WALK_KEEP-th step is stored"""
    taken = 0
    rng = np.random.RandomState({"uniform": 1, "small_actions": 2, "saturated": 3}[mode])
    parent = o.reset()
    up, down = parent["max_up"], parent["max_down"]
    N = o.mesh.N
    for k in range(40 if N == 16 else 20):
        children = []
        for child in range(3):
            if mode == "uniform":
                a_geo = rng.rand(N, 2); a_topo = rng.rand(N, 3)
            elif mode == "small_actions":
                a_geo = rng.rand(N, 2) * 0.2; a_topo = rng.rand(N, 3) * np.array([0.3, 0.3, 1.0])
            else:
                a_geo = rng.randn(N, 2) * 2 + 0.5; a_topo = rng.randn(N, 3) * 2 + 0.5
            a_geo = a_geo.astype(np.float32); a_topo = a_topo.astype(np.float32)
            if mode == "saturated" and k % 5 == 0:
                up = (rng.rand(N) * 40).astype(np.float32); down = (rng.rand(N) * 40).astype(np.float32)
            coin = bool(rng.rand() >= 0.5)
            g2, t2 = a_geo.copy(), a_topo.copy()
            try:
                out = o.step(parent["nN_x_n"], parent["nN_x_e"], up, down, g2, t2, coin)
            except SingularStiffness:
                continue
            if taken % WALK_KEEP == 0:
                record(rec, prefix, parent["nN_x_n"], parent["nN_x_e"], up, down, a_geo, a_topo, coin, out, (g2, t2), WALK_OUT)
            taken += 1
            up, down = out["max_up"], out["max_down"]
            children.append(out)
        if children:
            parent = children[rng.randint(len(children))]


def adversarial(o, rec, prefix):
    """test_adversarial_walk driven by the oracle; `well` marks the steps whose stiffness is conditioned below 1e6 (the
    steps on which the original comparison checked the FEM and observation fields); every ADV_KEEP-th step is stored"""
    taken = 0
    rng = np.random.RandomState(11)
    parent = o.reset()
    N = o.mesh.N
    for k in range(30 if N == 16 else 15):
        a_geo, a_topo = adversarial_actions(rng, N)
        up, down = adversarial_move_range(rng, N)
        coin = bool(rng.rand() >= 0.5)
        g2, t2 = a_geo.copy(), a_topo.copy()
        try:
            out = o.step(parent["nN_x_n"], parent["nN_x_e"], up, down, g2, t2, coin)
        except (SingularStiffness, ZeroDivisionError):
            continue
        if taken % ADV_KEEP == 0:
            record(rec, prefix, parent["nN_x_n"], parent["nN_x_e"], up, down, a_geo, a_topo, coin, out, (g2, t2), ADV_OUT)
            rec.setdefault(prefix + "well", []).append(np.linalg.cond(o.solve_only(out["y"], out["section"])["K"]) < 1e6)
        taken += 1
        parent = out


def tables(o, rec, prefix):
    m = o.mesh
    rec.update({prefix + k: np.array(v) for k, v in (
        ("conn", m.conn), ("tnsc", m.tnsc), ("res", m.res), ("top", m.top), ("pair", m.pair), ("x", m.x),
        ("loaded", m.loaded), ("has_loady", m.has_loady), ("target", [np.nan if t is None else t for t in m.target_top]),
        ("P", m.P), ("ndof", m.ndof), ("limits", [m.y_max, m.y_min, m.d_min, m.max_deformation]),
        ("sym_src", [m.sym_src_false, m.sym_src_true]), ("sym_elem_pairs", np.array(m.sym_elem_pairs).reshape(-1, 2)),
        ("A_n", o.A_n), ("mask", o.mask), ("nC_e", o.nC_e), ("int_obj", [o.int_obj1, o.int_obj2]))})
    reset = o.reset()
    rec.update({prefix + "reset_" + k: np.array(reset[k]) for k in WALK_OUT})


def pareto(rec):
    rng = np.random.RandomState(5)
    for max_front in (50, 20):
        for n in (1, 2, 7, 50):
            pf = np.array([[rng.rand(), rng.rand()] for _ in range(n)])
            x, A = pareto_state_data(pf, n // 2, max_front=max_front)
            key = "psd%d_n%d_" % (max_front, n)
            rec.update({key + "pf": pf, key + "x": x, key + "A": A})
    # the thinning loop of test_thinning_of_large_fronts_matches_reference (fronts above MAX_FRONT = 50 only): the first
    # THIN_KEEP of its cases
    rng = np.random.RandomState(5)
    t_id = 0
    for trial in range(40):
        n = rng.randint(120, 201)
        t = np.sort(rng.rand(n))
        pts = np.stack([t, 1.0 - t ** (0.5 + rng.rand()) + 0.002 * rng.rand(n), rng.rand(n) * 0.9, rng.rand(n) * 0.9], axis=1)
        pts = pts[rng.permutation(n)]
        F = len(pareto_oracle.front_indices(pts))
        if F <= 50 or t_id >= THIN_KEEP:
            continue
        pick = [int(k) for k in rng.permutation(F - 2)[:48]]
        front, *stats = pareto_oracle.front_stats(pts, thin_pick=pick)
        key = "thin%02d_" % t_id
        rec.update({key + "pts": pts, key + "pick": np.array(pick, dtype=np.int32), key + "front": np.array(front),
                    key + "stats": np.array(stats, dtype=np.float64),
                    key + "hv": np.array([pareto_oracle.hypervolume(front, (0.9, 0.95)), pareto_oracle.hypervolume(front)])})
        t_id += 1


def main():
    train, adv, par = {}, {}, {}
    for run in TRAIN_RUNS:
        o = TrussOracle(run)
        tables(o, train, run + "/")
        for mode in ("uniform", "small_actions", "saturated"):
            walk(o, mode, train, "%s/%s/" % (run, mode))
    for run in ALL_RUNS:
        adversarial(TrussOracle(run), adv, run + "/")
    pareto(par)
    for name, rec in (("twins_train", train), ("twins_adversarial", adv), ("twins_pareto", par)):
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **{k: np.stack(v) if isinstance(v, list) else v for k, v in rec.items()})
        print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
