"""CPU: oracle/pareto_oracle.py (restatement of utils.simple_cull / union_rectangles_fastest) against the golden
vectors recorded from the reference and, when the reference tree is present, against the imported reference itself."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import pareto_oracle, ref_harness          # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "pareto.npz")


def test_oracle_matches_golden():
    g = np.load(GOLD)
    for k in range(len(g["counts"])):
        pts = g["points"][k, :g["counts"][k]]
        front, max_d, dis_d, p_cd, sum_d, std_cd = pareto_oracle.front_stats(pts)
        F = int(g["front_len"][k])
        assert len(front) == F
        assert np.array_equal(front[:, :2], g["fronts"][k, :F])
        assert np.allclose([max_d, dis_d, p_cd, sum_d, std_cd], g["stats"][k], rtol=1e-12, atol=1e-14)
        for r, ref in enumerate(g["refs"]):
            assert abs(pareto_oracle.hypervolume(front, ref) - g["hv"][k, r]) <= 1e-12


def test_edge_cases():
    # single point (1,1): the reference short-circuits to 0 (utils.py:476)
    assert pareto_oracle.hypervolume([[1.0, 1.0, 0, 0]]) == 0.0
    assert pareto_oracle.hypervolume([]) == 0.0
    # one feasible point: no distances (dis 1, max 0, sum 0), std_cd 1
    f, max_d, dis_d, p_cd, sum_d, std_cd = pareto_oracle.front_stats([[0.4, 0.6, 0.5, 0.5], [0.1, 0.1, 2.0, 0.0]])
    assert len(f) == 1 and (max_d, dis_d, p_cd, sum_d, std_cd) == (0.0, 1.0, 0.0, 0.0, 1.0)
    assert abs(pareto_oracle.hypervolume(f) - 0.6 * 0.4) < 1e-15
    with pytest.raises(IndexError):                       # all infeasible: the reference indexes an empty list
        pareto_oracle.front_stats([[0.1, 0.1, 2.0, 0.0]])
    # points beyond 1 are clamped for the area, not for the reference-point strip
    assert abs(pareto_oracle.hypervolume([[1.5, 0.5, 0, 0]], (1, 1))) < 1e-15


def test_nan_key_places_nan_last_and_keeps_finite_orders():
    """front_indices / thin_order sort with NumPy's NaN convention (a NaN after every number, NaNs tied, then the index),
    the rule the kernel ranks by; finite orders are unchanged (also covered by the golden vectors)"""
    key = pareto_oracle.nan_last
    assert sorted([3.0, float("nan"), -np.inf, 1.0], key=key)[:3] == [-np.inf, 1.0, 3.0]
    assert key(float("nan")) == key(-float("nan")) and key(0.0) == key(-0.0)
    rng = np.random.RandomState(11)
    for trial in range(200):                                # finite: the plain (obj1, -obj2, index) sort
        n = rng.randint(1, 40)
        pts = np.round(rng.rand(n, 4) * 2, rng.randint(1, 4))
        pts[rng.randint(n), 2:] = 0.5
        pts[rng.rand(n) < 0.2, 0], pts[rng.rand(n) < 0.2, 0] = -0.0, 0.0     # -0.0 ties with 0.0
        feas = [i for i in range(n) if not (pts[i, 2] > 1 or pts[i, 3] > 1)]
        got = pareto_oracle.front_indices(pts)
        assert got == sorted(got, key=lambda i: (pts[i, 0], -pts[i, 1], i)) and set(got) <= set(feas)
    nan = float("nan")
    # obj1 NaN: never dominated, dominates nothing, last; obj2 NaN: after the numbers of its obj1 tie group
    pts = [[0.2, 0.8, 0, 0], [nan, 0.5, 0, 0], [0.6, 0.3, 0, 0], [0.9, 0.1, 0, 0], [0.6, nan, 0, 0], [0.6, 0.9, 0, 0]]
    assert pareto_oracle.front_indices(pts) == [0, 2, 4, 3, 1]
    assert pareto_oracle.front_indices([[nan, 0.1, 0, 0], [nan, nan, 0, 0], [nan, 0.4, 0, 0], [0.5, 0.5, 0, 0]]) == [3, 2, 0, 1]
    # a NaN constraint is feasible (NaN > 1 is false); NaN tuples are never duplicates of each other
    assert pareto_oracle.front_indices([[0.3, 0.3, nan, 0], [0.3, 0.3, nan, 0], [0.3, 0.3, 2, 0]]) == [0, 1]
    # a NaN crowd distance goes after every number in the descending crowd sort
    f = np.array([[0.0, 1.0], [0.1, 0.9], [nan, 0.5], [0.5, 0.5], [0.6, 0.4], [0.7, 0.1], [1.0, 0.0]])
    assert pareto_oracle.thin_order(f, [0, 1, 2, 3], max_front=6) == [0, 5, 4, 1, 2, 6]     # crowd: 5 > 4 > NaN, NaN, NaN
    assert all(np.isnan(pareto_oracle.front_stats(np.c_[f, np.zeros((7, 2))], thin_pick=[4, 3, 2, 1], max_front=6)[1:5]))


# Both reference-pinned checks run against the utils.py of a test run (MAX_FRONT = 50, the step-end draw of 48) and of the
# training driver (train/code/utils.py: MAX_FRONT = 20, a draw of 18).

@pytest.mark.skipif(not ref_harness.available(), reason="reference tree not present")
def test_oracle_matches_reference_utils():
    check_reference_utils("small_bridge", 50)


@pytest.mark.skipif(not ref_harness.available(), reason="reference tree not present")
def test_oracle_matches_training_utils():
    check_reference_utils("train", 20)


@pytest.mark.skipif(not ref_harness.available(), reason="reference tree not present")
def test_thinning_of_large_fronts_matches_reference():
    check_reference_thinning("small_bridge", 50)


@pytest.mark.skipif(not ref_harness.available(), reason="reference tree not present")
def test_thinning_at_the_training_max_front_matches_reference():
    check_reference_thinning("train", 20)


def check_reference_utils(run, max_front):
    """objectives in [0, 2] (the driver divides by the initial design's, so a worse design is above 1) and reference points
    on both sides of 1"""
    utils = ref_harness.load_utils(run)
    rng = np.random.RandomState(3)
    for trial in range(150):
        n = rng.randint(1, 51)
        pts = rng.rand(n, 4) * 2
        pts[:, 2:] *= 0.65
        pts[rng.randint(n), 2:] = 0.2
        if trial == 0:
            pts[0] = (1.0, 1.0, 0.2, 0.2)                   # the driver's first front: the initial design alone
            n, pts = 1, pts[:1]
        ref = [float(0.7 + 0.6 * rng.rand()), float(0.7 + 0.6 * rng.rand())]
        want = utils.simple_cull([list(map(float, p)) for p in pts])
        got = pareto_oracle.front_stats(pts, max_front=max_front)
        assert np.array_equal(got[0], np.array(want[0]))
        assert np.allclose(got[1:], want[1:], rtol=1e-12, atol=1e-14)
        hv_want = utils.union_rectangles_fastest([list(f) for f in want[0]], +1, -1, ref_point=ref)
        assert abs(pareto_oracle.hypervolume(got[0], ref) - hv_want) <= 1e-12
        # the hypervolume of an arbitrary (dominated) list too
        hv_all = utils.union_rectangles_fastest([list(map(float, p)) for p in pts], +1, -1, ref_point=ref)
        assert abs(pareto_oracle.hypervolume(pts, ref) - hv_all) <= 1e-12


def check_reference_thinning(run, max_front):
    """fronts of more than MAX_FRONT members (the step-end cull of up to 50 + 150 accumulated candidates,
    master_DDPG_truss2D_MO.py:437): the reference's random.sample is replaced by an explicit draw on both sides;
    objectives in [0, 2], reference points on both sides of 1"""
    utils = ref_harness.load_utils(run)
    rng = np.random.RandomState(5)
    done = 0
    for trial in range(40):
        n = rng.randint(120, 201)
        t = np.sort(rng.rand(n)) * 2
        pts = np.stack([t, 2.0 - 2.0 * (t / 2) ** (0.5 + rng.rand()) + 0.004 * rng.rand(n), rng.rand(n) * 0.9,
                        rng.rand(n) * 0.9], axis=1)
        pts = pts[rng.permutation(n)]
        F = len(pareto_oracle.front_indices(pts))
        if F <= max_front:
            continue
        pick = [int(k) for k in rng.permutation(F - 2)[:max_front - 2]]
        orig = utils.random.sample
        utils.random.sample = lambda pop, k: [pop[i] for i in pick[:k]]
        try:
            want = utils.simple_cull([list(map(float, p)) for p in pts])
        finally:
            utils.random.sample = orig
        got = pareto_oracle.front_stats(pts, thin_pick=pick, max_front=max_front)
        assert len(want[0]) == max_front and np.array_equal(got[0], np.array(want[0]))
        assert np.allclose(got[1:], want[1:], rtol=1e-12, atol=1e-14)
        ref = [0.9, 1.2] if trial % 2 else [1.1, 0.95]
        hv_want = utils.union_rectangles_fastest([list(f) for f in want[0]], +1, -1, ref_point=ref)
        assert abs(pareto_oracle.hypervolume(got[0], ref) - hv_want) <= 1e-12
        done += 1
    assert done >= 10
    with pytest.raises(ValueError):
        pareto_oracle.front_stats(pts, max_front=max_front)     # a large front needs the draw
