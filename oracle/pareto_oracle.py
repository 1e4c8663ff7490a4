"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's Pareto-front bookkeeping (SURVEY.md section 8f-2).

Follows ``test/00_small_bridge/code/utils.py`` (identical in the four test directories):

  * ``front_stats``  = ``simple_cull`` (:11-217): feasibility cut (con1 > 1 or con2 > 1 drops the point, :17-23), strict
    two-objective dominance (``dominates``, :8-9), the front as a SET of tuples sorted by obj1 (:56-57), and the spread
    statistics returned next to it: max / deviation / sum of the consecutive distances (:159-170) and the normalised
    crowding distances' 10-norm and standard deviation (:172-195).
  * ``hypervolume``  = ``union_rectangles_fastest`` (:463-530): area of the union of the rectangles
    [min(x,1), 1] x [0, 1 - min(y,1)], minus the strip the moving reference point cuts off.  The reference sweeps with
    a segment tree; for axis-aligned rectangles that all touch x = 1 and y = 0 the union is the integral of the running
    maximum height over the sorted x, which is what is evaluated here.

Parity status: **pinned** -- ``tests/test_pareto_oracle.py`` runs both functions against the imported reference
``utils.py`` on random point sets (float64 inputs, so both sides compute in float64) and against
``tests/golden/pareto.npz`` recorded from the reference by ``tests/golden/make_golden_pareto.py``.  (With the driver's
``np.float32`` points the reference's scalar arithmetic runs in float32; the statistics then agree to ~1e-6.)
The reference samples the front down with ``random.sample`` when it holds more than MAX_FRONT points (:120-142; 50 in the
test runs, 20 in ``train/code``): the first and the last member stay, MAX_FRONT - 2 of the others are drawn from the list sorted by crowd distance (descending, stable)
and keep the ORDER of the draw.  ``front_stats(points, thin_pick=...)`` reproduces it for an explicit draw: ``thin_pick`` is
what ``random.sample(range(F - 2), MAX_FRONT - 2)`` returned (positions in that sorted list); the pinning test feeds the same
positions to the reference by patching ``utils.random.sample``.
"""
from __future__ import annotations

import numpy as np

MAX_FRONT = 50


def nan_last(v):
    """sort key of a number with NumPy's NaN convention: after every number, NaNs tied.  The reference sorts with Python's
    comparisons, which are not an order once a NaN is present, so its result there depends on the input order: a known
    divergence (DESIGN.md section 4)."""
    return (1, 0.0) if v != v else (0, v)


def front_indices(points):
    """indices of the Pareto front of ``points`` [P,4] in the reference's order (obj1 ascending)"""
    pts = [tuple(float(v) for v in p) for p in np.asarray(points, dtype=np.float64)]
    feas = [i for i, p in enumerate(pts) if not (p[2] > 1 or p[3] > 1)]            # utils.py:17-23
    if not feas:
        raise IndexError("simple_cull: no feasible point (the reference indexes an empty list, utils.py:29)")
    front, seen = [], set()
    for i in feas:
        if pts[i] in seen:                                                         # paretoPoints is a set of tuples
            continue
        if any(pts[j][0] < pts[i][0] and pts[j][1] < pts[i][1] for j in feas):     # dominates(), strict in both
            continue
        seen.add(pts[i])
        front.append(i)
    front.sort(key=lambda i: (nan_last(pts[i][0]), nan_last(-pts[i][1]), i))       # sorted by obj1 (:57); ties: see tests
    return front


def thin_order(f, thin_pick, max_front=MAX_FRONT):
    """positions (into the obj1-sorted front ``f`` [F,>=2]) of the thinned front, in the reference's order (:104-131)"""
    F = len(f)
    d = np.sqrt((f[:-1, 0] - f[1:, 0]) ** 2 + (f[:-1, 1] - f[1:, 1]) ** 2)
    crowd = np.empty(F)
    crowd[0], crowd[-1] = d[0], d[-1]
    crowd[1:-1] = d[:-1] + d[1:]
    interior = sorted(range(1, F - 1), key=lambda i: nan_last(-crowd[i]))         # descending, stable: ties keep the obj1 order
    pick = [int(k) for k in thin_pick]
    if len(pick) != max_front - 2 or len(set(pick)) != len(pick) or min(pick) < 0 or max(pick) >= F - 2:
        raise ValueError("thin_pick must hold %d distinct positions below %d" % (max_front - 2, F - 2))
    return [0] + [interior[k] for k in pick] + [F - 1]


def front_stats(points, thin_pick=None, max_front=MAX_FRONT):
    """``simple_cull(points)``: (front [F,4], max_distance, dis_distance, p_norm_inv_cd, sum_distance, std_cd).  A front of
    more than ``max_front`` members is thinned with the draw ``thin_pick`` (see the module docstring); the statistics are then
    those of the thinned list in its draw order, as in the reference."""
    pts = np.asarray(points, dtype=np.float64)
    idx = front_indices(pts)
    f = pts[idx]
    if len(idx) > max_front:
        if thin_pick is None:
            raise ValueError("front of %d members: the reference draws %d of them at random; pass thin_pick" % (len(idx), max_front - 2))
        f = f[thin_order(f, thin_pick, max_front)]
    F = len(f)
    if F >= 2:                                                                      # :159-166
        d = np.sqrt((f[:-1, 0] - f[1:, 0]) ** 2 + (f[:-1, 1] - f[1:, 1]) ** 2)
        max_d = float(d.max())
        dis_d = float(np.sqrt(np.sum((d - max_d / len(d)) ** 2) / len(d)))
        sum_d = float(d.sum())
    else:                                                                           # :167-170
        dis_d, max_d, sum_d = 1.0, 0.0, 0.0
    if F > 3:                                                                       # :176-190
        c = np.abs(f[:-2, 0] - f[2:, 0]) + np.abs(f[:-2, 1] - f[2:, 1])
        if c.sum() == 0:
            std_cd, p_inv = 1.0, 0.0
        else:
            c = c / c.max()
            std_cd = float(np.std(c))
            p_inv = float(np.sum(np.abs(c) ** 10) ** 0.1)
    else:
        std_cd, p_inv = 1.0, 0.0
    return f, max_d, dis_d, p_inv, sum_d, std_cd


def hypervolume(R, ref_point=(1.0, 1.0)):
    """``union_rectangles_fastest(R, +1, -1, ref_point)`` for a list of points (only columns 0 and 1 are used)"""
    R = np.asarray(R, dtype=np.float64).reshape(-1, np.asarray(R).shape[-1] if np.asarray(R).ndim > 1 else 2)
    if len(R) == 0:
        return 0.0
    if len(R) == 1 and R[0][0] == 1 and R[0][1] == 1:                               # :476-477
        return 0.0
    x = np.minimum(R[:, 0], 1.0)
    h = 1.0 - np.minimum(R[:, 1], 1.0)
    order = np.argsort(x, kind="stable")
    xs, hs = x[order], np.maximum.accumulate(h[order])
    edges = np.append(xs, 1.0)
    area = float(np.sum((edges[1:] - edges[:-1]) * hs))
    rx, ry = float(ref_point[0]), float(ref_point[1])
    remove = (1 - rx) * (1 - R[:, 0].min()) + (1 - ry) * (1 - R[:, 1].min()) - (1 - rx) * (1 - ry)   # :527
    return area - remove
