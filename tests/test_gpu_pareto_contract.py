"""GPU: the Pareto-front kernels (csrc/tpareto.cu) at the edges the driver reaches and the C ABI accepts, each case against
oracle/pareto_oracle.py (front membership and order exact, the five statistics and the hypervolume to 1e-12, NaN where
the oracle gives NaN) and, for the Pareto graph, against oracle/truss_oracle.pareto_state_data bit for bit:

  * thinning at the training driver's MAX_FRONT = 20 and across 3..64, with exact crowd-distance ties;
  * batches past one pass of the grid (4 warps x 8 CTAs per SM), where warps reuse their shared memory;
  * the driver's value range: objectives normalised by the initial design, so above 1, the lone (1, 1) first front,
    reference points on both sides of 1, constraints at exactly 1;
  * counts, NULL outputs, P and the documented refusals of the C ABI;
  * non-finite points: NaN sorts after every number (NumPy's convention), statistics and hypervolume propagate it.
"""
import ctypes as C
import math
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import pareto_oracle                  # noqa: E402
from oracle.truss_oracle import pareto_state_data  # noqa: E402

EMPTY_STATS = [0.0, 1.0, 0.0, 0.0, 1.0]
TFEM_ERR_ARG, TFEM_ERR_ALIGN = -1, -4


@pytest.fixture(scope="module")
def pareto():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mop_truss_marl_b200 import pareto as mod
    return mod


@pytest.fixture(scope="module")
def grid_pass():
    """environments one launch covers before its warps start over: 4 warps x 8 CTAs per SM"""
    return 4 * 8 * torch.cuda.get_device_properties(0).multi_processor_count


def run(pareto, pts, counts=None, ref=(1.0, 1.0), picks=None, max_front=20):
    pts_d = torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float32)).cuda()
    cnt_d = None if counts is None else torch.from_numpy(np.ascontiguousarray(counts, np.int32)).cuda()
    pick_d = None if picks is None else torch.from_numpy(np.ascontiguousarray(picks, np.int32)).cuda()
    out = pareto.front_hv(pts_d, cnt_d, ref, thin_pick=pick_d, max_front=max_front)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def expected(p, ref, pick=None, max_front=20):
    """(front indices into p in list order, stats, hv) of the oracle; front thinned with `pick` when it is larger than
    max_front and a draw is given; None when no point is feasible"""
    p = np.asarray(p, np.float64)
    try:
        idx = pareto_oracle.front_indices(p)
    except IndexError:
        return None
    thin = pick if len(idx) > max_front else None
    if thin is not None:
        idx = [idx[k] for k in pareto_oracle.thin_order(p[idx], thin, max_front)]
    f, max_d, dis_d, p_cd, sum_d, std_cd = pareto_oracle.front_stats(p, thin_pick=thin, max_front=max_front if thin is not None
                                                                     else max(max_front, len(idx)))
    assert np.array_equal(f, p[idx], equal_nan=True)
    return idx, [max_d, dis_d, p_cd, sum_d, std_cd], pareto_oracle.hypervolume(f, ref)


def check_env(out, b, p, ref, pick=None, max_front=20):
    """environment b of a launch against the oracle: front_idx[:F] is a set of distinct points of this environment before it
    indexes anything, then membership and order exact, -1 padding, statistics and hypervolume to 1e-12"""
    n, P = len(p), out["front_idx"].shape[1]
    F, fi = int(out["front_len"][b]), out["front_idx"][b]
    assert 0 <= F <= n, (b, F, n)
    assert len(set(fi[:F].tolist())) == F and ((fi[:F] >= 0) & (fi[:F] < n)).all(), (b, fi[:F])
    assert (fi[F:] == -1).all() and len(fi) == P, b
    want = expected(p, ref, pick, max_front)
    if want is None:
        assert F == 0 and out["hv"][b] == 0.0 and np.array_equal(out["stats"][b], EMPTY_STATS), b
        return
    idx, stats, hv = want
    assert fi[:F].tolist() == idx, (b, fi[:F].tolist(), idx)
    assert np.allclose(out["stats"][b], stats, rtol=1e-12, atol=1e-14, equal_nan=True), (b, out["stats"][b], stats)
    assert np.allclose(out["hv"][b], hv, rtol=0, atol=1e-12, equal_nan=True), (b, out["hv"][b], hv)


def anti_chain(rng, F, lo=0.0, hi=1.0):
    """F mutually non-dominated feasible points with objectives in [lo, hi], in arbitrary order"""
    while True:
        x = np.sort(rng.uniform(lo, hi, F)).astype(np.float32)
        y = np.sort(rng.uniform(lo, hi, F))[::-1].astype(np.float32)
        if len(np.unique(x)) == F and len(np.unique(y)) == F:
            break
    p = np.stack([x, y, rng.rand(F) * 0.9, rng.rand(F) * 0.9], axis=1).astype(np.float32)
    return p[rng.permutation(F)]


def dyadic_chain(F, rng):
    """x = k/256, y = 1 - k/256: every gap is the same exact value, so every interior crowd distance ties and the stable
    rule (list order) alone orders the thinning"""
    k = np.arange(F, dtype=np.float64)
    p = np.stack([k / 256, 1 - k / 256, np.full(F, 0.5), np.full(F, 0.5)], axis=1).astype(np.float32)
    return p[rng.permutation(F)]


def with_dominated(rng, front, extra):
    """the front plus `extra` points each dominated by a front member, shuffled"""
    base = front[rng.randint(len(front), size=extra)].copy()
    base[:, :2] += (rng.rand(extra, 2) * 0.1 + 1e-3).astype(np.float32)
    p = np.concatenate([front, base]).astype(np.float32)
    return p[rng.permutation(len(p))]


def draw(rng, F, max_front):
    """random.sample(range(F - 2), max_front - 2) for a front that is thinned; garbage for one that is not (never read)"""
    if F > max_front:
        return rng.permutation(F - 2)[:max_front - 2].astype(np.int32)
    return np.where(rng.rand(max_front - 2) < 0.5, -1, 10 ** 6).astype(np.int32)


def pack(envs, P=None):
    P = P or max(len(e) for e in envs)
    pts = np.full((len(envs), P, 4), 7.0, np.float32)          # beyond count: infeasible garbage that must not be read
    for b, e in enumerate(envs):
        pts[b, :len(e)] = e
    return pts, np.array([len(e) for e in envs], np.int32)


# ---- thinning ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("max_front", [3, 20, 32, 33, 50, 64])
def test_thinning_across_max_front(pareto, max_front):
    """fronts of exactly max_front (not thinned), max_front + 1 and up to 256 members, random and dyadic (all crowd
    distances tied), with dominated points mixed in; draws in arbitrary order; unthinned rows of the draw are garbage"""
    rng = np.random.RandomState(max_front)
    sizes = [max_front, max_front + 1, max_front + 2, 2 * max_front, 256, rng.randint(max_front + 1, 257)]
    envs = []
    for F in sizes:
        envs.append(anti_chain(rng, F))
        envs.append(dyadic_chain(F, rng))
        if F + 20 <= 256:
            envs.append(with_dominated(rng, anti_chain(rng, F, 0.0, 2.0), 20))
    envs.append(anti_chain(rng, max_front - 1))
    pts, counts = pack(envs, 256)
    picks = np.stack([draw(rng, len(pareto_oracle.front_indices(e)), max_front) for e in envs])
    for ref in ((1.0, 1.0), (0.9, 1.3)):
        out = run(pareto, pts, counts, ref, picks, max_front)
        for b, e in enumerate(envs):
            check_env(out, b, e, ref, picks[b], max_front)
        assert out["front_len"].max() == max_front


def contracted_dist(ax, ay):
    """sqrt(fma(ax, ax, ay * ay)): the gap length as nvcc contracts it by default, computed exactly"""
    return math.sqrt(float(Fraction(ax) * Fraction(ax) + Fraction(ay * ay)))


def mirror_front(v):
    """the 4-point front (a, b), (c, d), (d, c), (b, a) for a < c < d < b: symmetric under obj1 <-> obj2, so its two
    interior members have exactly equal crowd distances when each product is rounded"""
    a, c, d, b = v
    return np.array([[a, b, .5, .5], [c, d, .5, .5], [d, c, .5, .5], [b, a, .5, .5]], np.float32)


def test_mirrored_gaps_tie_in_the_crowd_sort(pareto):
    """A front symmetric under obj1 <-> obj2 has mirrored gaps (p, q) / (q, p): with rounded products their crowd distances
    tie exactly and the stable sort keeps the list order. A contracted fma(p, p, q * q) and fma(q, q, p * p) differ for
    objectives spread over several binades, which flipped the member a draw picks (thinning to 3 of 4 keeps one of the two
    interior members)."""
    flip = np.array([float.fromhex(h) for h in ("0x1.ab96ecp-12", "0x1.b02d98p-10", "0x1.86ea3ep-6", "0x1.4d927ap-2")])
    f = mirror_front(flip).astype(np.float64)
    gap = [(f[k, 0] - f[k + 1, 0], f[k, 1] - f[k + 1, 1]) for k in range(3)]
    fused = [contracted_dist(*g) for g in gap]
    assert fused[0] + fused[1] < fused[1] + fused[2]            # contracted, the second interior member sorts first
    rng = np.random.RandomState(4)
    envs = [mirror_front(flip)]
    while len(envs) < 2000:                                       # more of them, about 1 in 20 a contraction flip
        v = np.sort((2.0 ** rng.uniform(-12, 1, 4)).astype(np.float32))
        if len(np.unique(v)) == 4:
            envs.append(mirror_front(v))
    envs = [e[rng.permutation(4)] for e in envs]
    pts, counts = pack(envs)
    picks = np.zeros((len(envs), 1), np.int32)
    out = run(pareto, pts, counts, (1.0, 1.0), picks, 3)
    for b, e in enumerate(envs):
        check_env(out, b, e, (1.0, 1.0), picks[b], 3)
    # and in a longer symmetric front at the driver's MAX_FRONT
    v = np.sort((2.0 ** rng.uniform(-12, 1, 40)).astype(np.float32)).astype(np.float64)
    half = np.stack([v[:20], v[::-1][:20]], axis=1)
    sym = np.concatenate([half, half[:, ::-1]])
    sym = np.concatenate([sym, np.full((40, 2), 0.5)], axis=1).astype(np.float32)
    pick = rng.permutation(38)[:18].astype(np.int32)
    out = run(pareto, sym[None], None, (1.0, 1.0), pick[None], 20)
    check_env(out, 0, sym, (1.0, 1.0), pick, 20)


# ---- more than one pass of the grid -------------------------------------------------------------------------------------

def light_env(rng):
    """at most 20 points, so never thinned at MAX_FRONT = 20"""
    n = rng.randint(1, 21)
    p = (rng.rand(n, 4) * [2.0, 2.0, 1.3, 1.3]).astype(np.float32)
    if rng.rand() < 0.2:
        p[:, 2] = 5.0                                            # no feasible point
    return p


def grid_batch(rng, B, grid_pass):
    """light environments, with 256-member anti-chains (thinned to 20) on a warp slot of one pass whose same slot in the next
    pass is light, and the other way round"""
    envs = [light_env(rng) for _ in range(B)]
    for b in range(0, B, 97):
        envs[b] = anti_chain(rng, 256, 0.0, 2.0)
        if b + grid_pass < B:
            envs[b + grid_pass] = light_env(rng)
        if b >= grid_pass:
            envs[b - grid_pass] = light_env(rng)
    return envs


def launch_each_alone(pareto, pts_d, cnt_d, pick_d, max_front, ref):
    """every environment in a launch of its own (B = 1, offset pointers into the batch's buffers)"""
    B, P = pts_d.shape[:2]
    oi = torch.full((B, P), -7, dtype=torch.int32, device="cuda")
    ol = torch.full((B,), -7, dtype=torch.int32, device="cuda")
    os_ = torch.full((B, 5), -7.0, dtype=torch.float64, device="cuda")
    oh = torch.full((B,), -7.0, dtype=torch.float64, device="cuda")
    r = (C.c_double * 2)(*ref)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib = pareto._lib
    for b in range(B):
        rc = lib.tpareto_front_hv_thin(1, P, C.c_void_p(pts_d[b].data_ptr()), C.c_void_p(cnt_d[b:].data_ptr()),
                                       C.cast(r, C.c_void_p), C.c_void_p(pick_d[b].data_ptr()), max_front,
                                       C.c_void_p(oi[b].data_ptr()), C.c_void_p(ol[b:].data_ptr()),
                                       C.c_void_p(os_[b].data_ptr()), C.c_void_p(oh[b:].data_ptr()), st)
        assert rc == 0
    torch.cuda.synchronize()
    return {"front_idx": oi.cpu().numpy(), "front_len": ol.cpu().numpy(), "stats": os_.cpu().numpy(), "hv": oh.cpu().numpy()}


def same_bits(a, b):
    return all(np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)) for k in ("front_idx", "front_len", "stats", "hv"))


@pytest.mark.parametrize("which", ["below", "equal", "above", "16384"])
def test_batches_past_one_grid_pass(pareto, grid_pass, which):
    B = {"below": grid_pass - 1, "equal": grid_pass, "above": grid_pass + 1, "16384": 16384}[which]
    rng = np.random.RandomState(B)
    max_front, ref = 20, (1.05, 0.95)
    envs = grid_batch(rng, B, grid_pass)
    pts, counts = pack(envs, 256)
    lens = [len(e) for e in envs]                                # the 256-point environments are anti-chains
    picks = np.stack([draw(rng, F, max_front) for F in lens])
    out = run(pareto, pts, counts, ref, picks, max_front)
    # bit-identical to the same environment in a reversed batch and in a batch of its own
    rev = run(pareto, pts[::-1], counts[::-1], ref, picks[::-1], max_front)
    assert same_bits(out, {k: v[::-1].copy() for k, v in rev.items()})
    alone = launch_each_alone(pareto, torch.from_numpy(pts).cuda(), torch.from_numpy(counts).cuda(),
                              torch.from_numpy(picks).cuda(), max_front, ref)
    assert same_bits(out, alone)
    # the oracle on >= 200 environments, all of the second pass's first warp slots among them
    second_first = [b for b in range(grid_pass, min(B, 2 * grid_pass)) if b % 4 == 0]
    sample = sorted(set(range(0, B, max(1, B // 200))) | set(second_first) | set(range(0, B, 97)) | {B - 1})
    assert len(sample) >= 200
    for b in sample:
        check_env(out, b, envs[b], ref, picks[b], max_front)
    assert max(lens) == 256 and out["front_len"].max() == max_front


# ---- the driver's value range ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ref", [(1.0, 1.0), (0.8, 0.9), (1.2, 1.4), (0.9, 1.25)])
def test_driver_value_range(pareto, ref):
    """objectives normalised by the initial design (point = obj / int_obj, so above 1 for a worse design), the driver's
    first front (the lone (1, 1)), constraints at exactly 1 (feasible) and one ulp above (infeasible), duplicates, -0.0 / 0.0,
    many exact ties in obj1"""
    rng = np.random.RandomState(int(ref[0] * 100 + ref[1] * 10))
    one_up = np.nextafter(np.float32(1), np.float32(2))
    envs = [
        np.array([[1, 1, 0.5, 0.5]], np.float32),
        np.array([[1, 1, 0.5, 0.5], [1.3, 1.2, 0.5, 0.5], [1.5, 0.8, 0.2, 0.3]], np.float32),
        np.array([[1, 1, 0.5, 0.5], [0.7, 0.9, 0.5, 0.5]], np.float32),
        np.array([[1, 1, 0.5, 0.5], [0.7, 1.4, 0.5, 0.5], [1.6, 0.2, 0.5, 0.5], [1.2, 1.3, 0.1, 0.1]], np.float32),
        np.array([[1, 1, 0.5, 0.5], [1, 1, 0.5, 0.5]], np.float32),
        np.array([[1.5, 1.7, 0.5, 0.5]], np.float32),
        np.array([[0.4, 0.6, 1.0, 1.0], [0.3, 0.5, one_up, 0.2], [0.2, 0.9, 0.1, one_up], [0.5, 0.4, 1.0, 0.0]], np.float32),
        np.array([[0.3, 0.3, 1.5, 0.1], [0.3, 0.3, 1.5, 0.1], [0.1, 0.1, 3.0, 3.0], [0.6, 0.6, 0.5, 0.5]], np.float32),
        np.array([[0.0, 0.7, 0.5, 0.5], [-0.0, 0.7, 0.5, 0.5], [0.5, -0.0, 0.5, 0.5], [0.5, 0.0, 0.5, 0.5]], np.float32),
        np.array([[-0.0, 0.9, 0.5, 0.5], [0.0, 0.4, 0.5, 0.5], [0.0, 0.8, 0.5, 0.5], [0.7, 0.0, 0.5, 0.5]], np.float32),
    ]
    for _ in range(60):
        n = rng.randint(1, 200)
        p = (rng.rand(n, 4) * [2.0, 2.0, 1.2, 1.2]).astype(np.float32)
        if rng.rand() < 0.3:
            p[:, 0] = np.round(p[:, 0] * 4) / 4                  # many exact ties in obj1
        if rng.rand() < 0.3:
            p[rng.randint(n, size=n // 3 + 1)] = p[rng.randint(n)]   # duplicates
        if rng.rand() < 0.3:
            p[:, 2] = np.where(rng.rand(n) < 0.5, np.float32(1.0), one_up)
        envs.append(p)
    for _ in range(10):
        envs.append(anti_chain(rng, rng.randint(2, 60), 0.0, 2.0))
    pts, counts = pack(envs, 256)
    out = run(pareto, pts, counts, ref)
    for b, e in enumerate(envs):
        check_env(out, b, e, ref, max_front=256)
    assert out["hv"][0] == 0.0 and out["front_len"][0] == 1 and out["front_len"][4] == 1 and out["hv"][4] == 0.0
    assert out["front_idx"][6, :2].tolist() == [0, 3]           # con == 1.0 stays, one ulp above is cut
    assert out["front_len"][8] == 2 and out["front_idx"][8, :2].tolist() == [0, 2]   # -0.0 duplicates 0.0


# ---- arguments ------------------------------------------------------------------------------------------------------------

def test_counts_are_clamped_to_0_P(pareto):
    """counts of 0 or below: an empty environment; above P: P points; NULL: P points"""
    rng = np.random.RandomState(2)
    B, P = 12, 40
    pts = (rng.rand(B, P, 4) * [1, 1, 1.2, 1.2]).astype(np.float32)
    pts[:, 0, 2:] = 0.1
    counts = np.array([0, -1, -(2 ** 31), P + 1, 2 ** 31 - 1, P, 1, 17, 0, P + 100, 39, 3], np.int32)
    out = run(pareto, pts, counts, (0.9, 0.9))
    for b in range(B):
        n = min(max(int(counts[b]), 0), P)
        if n == 0:
            assert out["front_len"][b] == 0 and (out["front_idx"][b] == -1).all() and out["hv"][b] == 0.0
            assert np.array_equal(out["stats"][b], EMPTY_STATS)
        else:
            check_env(out, b, pts[b, :n], (0.9, 0.9))
    full = run(pareto, pts, np.full(B, P, np.int32), (0.9, 0.9))
    null = run(pareto, pts, None, (0.9, 0.9))
    assert same_bits(full, null)
    for b in np.flatnonzero(counts >= P):
        assert all(np.array_equal(full[k][b:b + 1].view(np.uint8), out[k][b:b + 1].view(np.uint8)) for k in full)


def raw_call(pareto, thin, B, P, pts_ptr, cnt, ref, pick, max_front, outs):
    r = (C.c_double * 2)(*ref)
    p = lambda t: C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    if thin:
        return pareto._lib.tpareto_front_hv_thin(B, P, pts_ptr, p(cnt), C.cast(r, C.c_void_p), p(pick), max_front,
                                                 *[p(o) for o in outs], st)
    return pareto._lib.tpareto_front_hv(B, P, pts_ptr, p(cnt), C.cast(r, C.c_void_p), *[p(o) for o in outs], st)


def sentinels(B, P):
    return [torch.full((B, P), -5, dtype=torch.int32, device="cuda"), torch.full((B,), -5, dtype=torch.int32, device="cuda"),
            torch.full((B, 5), -5.5, dtype=torch.float64, device="cuda"), torch.full((B,), -5.5, dtype=torch.float64, device="cuda")]


@pytest.mark.parametrize("thin", [False, True])
def test_each_output_may_be_null(pareto, thin):
    """any one output NULL: the others are what a call with all four writes, bit for bit"""
    rng = np.random.RandomState(8)
    envs = [anti_chain(rng, rng.randint(1, 80), 0.0, 2.0) for _ in range(300)]
    pts, counts = pack(envs, 128)
    picks = np.stack([draw(rng, len(e), 20) for e in envs])
    pts_d, cnt_d, pick_d = torch.from_numpy(pts).cuda(), torch.from_numpy(counts).cuda(), torch.from_numpy(picks).cuda()
    B, P = pts.shape[:2]
    full = sentinels(B, P)
    assert raw_call(pareto, thin, B, P, C.c_void_p(pts_d.data_ptr()), cnt_d, (0.95, 1.1), pick_d, 20, full) == 0
    for k in range(4):
        outs = sentinels(B, P)
        outs[k] = None
        assert raw_call(pareto, thin, B, P, C.c_void_p(pts_d.data_ptr()), cnt_d, (0.95, 1.1), pick_d, 20, outs) == 0
        torch.cuda.synchronize()
        for j in range(4):
            if j != k:
                assert torch.equal(outs[j].view(torch.uint8) if outs[j].dtype == torch.float64 else outs[j],
                                   full[j].view(torch.uint8) if full[j].dtype == torch.float64 else full[j]), (k, j)
    res = dict(zip(("front_idx", "front_len", "stats", "hv"), (t.cpu().numpy() for t in full)))
    for b in range(0, B, 7):
        check_env(res, b, envs[b], (0.95, 1.1), picks[b] if thin else None, 20 if thin else 256)


@pytest.mark.parametrize("P", [1, 31, 33, 255, 256])
def test_points_per_environment(pareto, P):
    rng = np.random.RandomState(P)
    B = 70
    pts = (rng.rand(B, P, 4) * [2, 2, 1.3, 1.3]).astype(np.float32)
    pts[1] = anti_chain(rng, P, 0.0, 2.0)
    counts = rng.randint(1, P + 1, size=B).astype(np.int32)
    counts[:2] = P
    picks = np.stack([draw(rng, len(pareto_oracle.front_indices(pts[b, :counts[b]])) if (pts[b, :counts[b], 2:] <= 1).all(1).any()
                           else 0, 20) for b in range(B)])
    for thin in (False, True):
        out = run(pareto, pts, counts, (1.1, 0.9), picks if thin else None, 20)
        for b in range(B):
            check_env(out, b, pts[b, :counts[b]], (1.1, 0.9), picks[b] if thin else None, 20 if thin else 256)


def test_refusals_leave_outputs_untouched(pareto):
    """each documented refusal returns its code and message and writes nothing"""
    B, P = 6, 32
    rng = np.random.RandomState(1)
    big = torch.from_numpy(rng.rand(B * 257 * 4 + 8).astype(np.float32)).cuda()
    pts_ptr = C.c_void_p(big.data_ptr())
    cnt = torch.full((B,), P, dtype=torch.int32, device="cuda")
    pick = torch.zeros(B, 62, dtype=torch.int32, device="cuda")
    cases = [
        (False, 0, None, 50, TFEM_ERR_ARG, "P must be in 1..256"),
        (False, 257, None, 50, TFEM_ERR_ARG, "P must be in 1..256"),
        (True, 0, pick, 20, TFEM_ERR_ARG, "P must be in 1..256"),
        (True, 257, pick, 20, TFEM_ERR_ARG, "P must be in 1..256"),
        (True, P, pick, 2, TFEM_ERR_ARG, "max_front must be in 3..64"),
        (True, P, pick, 65, TFEM_ERR_ARG, "max_front must be in 3..64"),
        (True, P, None, 20, TFEM_ERR_ARG, "null thin_pick"),
    ]
    for thin, p, pk, mf, code, msg in cases:
        outs = sentinels(B, 257)
        assert raw_call(pareto, thin, B, p, pts_ptr, cnt, (1, 1), pk, mf, outs) == code
        assert pareto._lib.tpareto_last_error().decode() == msg
        torch.cuda.synchronize()
        assert all((o == -5).all() if o.dtype == torch.int32 else (o == -5.5).all() for o in outs), (thin, p, mf)
    for thin in (False, True):                                     # points 4 bytes past a 16-byte boundary
        outs = sentinels(B, P)
        assert raw_call(pareto, thin, B, P, C.c_void_p(big.data_ptr() + 4), cnt, (1, 1), pick, 20, outs) == TFEM_ERR_ALIGN
        assert pareto._lib.tpareto_last_error().decode() == "points must be 16-byte aligned"
        torch.cuda.synchronize()
        assert all((o == -5).all() if o.dtype == torch.int32 else (o == -5.5).all() for o in outs)


# ---- non-finite points ----------------------------------------------------------------------------------------------------

NONFINITE = [np.nan, np.inf, -np.inf]


def nonfinite_envs(rng):
    """every non-finite value in every column of small fronts, alone, twice and next to ties"""
    envs = []
    for v in NONFINITE:
        for col in range(4):
            for _ in range(6):
                n = rng.randint(2, 12)
                p = anti_chain(rng, n, 0.0, 2.0)
                p[rng.randint(n, size=rng.randint(1, 3)), col] = v
                if rng.rand() < 0.3:
                    p[rng.randint(n), 0] = p[rng.randint(n), 0]       # an obj1 tie
                envs.append(p)
    envs.append(np.array([[0.2, 0.8, 0, 0], [np.nan, 0.5, 0, 0], [0.6, 0.3, 0, 0], [0.9, 0.1, 0, 0]], np.float32))
    envs.append(np.array([[0.6, 0.8, 0, 0], [0.6, np.nan, 0, 0], [0.6, 0.3, 0, 0], [0.2, 0.9, 0, 0]], np.float32))
    envs.append(np.array([[np.nan, np.nan, np.nan, np.nan]] * 3, np.float32))
    envs.append(np.array([[np.inf, 0.5, 0, 0], [np.inf, 0.2, 0, 0], [-np.inf, np.inf, 0, 0], [0.4, -np.inf, 0, 0]], np.float32))
    return envs


def test_non_finite_points(pareto):
    """A NaN objective is never dominated and dominates nothing; a NaN constraint is feasible (NaN > 1 is false). The list
    puts NaN after every number in obj1 and, within equal obj1, in the obj2 key (NumPy's sort convention); the statistics
    and the hypervolume are the oracle's, NaN included"""
    rng = np.random.RandomState(12)
    envs = nonfinite_envs(rng)
    pts, counts = pack(envs)
    for ref in ((1.0, 1.0), (0.9, 1.2)):
        out = run(pareto, pts, counts, ref)
        for b, e in enumerate(envs):
            check_env(out, b, e, ref, max_front=256)
    assert np.isnan(out["hv"]).sum() >= 20 and np.isnan(out["stats"][:, 0]).sum() >= 20


def test_nan_rank_in_a_reused_warp_slot(pareto, grid_pass):
    """The NaN environment runs in the grid's second pass on the warp that ran a 200-member anti-chain stored in descending
    obj1 in the first, so any list slot the ranking left unwritten would hold an index of that environment (>= 4)"""
    rng = np.random.RandomState(21)
    B = grid_pass + 8
    envs = [light_env(rng) for _ in range(B)]
    nan_env = np.array([[0.2, 0.8, 0, 0], [np.nan, 0.5, 0, 0], [0.6, 0.3, 0, 0], [0.9, 0.1, 0, 0]], np.float32)
    for s in range(3, 8):
        chain = anti_chain(rng, 200)
        envs[s] = chain[np.argsort(-chain[:, 0], kind="stable")]
        envs[grid_pass + s] = nan_env if s % 2 else nan_env[[0, 2, 1, 3]]
    pts, counts = pack(envs, 256)
    out = run(pareto, pts, counts, (1.0, 1.0))
    for b in list(range(0, 8)) + list(range(grid_pass, B)):
        check_env(out, b, envs[b], (1.0, 1.0), max_front=256)
    assert out["front_idx"][grid_pass + 3, :4].tolist() == [0, 2, 3, 1] and np.isnan(out["hv"][grid_pass + 3])


def test_non_finite_points_thinned(pareto):
    """non-finite members in fronts that are thinned: NaN crowd distances sort after every number, stable"""
    rng = np.random.RandomState(13)
    envs, picks = [], []
    for v in NONFINITE:
        for col in range(2):
            for _ in range(8):
                F = rng.randint(21, 120)
                p = anti_chain(rng, F, 0.0, 2.0)
                p[rng.randint(F, size=rng.randint(1, 4)), col] = v
                envs.append(p)
    pts, counts = pack(envs, 128)
    picks = np.stack([draw(rng, len(pareto_oracle.front_indices(e)), 20) for e in envs])
    out = run(pareto, pts, counts, (1.0, 1.0), picks, 20)
    for b, e in enumerate(envs):
        check_env(out, b, e, (1.0, 1.0), picks[b], 20)


# ---- the driver's device chain: points -> front (thinned) -> Pareto graph --------------------------------------------------

def oracle_graph(front_pts, index, rows, max_front):
    wx, wA = np.zeros((rows, 4), np.float32), np.zeros((rows, rows), np.float32)
    if len(front_pts):
        x, A = pareto_state_data([(p[0], p[1]) for p in front_pts], index=index, max_front=max_front)
        m = min(len(front_pts), rows)
        wx[:m], wA[:m, :m] = x[:m], A[:m, :m]
    return wx, wA


@pytest.mark.parametrize("rows,max_front", [(20, 20), (50, 50)])
def test_front_to_state_data_chain(pareto, rows, max_front):
    """front_hv_thin's outputs fed to state_data on the device, as the driver's step does: x_p / A_p bit for bit the
    oracle chain's"""
    rng = np.random.RandomState(rows)
    envs = []
    for _ in range(150):
        kind = rng.randint(3)
        F = rng.randint(1, 200)
        envs.append(anti_chain(rng, F, 0.0, 2.0) if kind == 0 else light_env(rng) if kind == 1
                    else with_dominated(rng, anti_chain(rng, max(F // 2, 1), 0.0, 2.0), 30))
    envs[0] = np.array([[1, 1, 0.5, 0.5]], np.float32)
    pts, counts = pack(envs, 256)
    idxs = [pareto_oracle.front_indices(e) if (np.asarray(e[:, 2:], np.float64) <= 1).all(1).any() else [] for e in envs]
    picks = np.stack([draw(rng, len(i), max_front) for i in idxs])
    pts_d = torch.from_numpy(pts).cuda()
    out = pareto.front_hv(pts_d, torch.from_numpy(counts).cuda(), (1.0, 1.0), thin_pick=torch.from_numpy(picks).cuda(),
                          max_front=max_front)
    lens = out["front_len"].cpu().numpy()
    index = np.array([rng.randint(max(int(n), 1)) for n in lens], np.int32)
    x_p, A_p = pareto.state_data(pts_d, out["front_idx"], out["front_len"], torch.from_numpy(index).cuda(), rows=rows,
                                 max_front=max_front)
    torch.cuda.synchronize()
    x_p, A_p = x_p.cpu().numpy(), A_p.cpu().numpy()
    for b, e in enumerate(envs):
        idx = idxs[b]
        if len(idx) > max_front:
            idx = [idx[k] for k in pareto_oracle.thin_order(e[idx].astype(np.float64), picks[b], max_front)]
        assert lens[b] == len(idx)
        wx, wA = oracle_graph(e[idx], int(index[b]), rows, max_front)
        assert np.array_equal(x_p[b].view(np.uint32), wx.view(np.uint32)), b
        assert np.array_equal(A_p[b].view(np.uint32), wA.view(np.uint32)), b


def test_state_data_widest(pareto):
    """P_out = 64 rows from P_in = 256 points, front_len 0, inside and above P_in (clamped to P_in)"""
    rng = np.random.RandomState(64)
    B, P_in, rows, max_front = 40, 256, 64, 50
    pts = rng.rand(B, P_in, 4).astype(np.float32)
    perm = np.stack([rng.permutation(P_in) for _ in range(B)]).astype(np.int32)
    lens = rng.randint(1, P_in + 1, size=B).astype(np.int32)
    lens[:6] = (0, P_in, P_in + 1, 2 ** 31 - 1, 64, 65)
    index = np.array([rng.randint(max(min(int(n), P_in), 1)) for n in lens], np.int32)
    x_p, A_p = pareto.state_data(torch.from_numpy(pts).cuda(), torch.from_numpy(perm).cuda(), torch.from_numpy(lens).cuda(),
                                 torch.from_numpy(index).cuda(), rows=rows, max_front=max_front)
    torch.cuda.synchronize()
    x_p, A_p = x_p.cpu().numpy(), A_p.cpu().numpy()
    for b in range(B):
        n = min(int(lens[b]), P_in)
        wx, wA = oracle_graph(pts[b, perm[b, :n]], int(index[b]), rows, max_front)
        assert np.array_equal(x_p[b].view(np.uint32), wx.view(np.uint32)), b
        assert np.array_equal(A_p[b].view(np.uint32), wA.view(np.uint32)), b
