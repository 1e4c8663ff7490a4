"""GPU: mixed-family batches (tfem_step_mixed / tfem_reset_mixed, batched_env.MixedTrussEnv).  Every environment of a
mixed batch must be BIT-IDENTICAL, in every output, to the same environment stepped by a single-family BatchedTrussEnv
on the same inputs: the arithmetic and the table values are the same, only the pointer they are read through differs."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from util import adversarial_actions, adversarial_move_range

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

FIELDS = ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "point", "point64", "d", "axial", "ratio", "U",
          "reactions", "status", "y", "y_weak", "move_range")


def bits(t):
    return np.ascontiguousarray(t.detach().cpu().numpy()).view(np.uint8)


def assert_bits(got, want, tag):
    assert tuple(got.shape) == tuple(want.shape), (tag, got.shape, want.shape)
    a, b = bits(got), bits(want)
    if not np.array_equal(a, b):
        g, w = got.detach().cpu().numpy(), want.detach().cpu().numpy()
        bad = np.argwhere(a.reshape(len(g), -1) != b.reshape(len(w), -1))[0]
        raise AssertionError("%s differs first in environment %d: %r vs %r" % (tag, bad[0], g[bad[0]], w[bad[0]]))


class Twin:
    """a MixedTrussEnv and, per family, a BatchedTrussEnv holding that family's environments in batch order"""

    def __init__(self, families, ids):
        from mop_truss_marl_b200 import batched_env
        self.ids = np.asarray(ids, np.uint8)
        self.B = len(self.ids)
        self.mix = batched_env.MixedTrussEnv(families, self.B)
        self.dev = self.mix.device
        self.rows = [np.nonzero(self.ids == f)[0] for f in range(len(families))]
        self.single = [batched_env.BatchedTrussEnv(n, len(r)) if len(r) else None for n, r in zip(families, self.rows)]
        self.N = self.mix.N

    def pairs(self):
        for r, s in zip(self.rows, self.single):
            if s is not None:
                yield torch.from_numpy(r).to(self.dev), s

    def reset(self):
        self.mix.reset(torch.from_numpy(self.ids).to(self.dev))
        for _, s in self.pairs():
            s.reset()

    def load(self, set_node=None, move_range=None):
        """overwrite the parent state of every environment (numpy [B, ...]) in both batches"""
        for name, v in (("nN_x_n", set_node), ("move_range", move_range)):
            if v is None:
                continue
            getattr(self.mix, name).copy_(torch.from_numpy(np.ascontiguousarray(v)))
            for r, s in self.pairs():
                getattr(s, name).copy_(torch.from_numpy(np.ascontiguousarray(v[r.cpu().numpy()])))

    def step(self, a_geo, a_topo, coin):
        """the same action tensors (torch [B, ...] on the device) for both; returns the in-place clipped copies"""
        per = [(r, s, a_geo[r].clone(), a_topo[r].clone(), coin[r].clone()) for r, s in self.pairs()]
        self.mix.step(a_geo, a_topo, coin)
        for r, s, g, t, c in per:
            s.step(g, t, c)
        torch.cuda.synchronize()
        for r, s, g, t, c in per:
            assert_bits(a_geo[r], g, "clipped a_geo")
            assert_bits(a_topo[r], t, "clipped a_topo")

    def compare(self, tag=""):
        torch.cuda.synchronize()
        for r, s in self.pairs():
            for k in FIELDS:
                assert_bits(getattr(self.mix, k)[r], getattr(s, k), "%s %s %s" % (tag, s.spec.name, k))


def random_ids(rng, F, B):
    ids = rng.randint(0, F, size=B).astype(np.uint8)
    ids[:F] = np.arange(F)                    # every family present
    rng.shuffle(ids)
    return ids


def walk(tw, rng, steps=4):
    B, N, dev = tw.B, tw.N, tw.dev
    for s in range(steps):
        kind = s % 3
        if kind == 0:
            a_geo, a_topo = rng.rand(B, N, 2), rng.rand(B, N, 3)
        elif kind == 1:
            a_geo, a_topo = 0.3 * rng.rand(B, N, 2), 0.3 * rng.rand(B, N, 3)
        else:
            a_geo, a_topo = rng.randn(B, N, 2), rng.randn(B, N, 3)
        coin = (rng.rand(B) >= 0.5).astype(np.uint8)
        tw.step(torch.from_numpy(a_geo.astype(np.float32)).to(dev), torch.from_numpy(a_topo.astype(np.float32)).to(dev),
                torch.from_numpy(coin).to(dev))
        tw.compare("step %d" % s)


@pytest.mark.parametrize("which", ["train", "small", "large"])
def test_reset_and_walk_bit_identical(which):
    from mop_truss_marl_b200.families import TRAIN_FAMILIES
    families = {"train": TRAIN_FAMILIES, "small": ("small_bridge", "small_roof"), "large": ("large_bridge", "large_roof")}[which]
    rng = np.random.RandomState(11)
    tw = Twin(families, random_ids(rng, len(families), 96))
    tw.reset()
    tw.compare("reset")
    assert int(tw.mix.status.abs().max()) == 0
    walk(tw, rng)
    assert int(tw.mix.status.abs().max()) == 0


@pytest.mark.parametrize("families", [("train0_roof", "train3_bridge", "train4_roof"), ("large_roof", "large_bridge")])
def test_adversarial_and_degenerate_bit_identical(families):
    rng = np.random.RandomState(5)
    tw = Twin(families, random_ids(rng, len(families), 64))
    B, N, dev = tw.B, tw.N, tw.dev
    tw.reset()
    for s in range(3):
        acts = [adversarial_actions(rng, N) for _ in range(B)]
        mrs = [adversarial_move_range(rng, N) for _ in range(B)]
        tw.load(move_range=np.stack([np.stack([u, d], axis=-1) for u, d in mrs]).astype(np.float32))
        coin = (rng.rand(B) >= 0.5).astype(np.uint8)
        tw.step(torch.from_numpy(np.stack([a for a, _ in acts])).to(dev), torch.from_numpy(np.stack([t for _, t in acts])).to(dev),
                torch.from_numpy(coin).to(dev))
        tw.compare("adversarial %d" % s)
    # degenerate parent geometry: non-finite heights in a few environments set a status bit (every node: the symmetry
    # copy would replace a single one by its mirror, and supports are pinned to 0)
    tw.reset()
    set_node = tw.mix.nN_x_n.cpu().numpy().copy()
    sick = rng.choice(B, 6, replace=False)
    set_node[sick, :, 1] = np.nan
    tw.load(set_node=set_node)
    tw.step(torch.from_numpy(rng.rand(B, N, 2).astype(np.float32)).to(dev),
            torch.from_numpy(rng.rand(B, N, 3).astype(np.float32)).to(dev), torch.zeros(B, dtype=torch.uint8, device=dev))
    tw.compare("degenerate")
    status = tw.mix.status.cpu().numpy()
    assert (status[sick] != 0).all() and (status[np.setdiff1d(np.arange(B), sick)] == 0).all()


def test_rows_pieces_and_parent_children():
    from mop_truss_marl_b200 import batched_env
    from mop_truss_marl_b200.families import TRAIN_FAMILIES
    rng = np.random.RandomState(2)
    B = 96
    ids = torch.from_numpy(random_ids(rng, 10, B)).cuda()
    one, pieces, parent = (batched_env.MixedTrussEnv(TRAIN_FAMILIES, B) for _ in range(3))
    for e in (one, pieces, parent):
        e.reset(ids)
    child, child_rows = batched_env.MixedTrussEnv(TRAIN_FAMILIES, B), batched_env.MixedTrussEnv(TRAIN_FAMILIES, B)
    for s in range(3):
        a_geo = torch.from_numpy(rng.rand(B, 12, 2).astype(np.float32)).cuda()
        a_topo = torch.from_numpy(rng.rand(B, 12, 3).astype(np.float32)).cuda()
        coin = torch.from_numpy((rng.rand(B) >= 0.5).astype(np.uint8)).cuda()
        acts = [(a_geo.clone(), a_topo.clone()) for _ in range(4)]
        before = {k: getattr(parent, k).clone() for k in FIELDS}
        child.step(*acts[2], coin, parent=parent)
        for lo, hi in ((0, 40), (40, 96)):
            child_rows.step(acts[3][0][lo:hi].contiguous(), acts[3][1][lo:hi].contiguous(), coin[lo:hi].contiguous(),
                            rows=(lo, hi), parent=parent)
        torch.cuda.synchronize()
        for k in FIELDS:                                  # the parent is read, not written
            assert_bits(getattr(parent, k), before[k], "parent " + k)
        one.step(*acts[0], coin)
        for lo, hi in ((0, 32), (32, 72), (72, 96)):
            g, t = acts[1][0][lo:hi].contiguous(), acts[1][1][lo:hi].contiguous()
            pieces.step(g, t, coin[lo:hi].contiguous(), rows=(lo, hi))
        torch.cuda.synchronize()
        assert torch.equal(child.family_ids, ids) and torch.equal(child_rows.family_ids, ids)
        for k in FIELDS:
            assert_bits(getattr(pieces, k), getattr(one, k), "rows= " + k)
            assert_bits(getattr(child, k), getattr(one, k), "parent= " + k)
            assert_bits(getattr(child_rows, k), getattr(one, k), "parent= rows= " + k)
        parent.step(*acts[0], coin)                       # the next parent: same state as `one`
    with pytest.raises(ValueError):
        child.step(a_geo, a_topo, coin, parent=batched_env.BatchedTrussEnv("train0_roof", B))


def test_out_of_range_family_id():
    from mop_truss_marl_b200 import capi
    from mop_truss_marl_b200.families import TRAIN_FAMILIES
    families = TRAIN_FAMILIES[:4]
    rng = np.random.RandomState(9)
    ids = random_ids(rng, 4, 64)
    tw = Twin(families, ids)
    tw.reset()
    bad = np.array([3, 17, 40, 63])
    mix = tw.mix
    bad_ids = torch.from_numpy(ids).cuda()
    bad_ids[torch.from_numpy(bad).cuda()] = torch.tensor([4, 255, 16, 200], dtype=torch.uint8, device="cuda")
    # a reset with bad ids: those environments get the status and keep every output buffer's sentinel
    sentinel = {k: getattr(mix, k) for k in FIELDS if k != "status"}
    for k, t in sentinel.items():
        t.fill_(7)
    mix.reset(bad_ids)
    torch.cuda.synchronize()
    st = mix.status.cpu().numpy()
    assert (st[bad] == capi.STATUS_BAD_FAMILY).all() and (np.delete(st, bad) == 0).all()
    for k, t in sentinel.items():
        assert bool((t[torch.from_numpy(bad).cuda()] == 7).all()), k
    # a step: the same, and the action buffers are not clipped either
    tw.reset()
    mix.family_ids.copy_(bad_ids)                         # as if reset with them; the good environments are reset
    keep = {k: getattr(mix, k)[torch.from_numpy(bad).cuda()].clone() for k in FIELDS if k != "status"}
    B, N = tw.B, tw.N
    a_geo = torch.from_numpy((3 * rng.randn(B, N, 2)).astype(np.float32)).cuda()
    a_topo = torch.from_numpy((3 * rng.randn(B, N, 3)).astype(np.float32)).cuda()
    coin = torch.ones(B, dtype=torch.uint8, device="cuda")
    raw = (a_geo.clone(), a_topo.clone())
    per = [(s, a_geo[r].clone(), a_topo[r].clone(), coin[r].clone()) for r, s in tw.pairs()]
    mix.step(a_geo, a_topo, coin)
    for s, g, t, c in per:
        s.step(g, t, c)
    torch.cuda.synchronize()
    rows = torch.from_numpy(bad).cuda()
    st = mix.status.cpu().numpy()
    assert (st[bad] == capi.STATUS_BAD_FAMILY).all()
    for k, v in keep.items():
        assert_bits(getattr(mix, k)[rows], v, "bad-id env " + k)
    assert_bits(a_geo[rows], raw[0][rows], "bad-id a_geo")
    assert_bits(a_topo[rows], raw[1][rows], "bad-id a_topo")
    # the neighbours are what the single-family batches compute
    good = np.setdiff1d(np.arange(B), bad)
    for f, s in enumerate(tw.single):
        r = np.nonzero(ids[good] == f)[0]
        idx = torch.from_numpy(good[r]).cuda()
        pos = torch.from_numpy(np.searchsorted(tw.rows[f], good[r])).cuda()
        for k in FIELDS:
            assert_bits(getattr(mix, k)[idx], getattr(s, k)[pos], "neighbour %s" % k)


def variants16():
    from mop_truss_marl_b200 import FAMILIES
    out = []
    for k in range(16):
        base = FAMILIES["small_bridge" if k % 2 else "small_roof"]
        out.append(dataclasses.replace(base, name="v%d" % k, tar_y=tuple(t * (1 + 0.03 * k) for t in base.tar_y),
                                       loady=base.loady * (1 + 0.1 * k)))
    return out


def test_family_count_limits_and_two_live_handles():
    from mop_truss_marl_b200 import batched_env, capi
    with pytest.raises(capi.TfemError, match="at most 2 families"):
        batched_env.MixedTrussEnv(("large_bridge", "large_roof", "large_bridge"), 8)
    rng = np.random.RandomState(4)
    big = Twin(variants16(), random_ids(rng, 16, 160))
    small = Twin(variants16()[:2], random_ids(rng, 2, 48))  # created after: must not shrink what `big` launches with
    large = Twin(("large_bridge", "large_roof"), random_ids(rng, 2, 32))
    for tw in (big, small, large):
        tw.reset()
    for s in range(3):
        for tw in (big, small, large, big):
            B, N, dev = tw.B, tw.N, tw.dev
            tw.step(torch.from_numpy(rng.rand(B, N, 2).astype(np.float32)).to(dev),
                    torch.from_numpy(rng.rand(B, N, 3).astype(np.float32)).to(dev),
                    torch.from_numpy((rng.rand(B) >= 0.5).astype(np.uint8)).to(dev))
            tw.compare("interleaved %d" % s)
    assert int(big.mix.status.abs().max()) == 0


def test_single_family_calls_refused_and_rollout_refused():
    from mop_truss_marl_b200 import actor, batched_env, capi, host_pipeline, tf_checkpoint
    from mop_truss_marl_b200.families import TRAIN_FAMILIES
    mix = batched_env.MixedTrussEnv(TRAIN_FAMILIES, 32)
    mix.reset(torch.zeros(32, dtype=torch.uint8, device="cuda"))
    y = torch.zeros(32, 12, dtype=torch.float64, device="cuda")
    sec = torch.zeros(32, 26, dtype=torch.int32, device="cuda")
    with pytest.raises(capi.TfemError, match="tfem_solve_only"):
        mix.solve_only(y, sec)
    with pytest.raises(capi.TfemError, match="tfem_solve_dense_dmma"):
        mix.solve_dense_dmma(y, sec)
    with pytest.raises(capi.TfemError, match="use tfem_step_mixed"):
        mix_single_step(mix)
    pol = actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=3), 12, 32)
    with pytest.raises(capi.TfemError, match="several families"):
        host_pipeline.HostRollout(mix, pol)
    # a single-family handle has no mixed kernel configured
    env = batched_env.BatchedTrussEnv("train0_roof", 4)
    from mop_truss_marl_b200.batched_env import _ptr
    fam = torch.zeros(4, dtype=torch.uint8, device="cuda")
    rc = capi.lib.tfem_reset_mixed(env.handle.ptr, 4, _ptr(fam), _ptr(env.move_range), C.byref(env._out), env._stream())
    assert rc == -1 and b"tfem_create_mixed" in capi.lib.tfem_last_error()


def mix_single_step(mix):
    """the base class's single-family step launch on a mixed batch"""
    from mop_truss_marl_b200 import batched_env, capi
    sin = capi.StepIn()
    for name, t in (("set_node", mix.nN_x_n), ("set_element", mix.nN_x_e), ("move_range", mix.move_range)):
        setattr(sin, name, batched_env._ptr(t))
    g, t = torch.zeros(mix.B, 12, 2, device="cuda"), torch.zeros(mix.B, 12, 3, device="cuda")
    sin.a_geo, sin.a_topo = batched_env._ptr(g), batched_env._ptr(t)
    batched_env.BatchedTrussEnv._launch_step(mix, 0, mix.B, sin, mix._out)


def test_actor_in_the_loop_bit_identical():
    from mop_truss_marl_b200 import actor, tf_checkpoint
    from mop_truss_marl_b200.families import TRAIN_FAMILIES
    rng = np.random.RandomState(21)
    B = 256
    tw = Twin(TRAIN_FAMILIES, random_ids(rng, 10, B))
    tw.reset()
    dev = tw.dev
    pol = actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=20), 12, B, seed=20)
    x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50], device=dev).repeat(B, 1, 1).contiguous()
    A_p = torch.ones(B, 1, 1, device=dev)
    g = torch.Generator(device=dev).manual_seed(0)
    mix = tw.mix
    for s in range(6):
        a_geo, a_topo = pol.act(mix.x_n, mix.A_n, mix.A_s, mix.A_n_ts, mix.A_n_cs, x_p, A_p)
        coin = (torch.rand(B, device=dev, generator=g) >= 0.5).to(torch.uint8)
        tw.step(a_geo, a_topo, coin)
        tw.compare("actor step %d" % s)
    pol.check()
    assert int(mix.status.abs().max()) == 0
