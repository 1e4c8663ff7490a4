"""The training driver's batch from a host-resident parent: one MixedHostRollout over the ten train families against the
best a caller of the one-family rollout can do, ten HostRollouts stepped one after another (DESIGN.md section 3.2).

Workload: the ten families.TRAIN_FAMILIES with seeded random family ids, B = 4096 and B = 1024, three 12-node agents
with OU noise on, pieces "auto", compact columns (alloc_host()).

  mixed        one MixedHostRollout(env, [a0, a1, a2]).step_agents over the whole batch
  per_family   ten HostRollout(BatchedTrussEnv(family f), [a0, a1, a2]), each over its family's contiguous slice of a
               family-sorted pinned state tuple, stepped one after another.  The sort is done once, before the timing.
               Every family's slice starts on a multiple of 16 environments, so that each of its arrays stays
               16-byte aligned, as the transfer kernel of a captured step requires.

The one-agent step (actor a0: MixedHostRollout.step against ten HostRollout.step) is measured the same way.

Method (that of scripts/agents_e2e_bench.py): per step a device synchronise, a CUDA event on the current stream, the
arm's calls (each returns after its last download has landed), a second event and its synchronise; W warm-up steps,
then K timed steps with the four arms alternating step by step, so that clock and neighbour drift hit them alike.  The
parent is the same buffer every step, so every arm replays its captured CUDA graphs.  Medians with p10-p90.

After the timing both arms run again with noise off (the OU noise is keyed per piece, and the arms cut the batch into
different pieces) and the script checks that every environment of every child is bit-identical between them.

    python scripts/mixed_host_bench.py --out profiles/r4_mixed_host.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from mop_truss_marl_b200 import actor, batched_env, capi, tf_checkpoint  # noqa: E402
from mop_truss_marl_b200.families import TRAIN_FAMILIES  # noqa: E402
from mop_truss_marl_b200.host_pipeline import HostRollout, MixedHostRollout, STATE_IN  # noqa: E402
from scripts.agents_e2e_bench import gpu_info, stats  # noqa: E402

K_AGENTS = 3
ALIGN = 16                      # environments: a slice starting on a multiple of 16 keeps every array 16-byte aligned


def agents(env):
    return [actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=40 + k), env.N, env.B, device=env.device,
                               seed=200 + k, theta=0.1 + 0.05 * k, sigma=0.1 + 0.05 * k) for k in range(K_AGENTS)]


def sliced(bufs, lo, hi):
    return {k: v[lo:hi] for k, v in bufs.items()}


def case(B, steps, warmup, dev):
    rng = np.random.RandomState(B)
    ids = rng.randint(0, len(TRAIN_FAMILIES), size=B).astype(np.uint8)
    env = batched_env.MixedTrussEnv(TRAIN_FAMILIES, B, device=dev)
    env.reset(torch.from_numpy(ids).to(dev))
    acts = agents(env)

    # ---- arm A: one mixed rollout ----
    mix3, mix1 = MixedHostRollout(env, acts, pieces="auto"), MixedHostRollout(env, acts[0], pieces="auto")
    parent = mix3.alloc_host()
    for k in STATE_IN:
        parent[k].copy_(getattr(env, k))
    parent["node_y"].copy_(env.nN_x_n[:, :, 1])
    parent["element_section"].copy_(env.nN_x_e[:, :, 0])
    parent["family"].copy_(env.family_ids)
    outs3, out1 = mix3.alloc_host_children(), mix1.alloc_host()
    x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50]).repeat(B, 1, 1).contiguous().pin_memory()
    A_p = torch.ones(B, 1, 1).pin_memory()
    g = torch.Generator().manual_seed(1)
    coins = [(torch.rand(B, generator=g) >= 0.5).to(torch.uint8).pin_memory() for _ in range(K_AGENTS)]
    torch.cuda.synchronize()

    # ---- arm B: the family-sorted copy of the same parent, one rollout pair per family ----
    rows = [np.nonzero(ids == f)[0] for f in range(len(TRAIN_FAMILIES))]
    starts, pos = [], np.empty(B, np.int64)
    top = 0
    for r in rows:
        starts.append(top)
        pos[r] = top + np.arange(len(r))
        top += -(-len(r) // ALIGN) * ALIGN
    Bs = top
    pos_t = torch.from_numpy(pos)
    per3, per1 = [], []
    for f, r in enumerate(rows):
        e = batched_env.BatchedTrussEnv(TRAIN_FAMILIES[f], len(r), device=dev)
        per3.append(HostRollout(e, acts, pieces="auto"))
        per1.append(HostRollout(e, acts[0], pieces="auto"))

    def alloc_sorted():                     # HostRollout.alloc_host at the padded size
        return {k: torch.empty((Bs,) + tuple(v.shape[1:]), dtype=v.dtype).pin_memory() for k, v in parent.items()
                if k != "family"}

    s_parent = alloc_sorted()
    for k, v in s_parent.items():
        v[pos_t] = parent[k]
    s_outs3, s_out1 = [alloc_sorted() for _ in range(K_AGENTS)], alloc_sorted()
    s_xp = torch.empty(Bs, 1, 4).pin_memory()
    s_Ap = torch.empty(Bs, 1, 1).pin_memory()
    s_xp[pos_t], s_Ap[pos_t] = x_p, A_p
    s_coins = [torch.zeros(Bs, dtype=torch.uint8).pin_memory() for _ in range(K_AGENTS)]
    for sc, c in zip(s_coins, coins):
        sc[pos_t] = c
    slices = []
    for f, r in enumerate(rows):
        lo, hi = starts[f], starts[f] + len(r)
        slices.append((sliced(s_parent, lo, hi), [c[lo:hi] for c in s_coins], s_xp[lo:hi], s_Ap[lo:hi],
                       [sliced(o, lo, hi) for o in s_outs3], sliced(s_out1, lo, hi)))

    def mixed_agents():
        mix3.step_agents(parent, coins, x_p, A_p, outs3)

    def per_family_agents():
        for roll, (p, c, xp, Ap, o3, _) in zip(per3, slices):
            roll.step_agents(p, c, xp, Ap, o3)

    def mixed_one():
        mix1.step(parent, coins[0], x_p, A_p, out1)

    def per_family_one():
        for roll, (p, c, xp, Ap, _, o1) in zip(per1, slices):
            roll.step(p, c[0], xp, Ap, o1)

    arms = {"mixed_step_agents": mixed_agents, "per_family_step_agents": per_family_agents,
            "mixed_step": mixed_one, "per_family_step": per_family_one}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = {v: [] for v in arms}
    for i in range(warmup + steps):
        for v, fn in arms.items():
            torch.cuda.synchronize()
            ev[0].record()
            fn()
            ev[1].record()
            ev[1].synchronize()
            if i >= warmup:
                ms[v].append(ev[0].elapsed_time(ev[1]))
    for a in acts:
        a.check()

    # ---- noise off: both arms must give the same children, environment by environment ----
    saved = [(a.theta, a.sigma) for a in acts]
    for a in acts:
        a.theta = a.sigma = 0.0
    same = True
    for _ in range(3):                      # direct, captured, replayed
        for fn in arms.values():
            fn()
        for k in range(K_AGENTS):
            same = same and all(torch.equal(outs3[k][n].view(torch.uint8), s_outs3[k][n][pos_t].view(torch.uint8))
                                for n in s_outs3[k])
        same = same and all(torch.equal(out1[n].view(torch.uint8), s_out1[n][pos_t].view(torch.uint8)) for n in s_out1)
        same = same and all(torch.equal(o["family"], parent["family"]) for o in outs3 + [out1])
    for a, (th, sg) in zip(acts, saved):
        a.theta, a.sigma = th, sg
    status_bad = int((outs3[0]["status"] != 0).sum())

    up_m, down_m = mix3.bytes_per_step()
    per_bytes = [r.bytes_per_step() for r in per3]
    s = {v: stats(ms[v]) for v in arms}
    return {"case": "train10_%d" % B, "families": len(TRAIN_FAMILIES), "B": B, "agents": K_AGENTS,
            "family_sizes": [len(r) for r in rows], "pieces_mixed": len(mix3.ranges),
            "pieces_per_family": [len(r.ranges) for r in per3], "state": "compact columns, OU noise on",
            "ms": s, "speedup_step_agents": s["per_family_step_agents"]["median"] / s["mixed_step_agents"]["median"],
            "speedup_step": s["per_family_step"]["median"] / s["mixed_step"]["median"],
            "bytes_mixed": {"h2d": up_m, "d2h": down_m},
            "bytes_per_family": {"h2d": sum(b[0] for b in per_bytes), "d2h": sum(b[1] for b in per_bytes)},
            "children_bit_identical_noise_off": bool(same), "status_nonzero": status_bad,
            "steps": steps, "warmup": warmup}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--out", default=None, help="JSON lines file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mixed_host_bench.py measures the GPU: no CUDA device")
    if args.steps < 40:
        raise SystemExit("--steps: at least 40 timed steps")
    dev = torch.device("cuda", 0)
    records = [{"gpu_before": gpu_info(), "torch": torch.__version__, "library": capi.lib.tfem_version().decode(),
                "method": "device synchronise, CUDA events around each arm's calls (which end when the last download "
                          "has landed), arms alternate step by step; pinned host buffers, the same parent every step"}]
    print(json.dumps(records[0]), flush=True)
    for B in (4096, 1024):
        records.append(case(B, args.steps, args.warmup, dev))
        print(json.dumps(records[-1]), flush=True)
    records.append({"gpu_after": gpu_info()})
    print(json.dumps(records[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in records:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
