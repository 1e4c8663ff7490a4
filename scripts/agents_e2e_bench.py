"""The driver's three-agent step from a host-resident parent: three one-agent HostRollout.step calls (the parent goes up
three times) against one HostRollout.step_agents call (the parent goes up once), DESIGN.md section 3.2.

Both arms run the same three actors (twins: same weights, seeds and noise parameters) on the same pinned parent with the
same coins, so they compute the same children; the script checks that bit for bit after the timed steps.  The parent is
the same buffer every step, so after two steps both arms replay their captured CUDA graphs.

Method: per step, a device synchronise, a CUDA event on the current stream, the variant's calls (each returns after its
last download has landed), a second event and its synchronise; W warm-up steps per variant, then K timed steps with the
two variants alternating step by step, so that clock and neighbour drift hit them alike.  Medians with p10-p90.

  1. small_bridge, B = 4096, pieces "auto", compact columns (alloc_host())
  2. the same with alloc_host(raw_tables=False)
  3. large_bridge, B = 8192, pieces "auto", compact columns

    python scripts/agents_e2e_bench.py --out profiles/r3_agents_e2e.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from mop_truss_marl_b200 import actor, batched_env, capi, tf_checkpoint  # noqa: E402
from mop_truss_marl_b200.host_pipeline import HostRollout, STATE_IN  # noqa: E402

K_AGENTS = 3


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]))
    except Exception as e:  # the timing does not depend on it; say so in the record
        return {"error": repr(e)}


def stats(ms):
    a = np.asarray(ms)
    return {"median": float(np.median(a)), "p10": float(np.percentile(a, 10)), "p90": float(np.percentile(a, 90))}


def agents(env):
    return [actor.BatchedActor(tf_checkpoint.random_actor_weights(seed=40 + k), env.N, env.B, device=env.device,
                               seed=200 + k, theta=0.1 + 0.05 * k, sigma=0.1 + 0.05 * k) for k in range(K_AGENTS)]


def case(name, family, B, raw_tables, steps, warmup, dev):
    env = batched_env.BatchedTrussEnv(family, B, device=dev)
    env.reset()
    multi = HostRollout(env, agents(env), pieces="auto")
    singles = [HostRollout(env, a, pieces="auto") for a in agents(env)]
    parent = multi.alloc_host(raw_tables=raw_tables)
    for k in STATE_IN:
        if k in parent:
            parent[k].copy_(getattr(env, k))
    parent["node_y"].copy_(env.nN_x_n[:, :, 1])
    parent["element_section"].copy_(env.nN_x_e[:, :, 0])
    torch.cuda.synchronize()
    outs_m = multi.alloc_host_children(raw_tables=raw_tables)
    outs_s = [s.alloc_host(raw_tables=raw_tables) for s in singles]
    g = torch.Generator().manual_seed(1)
    x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50]).repeat(B, 1, 1).contiguous().pin_memory()
    A_p = torch.ones(B, 1, 1).pin_memory()
    coins = [(torch.rand(B, generator=g) >= 0.5).to(torch.uint8).pin_memory() for _ in range(K_AGENTS)]

    def three():
        for k in range(K_AGENTS):
            singles[k].step(parent, coins[k], x_p, A_p, outs_s[k])

    def one():
        multi.step_agents(parent, coins, x_p, A_p, outs_m)

    variants = {"three_step_calls": three, "one_step_agents_call": one}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = {v: [] for v in variants}
    host_ms = {v: [] for v in variants}
    for i in range(warmup + steps):
        for v, fn in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev[0].record()
            fn()
            ev[1].record()
            ev[1].synchronize()
            if i >= warmup:
                ms[v].append(ev[0].elapsed_time(ev[1]))
                host_ms[v].append((time.perf_counter() - t0) * 1e3)
    same = all(torch.equal(outs_m[k][n].view(torch.uint8), outs_s[k][n].view(torch.uint8))
               for k in range(K_AGENTS) for n in outs_m[k])
    up1, down1 = singles[0].bytes_per_step(raw_tables=raw_tables)
    upm, downm = multi.bytes_per_step(raw_tables=raw_tables)
    for p in multi.actors + [s.actor for s in singles]:
        p.check()
    three_s, one_s = stats(ms["three_step_calls"]), stats(ms["one_step_agents_call"])
    return {"case": name, "family": family, "B": B, "pieces": len(multi.ranges), "agents": K_AGENTS,
            "state": "compact columns" + ("" if raw_tables else ", raw_tables=False"),
            "three_step_calls_ms": three_s, "one_step_agents_call_ms": one_s,
            "three_step_calls_host_ms": stats(host_ms["three_step_calls"]),
            "one_step_agents_call_host_ms": stats(host_ms["one_step_agents_call"]),
            "speedup_median": three_s["median"] / one_s["median"],
            "bytes_three_calls": {"h2d": 3 * up1, "d2h": 3 * down1}, "bytes_one_call": {"h2d": upm, "d2h": downm},
            "children_bit_identical": bool(same), "steps": steps, "warmup": warmup}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--out", default=None, help="JSON lines file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("agents_e2e_bench.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    records = [{"gpu_before": gpu_info(), "torch": torch.__version__, "library": capi.lib.tfem_version().decode(),
                "method": "device synchronise, CUDA events around each variant's calls (which end when the last download "
                          "has landed), variants alternate step by step; pinned host buffers, the same parent every step"}]
    print(json.dumps(records[0]), flush=True)
    for name, family, B, raw in (("small_bridge_4096_compact", "small_bridge", 4096, True),
                                 ("small_bridge_4096_no_raw_tables", "small_bridge", 4096, False),
                                 ("large_bridge_8192_compact", "large_bridge", 8192, True)):
        records.append(case(name, family, B, raw, args.steps, args.warmup, dev))
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
