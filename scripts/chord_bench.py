"""Env-step and actor rates for every chord length num_x = 3..16 (DESIGN.md section 3.1): one bridge family per num_x
with 5 m spans (train/code's ENV, no symmetry step), B = 4096 environments.

  fem        the env-step alone, uniform random actions, own state fed back
  act+step   BatchedActor.act (trained agent 1 of 2000pickle_base, OU noise, a one-row Pareto graph) followed by the
             env-step on its actions

Method of bench.py: CUDA events around each step, a 256 MiB L2 flush between steps, warm-up steps first; the two workloads
of one num_x alternate step by step so that clock drift hits them alike.  Each line gives the median step time with its
10th and 90th percentiles, env-steps/s, the algorithmic bytes per env-step of SURVEY.md section 8d with the resulting share
of the HBM roof, the most families a mixed handle of this num_x takes, and the GPU's name, power limit and SM clock read
in the same run.  num_x = 6, 8 and 16 are the shapes of the reference and anchor the new ones.

    python scripts/chord_bench.py --steps 200 --out profiles/r4_chord_lengths.jsonl
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import algorithmic_bytes, trained_actor_weights  # noqa: E402
from mop_truss_marl_b200 import actor, batched_env, capi  # noqa: E402
from mop_truss_marl_b200.families import SYM_NONE, FamilySpec  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]))
    except Exception as exc:                                   # the rates stand without it; say why it is missing
        return {"error": str(exc)[:200]}


def bridge(num_x):
    tar = tuple(1.0 + 2.0 * abs(2 * i - (num_x - 1)) / (num_x - 1) for i in range(num_x))
    return FamilySpec("bridge%d_5m" % num_x, num_x, (5.0,) * (num_x - 1), (5.0,), tar, 0.2, 0, -100000, "bridge", 1, SYM_NONE)


def max_families(spec):
    variants = [dataclasses.replace(spec, name="%s_v%d" % (spec.name, k), loady=spec.loady * (1 + 0.1 * k))
                for k in range(capi.MAX_FAMILIES)]
    try:
        batched_env.MixedTrussEnv(variants, 8)
        return capi.MAX_FAMILIES
    except capi.TfemError as e:
        return int(re.search(r"at most (\d+) families", str(e)).group(1))


def stats(ms, B):
    ms = np.asarray(ms)
    med, p10, p90 = (float(np.percentile(ms, q)) for q in (50, 10, 90))
    return {"ms_median": med, "ms_p10": p10, "ms_p90": p90, "env_steps_per_s": B / (med * 1e-3),
            "env_steps_per_s_p10_p90": [B / (p90 * 1e-3), B / (p10 * 1e-3)]}


def run(num_x, B, steps, warmup, flush, peak_gbs, weights):
    dev = torch.device("cuda:0")
    spec = bridge(num_x)
    env = batched_env.BatchedTrussEnv(spec, B)
    env.reset()
    pol = actor.BatchedActor(weights, env.N, B)
    gen = torch.Generator(device=dev).manual_seed(num_x)
    acts = [(torch.rand(B, env.N, 2, device=dev, generator=gen), torch.rand(B, env.N, 3, device=dev, generator=gen),
             (torch.rand(B, device=dev, generator=gen) >= 0.5).to(torch.uint8)) for _ in range(8)]
    x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50], device=dev).repeat(B, 1, 1).contiguous()
    A_p = torch.ones(B, 1, 1, device=dev)
    geo, topo = torch.empty(B, env.N, 2, device=dev), torch.empty(B, env.N, 3, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    t_fem, t_loop = [], []
    for i in range(warmup + steps):
        a_geo, a_topo, coin = acts[i % 8][0].clone(), acts[i % 8][1].clone(), acts[i % 8][2]   # steps clip in place
        flush.fill_(i & 0xFF)
        ev[0].record()
        env.step(a_geo, a_topo, coin)
        ev[1].record()
        flush.fill_((i + 1) & 0xFF)
        ev[2].record()
        pol.act(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p, out=(geo, topo))
        env.step(geo, topo, coin)
        ev[3].record()
        torch.cuda.synchronize()
        if i >= warmup:
            t_fem.append(ev[0].elapsed_time(ev[1]))
            t_loop.append(ev[2].elapsed_time(ev[3]))
    pol.check()
    bad = int((env.status != 0).sum().item())
    abytes = algorithmic_bytes(env.N, env.E, env.ndof)
    base = {"num_x": num_x, "family": spec.name, "nodes": env.N, "elements": env.E, "free_dofs": env.ndof, "envs": B,
            "timed_steps": steps, "warmup_steps": warmup, "status_nonzero_envs_last_step": bad,
            "mixed_max_families": max_families(spec), "anchor": num_x in (6, 8, 16)}
    fem = stats(t_fem, B)
    fem_gbs = abytes * fem["env_steps_per_s"] / 1e9
    lines = [dict(base, workload="fem", **fem, algorithmic_bytes_per_env_step=abytes, achieved_gbs=fem_gbs,
                  hbm_roof_fraction=fem_gbs / peak_gbs),
             dict(base, workload="act+step", actor="trained 2000pickle_base agent 1, OU noise, 1-row Pareto graph",
                  **stats(t_loop, B))]
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--chords", default="3-16", help="num_x range a-b or a comma list")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("chord_bench.py measures on a CUDA device; none is visible")
    if "-" in args.chords:
        lo, hi = (int(v) for v in args.chords.split("-"))
        chords = list(range(lo, hi + 1))
    else:
        chords = [int(v) for v in args.chords.split(",")]
    weights = trained_actor_weights(1)
    if weights is None:
        raise SystemExit("tests/golden/actor_2000pickle_base.npz is missing")
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    gpu_before = gpu_info()
    lines = []
    for nx in chords:
        lines += run(nx, args.batch, args.steps, args.warmup, flush, peak, weights)
    gpu_after = gpu_info()
    out = open(args.out, "w") if args.out else None
    for line in lines:
        line.update(gpu=gpu_before, gpu_after=gpu_after, hbm_peak_gbs=peak,
                    l2="flushed between timed steps (256 MiB write)")
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
