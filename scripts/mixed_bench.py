"""Mixed-family batches on the GPU: one tfem_step_mixed launch against the same environments grouped by family and
stepped as one tfem_step launch per family (DESIGN.md section 3.1).

Method of bench.py: CUDA events around each step, a 256 MiB L2 flush between steps, 8 + W warm-up steps, K timed steps
per variant; the variants of one measurement run alternately (one step of each per round), so that clock and
neighbour drift hit them alike.  Every variant calls the C ABI with argument structs built once, so the numbers are the
library's and not the Python wrappers'.  The split variant's ten launches read and write row slices of ONE batch (the
best a caller of the single-family API can do: no gather, no copy); the actor then acts on that batch in one launch.

  1. mixed vs split: the ten train families (families.TRAIN_FAMILIES), seeded random ids, B = 4096 and 1024
  2. overhead: an all-one-family batch through a mixed handle of 1 and of F families against tfem_step
  3. closed loop: the 12-node BatchedActor.act + the env-step, mixed vs split

    python scripts/mixed_bench.py --out profiles/r3_mixed_bench.jsonl
"""
from __future__ import annotations

import argparse
import ctypes as C
import dataclasses
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from mop_truss_marl_b200 import actor, batched_env, capi, tf_checkpoint  # noqa: E402
from mop_truss_marl_b200.batched_env import _ptr  # noqa: E402
from mop_truss_marl_b200.families import FAMILIES, TRAIN_FAMILIES, family_desc  # noqa: E402

NACT = 16


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]))
    except Exception as e:  # the timing does not depend on it; say so in the record
        return {"error": repr(e)}


def variants(base, k):
    """k families of base's topology: base itself and k-1 with other targets and loads"""
    b = FAMILIES[base]
    return [b] + [dataclasses.replace(b, name="%s_v%d" % (base, i), tar_y=tuple(t * (1 + 0.03 * i) for t in b.tar_y),
                                      loady=b.loady * (1 + 0.1 * i)) for i in range(1, k)]


class Variant:
    """one way of stepping a batch; step(i) enqueues step i with the i % NACT-th pre-generated action set"""

    def __init__(self, name, env, launches, dev, gen, pol=None):
        self.name, self.env, self.dev, self.pol = name, env, dev, pol
        B, N = env.B, env.N
        self.acts = [(torch.rand(B, N, 2, device=dev, generator=gen), torch.rand(B, N, 3, device=dev, generator=gen),
                      (torch.rand(B, device=dev, generator=gen) >= 0.5).to(torch.uint8)) for _ in range(NACT)]
        if pol is not None:                                  # the actor writes the actions the env-step reads
            buf = (torch.empty(B, N, 2, device=dev), torch.empty(B, N, 3, device=dev))
            self.acts = [(buf[0], buf[1], c) for _, _, c in self.acts]
            self.x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50], device=dev).repeat(B, 1, 1).contiguous()
            self.A_p = torch.ones(B, 1, 1, device=dev)
        self.calls = [launches(env, a) for a in self.acts]

    def step(self, i):
        if self.pol is not None:
            e, (g, t, _) = self.env, self.acts[i % NACT]
            self.pol.act(e.x_n, e.A_n, e.A_s, e.A_n_ts, e.A_n_cs, self.x_p, self.A_p, out=(g, t))
        stream = C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)
        for fn, args in self.calls[i % NACT]:
            capi.check(fn(*args, stream))


def step_in(env, a, lo, hi):
    s = capi.StepIn()
    s.set_node, s.set_element = _ptr(env.nN_x_n[lo:hi]), _ptr(env.nN_x_e[lo:hi])
    s.a_geo, s.a_topo, s.coin = _ptr(a[0][lo:hi]), _ptr(a[1][lo:hi]), _ptr(a[2][lo:hi])
    s.move_range = _ptr(env.move_range[lo:hi])
    return s


def mixed_launches(env, a):
    # byref() keeps its object alive as long as the call list holds it
    return [(capi.lib.tfem_step_mixed, [env.handle.ptr, env.B, _ptr(env.family_ids), C.byref(step_in(env, a, 0, env.B)),
                                        C.byref(env._out)])]


def single_launches(env, a):
    return [(capi.lib.tfem_step, [env.handle.ptr, env.B, C.byref(step_in(env, a, 0, env.B)), C.byref(env._out)])]


def split_launches(handles, bounds):
    def make(env, a):
        calls = []
        for h, (lo, hi) in zip(handles, bounds):
            if hi == lo:
                continue
            calls.append((capi.lib.tfem_step, [h.ptr, hi - lo, C.byref(step_in(env, a, lo, hi)), C.byref(env._make_out(lo, hi))]))
        return calls
    return make


def mixed_env(specs, ids, dev):
    env = batched_env.MixedTrussEnv(specs, len(ids), device=dev)
    env.reset(torch.from_numpy(np.ascontiguousarray(ids, np.uint8)).to(dev))
    return env


def split_env(specs, ids, dev):
    """the batch ordered by family, one single-family handle per family over row slices of it"""
    counts = np.bincount(ids, minlength=len(specs))
    edges = np.concatenate([[0], np.cumsum(counts)])
    env = mixed_env(specs, np.repeat(np.arange(len(specs)), counts), dev)   # allocation + the per-family reset
    index = dev.index if dev.index is not None else 0
    handles = [capi.Handle(family_desc(s), index) for s in specs]
    env._handles = handles
    return env, split_launches(handles, list(zip(edges[:-1], edges[1:])))


def train_ids(rng, B):
    """seeded random family ids with an even count per family: every family's slice of the split layout then starts
    16-byte aligned, which tfem_step requires (an nN_x_e row of the 6 x 2 shapes is 2 184 B)"""
    ids = np.repeat(rng.randint(0, len(TRAIN_FAMILIES), size=B // 2), 2).astype(np.uint8)
    rng.shuffle(ids)
    return ids


def run(label, variants_, K, W, flush, out):
    for i in range(8):                                   # bench.py: the state after 8 steps of i.i.d. actions
        for v in variants_:
            v.step(i)
    for i in range(W):
        for v in variants_:
            flush.fill_(i & 0xFF)
            v.step(i)
    torch.cuda.synchronize()
    ev = {v.name: [] for v in variants_}
    for i in range(K):
        for v in variants_:
            flush.fill_(i & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            v.step(i)
            e1.record()
            ev[v.name].append((e0, e1))
    torch.cuda.synchronize()
    rec = {"measurement": label, "B": variants_[0].env.B, "steps": K, "warmup": 8 + W, "variants": {}}
    for v in variants_:
        ms = np.array([a.elapsed_time(b) for a, b in ev[v.name]])
        rec["variants"][v.name] = {
            "median_us": round(float(np.median(ms)) * 1e3, 2), "p10_us": round(float(np.percentile(ms, 10)) * 1e3, 2),
            "p90_us": round(float(np.percentile(ms, 90)) * 1e3, 2), "min_us": round(float(ms.min()) * 1e3, 2),
            "env_step_launches": len(v.calls[0]),
            "status_bad": int((v.env.status != 0).sum().item())}
    med = {k: r["median_us"] for k, r in rec["variants"].items()}
    base = variants_[0].name
    rec["median_ratio_to_" + base] = {k: round(m / med[base], 4) for k, m in med.items()}
    print(json.dumps(rec), flush=True)
    out.append(rec)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="JSON lines file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mixed_bench.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(args.seed)
    rng = np.random.RandomState(args.seed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    records = [{"gpu_before": gpu_info(), "torch": torch.__version__, "library": capi.lib.tfem_version().decode(),
                "method": "CUDA events around each step, 256 MiB L2 flush between steps, variants alternate step by step"}]
    print(json.dumps(records[0]), flush=True)
    train = [FAMILIES[n] for n in TRAIN_FAMILIES]
    K, W = args.steps, args.warmup

    # 1. mixed vs split, env-step only
    for B in (4096, 1024):
        ids = train_ids(rng, B)
        m = mixed_env(train, ids, dev)
        s, s_launch = split_env(train, ids, dev)
        run("train10 env-step: one tfem_step_mixed vs ten tfem_step", [
            Variant("split_10_launches", s, s_launch, dev, gen), Variant("mixed_1_launch", m, mixed_launches, dev, gen)],
            K, W, flush, records)

    # 2. overhead of the mixed kernel on an all-one-family batch
    for base, B, F in (("train0_roof", 4096, 10), ("small_bridge", 4096, 10), ("large_bridge", 8192, 2)):
        fams = train if base == "train0_roof" else variants(base, F)
        zeros = np.zeros(B, np.uint8)
        one = batched_env.BatchedTrussEnv(base, B, device=dev)
        one.reset()
        run("%s all-one-family: tfem_step vs mixed handles of 1 and %d families" % (base, F), [
            Variant("tfem_step", one, single_launches, dev, gen),
            Variant("mixed_F1", mixed_env(fams[:1], zeros, dev), mixed_launches, dev, gen),
            Variant("mixed_F%d" % F, mixed_env(fams, zeros, dev), mixed_launches, dev, gen)], K, W, flush, records)

    # 3. closed loop: actor + env-step
    weights = tf_checkpoint.random_actor_weights(seed=20)
    for B in (4096, 1024):
        ids = train_ids(rng, B)
        m = mixed_env(train, ids, dev)
        s, s_launch = split_env(train, ids, dev)
        pol_s = actor.BatchedActor(weights, 12, B, device=dev, seed=20)
        pol_m = actor.BatchedActor(weights, 12, B, device=dev, seed=20)
        run("train10 closed loop: BatchedActor.act + env-step, mixed vs split", [
            Variant("split_10_launches", s, s_launch, dev, gen, pol=pol_s),
            Variant("mixed_1_launch", m, mixed_launches, dev, gen, pol=pol_m)], K, W, flush, records)
        pol_s.check()
        pol_m.check()

    records.append({"gpu_after": gpu_info()})
    print(json.dumps(records[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in records:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
