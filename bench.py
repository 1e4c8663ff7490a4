#!/usr/bin/env python
"""Benchmark of the batched truss env-step (BASELINE.json metric: FEM env-steps/sec).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # CPU arm: the oracle port on all host cores

One "step" = one pass of the hot path over one batch: every environment of the batch executes one
``_game_modify``-equivalent (action decode + constraint/symmetry passes + FEM assemble/solve/post +
observation tensors + objective point).  Per-GPU batch is fixed (weak scaling); ranks share nothing.

Timed region (GPU arm): inputs already resident in HBM, one CUDA-event pair per step on the launching
stream, L2 flushed (256 MiB write) between steps because the 52 MB working set would otherwise stay in
the 126 MB L2; value = (envs per step x N GPUs) / mean step time, max over ranks.
e2e: the same step through ``tfem_step_host`` -- pinned HOST state tables + actions in, every float32
tensor the reference returns out (host<->device copies inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "FEM env-steps/sec (batched truss solve)"
UNIT = "env-steps/s"


def algorithmic_bytes(N, E, ndof):
    """SURVEY.md section 8d: everything _game_modify consumes and produces at the reference's dtypes,
    topology constants excluded."""
    inb = 4 * (12 * N + 21 * E + 5 * N)
    outb = 4 * (13 * N + 3 * N * N + 12 * N + 21 * E + 4) + 8 * (ndof + 2 * E + 1)
    return inb + outb


# --------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """polls SM clock / throttle reasons during the timed region (NVML; same fields as the nvidia-smi
    recipe in B200_PROFILING.md)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------------------
def oracle_steps_per_sec(family, seconds, seed=0, with_actor=False):
    """the CPU port driven like the GPU batch (own state fed back; actions from the numpy actor restatement
    with random-init weights + OU noise, or i.i.d. uniform when with_actor is False); returns (steps, elapsed)"""
    from oracle.truss_oracle import TrussOracle
    o = TrussOracle(family)
    rng = np.random.RandomState(seed)
    N = o.mesh.N
    st = o.reset()
    if with_actor:
        from oracle import actor_oracle
        from mop_truss_marl_b200.tf_checkpoint import random_actor_weights
        w = trained_actor_weights(1) or random_actor_weights(seed=20)
        x_p = np.array([[1, 1, 1, 1 / 50]], dtype=np.float32)
        A_p = np.ones((1, 1), dtype=np.float32)

    def actions():
        if not with_actor:
            return rng.rand(N, 2).astype(np.float32), rng.rand(N, 3).astype(np.float32)
        return actor_oracle.act(w, (st["x_n"], o.A_n, st["A_s"], st["A_n_ts"], st["A_n_cs"], x_p, A_p), rng=rng)
    for _ in range(3):
        a_geo, a_topo = actions()
        st = o.step(st["nN_x_n"], st["nN_x_e"], st["max_up"], st["max_down"], a_geo, a_topo, rng.rand() >= 0.5)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        a_geo, a_topo = actions()
        st = o.step(st["nN_x_n"], st["nN_x_e"], st["max_up"], st["max_down"], a_geo, a_topo, rng.rand() >= 0.5)
        n += 1
    return n, time.perf_counter() - t0


def c_oracle_env_steps_per_sec(family, seconds=2.0, B=2048, seed=0):
    """the compiled CPU port (oracle/truss_oracle.c, OpenMP on every host core) stepping B environments in a closed
    loop with i.i.d. uniform actions: transition + FEM + objectives (it does not build the observation tensors, so it
    does LESS work per env-step than the GPU path or the reference).  Returns (env_steps, elapsed, cores)."""
    from oracle.c_oracle import COracle
    co = COracle(family)
    N, E = co.N, co.E
    rng = np.random.RandomState(seed)
    st = co.py.reset()
    set_node = np.repeat(st["nN_x_n"][None], B, axis=0).astype(np.float32)
    set_elem = np.repeat(st["nN_x_e"][None], B, axis=0).astype(np.float32)
    stale = np.repeat(np.stack([st["max_up"], st["max_down"]], axis=-1)[None], B, axis=0).astype(np.float32)
    acts = [(rng.rand(B, N, 2).astype(np.float32), rng.rand(B, N, 3).astype(np.float32),
             (rng.rand(B) >= 0.5).astype(np.uint8)) for _ in range(4)]
    n, t0 = 0, time.perf_counter()
    while True:
        a_geo, a_topo, coin = acts[n % 4]
        out = co.step(set_node, set_elem, a_geo.copy(), a_topo.copy(), coin, stale)
        set_node[:, :, 1] = out["y"].astype(np.float32)
        set_elem[:, :, 0] = out["section"]
        stale = out["move_range"]
        n += 1
        if n >= 2 and time.perf_counter() - t0 >= seconds:
            break
    return n * B, time.perf_counter() - t0, co.threads


def _oracle_worker(args):
    family, seconds, seed, with_actor = args
    import warnings
    warnings.filterwarnings("ignore")
    return oracle_steps_per_sec(family, seconds, seed, with_actor)


def run_reference_arm(args, rank, world):
    """the reference's CPU implementation of the path = the oracle port (the Python reference itself
    cannot travel to the GPU box), one env per process on every host core"""
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    per_step_seconds = max(0.25, min(10.0, 120.0 / max(1, args.steps + args.warmup)))   # whole run ~2 minutes
    if args.ref_step_seconds:
        per_step_seconds = float(args.ref_step_seconds)
    with_actor = not args.no_actor
    ctx = mp.get_context("fork")
    rates = []
    with ctx.Pool(cores) as pool:
        for it in range(args.warmup + args.steps):
            res = pool.map(_oracle_worker, [(args.family, per_step_seconds, 1000 * it + c, with_actor) for c in range(cores)])
            total = sum(n for n, _ in res)
            elapsed = max(t for _, t in res)
            if it >= args.warmup:
                rates.append(total / elapsed)
    value = float(np.mean(rates))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step_seconds * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 (FEM) + f32 (actor)" if with_actor else "f64", "data": "synthetic",
        "config": bench_config(args, max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d processes x %.2f s of oracle env-steps per bench step (one env each, %s, own "
                                   "state fed back)" % (cores, per_step_seconds,
                                                        "numpy actor + OU noise" if with_actor else "uniform actions")},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_name(args):
    if getattr(args, "no_actor", False):
        return "%s B=%d per GPU: batched FEM env-step (_game_modify equivalent), uniform random actions" % (
            args.family, args.batch)
    return "%s B=%d per GPU: actor forward (act, OU noise) + batched FEM env-step (_game_modify equivalent)" % (
        args.family, args.batch)


def cpu_baselines(args):
    """(cpu_baseline, cpu_baseline_c_env_step) of the JSON line: the Python oracle port on one core (numpy actor + env-step)
    and the C port of the env-step on every host core, each on a bounded sample"""
    use_actor = not args.no_actor
    n_cpu, t_cpu = oracle_steps_per_sec(args.family, args.cpu_seconds, with_actor=use_actor)
    factor = ""
    fpath = os.path.join(ROOT, "profiles", "r2_port_vs_reference.json")
    if os.path.exists(fpath):
        try:
            f = json.load(open(fpath)).get(args.family)
            if f:
                factor = ("; the port runs %.2fx the steps/s of the reference's own _game_modify loop (measured once in the "
                          "build container, scripts/port_vs_reference.py: %.0f vs %.0f env-steps/s on one core, env-step only)"
                          % (f["port_over_reference"], f["port_steps_per_s"], f["reference_steps_per_s"]))
        except Exception:
            pass
    cpu_line = {"value": n_cpu / t_cpu, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": "%d oracle steps (%s) of %s in %.1f s, one process%s" % (
                    n_cpu, "numpy actor + env-step" if use_actor else "env-step", args.family, t_cpu, factor)}
    try:
        nc, tc, cores_c = c_oracle_env_steps_per_sec(args.family, seconds=min(3.0, max(0.3, args.cpu_seconds / 4)))
        c_line = {"value": nc / tc, "unit": UNIT, "cores": cores_c, "kind": "port",
                  "sample": "%d env-steps of %s in %.2f s: oracle/truss_oracle.c (C, OpenMP), FEM env-step only "
                            "(transition + solve + objectives, no observation tensors, no actor)" % (nc, args.family, tc)}
    except Exception as exc:                          # no gcc on the box: the Python port above is the baseline
        c_line = {"unavailable": str(exc)[:200]}
    return cpu_line, c_line


def family_dims(family):
    """(nodes, elements, free dofs) of a family from the oracle's mesh tables (no GPU needed: both arms print them)"""
    from oracle.truss_oracle import FAMILIES, build_mesh
    m = build_mesh(FAMILIES[family])
    return int(m.N), int(m.E), int(m.ndof)


def trained_actor_weights(agent):
    """the reference's trained checkpoint model/2000pickle_base/Agent<agent>_Actor_pickle, from the committed fixture
    tests/golden/actor_2000pickle_base.npz (tests/golden/make_actor_golden.py); None when the fixture is absent"""
    from mop_truss_marl_b200.tf_checkpoint import ACTOR_LAYERS
    path = os.path.join(ROOT, "tests", "golden", "actor_2000pickle_base.npz")
    if not os.path.exists(path):
        return None
    z = np.load(path)
    return {name: (z["agent%d/%s/kernel" % (agent, name)], z["agent%d/%s/bias" % (agent, name)]) for name in ACTOR_LAYERS}


def bench_config(args, world):
    """the `config` object of the JSON line: identical for the B200 arm and the reference arm"""
    N, E, ndof = family_dims(args.family)
    use_actor = not args.no_actor
    trained = use_actor and trained_actor_weights(1) is not None
    return {"workload": workload_name(args), "family": args.family, "envs_per_gpu": args.batch,
            "nodes": N, "elements": E, "free_dofs": ndof,
            "l2": "not flushed" if args.no_flush else "flushed between timed steps (256 MiB write; B200 arm only: the CPU arm has no such cache to flush)",
            "actions": (("actor outputs (trained 2000pickle_base checkpoint, agent 1 + rank % 3)" if trained else
                         "actor outputs (random-init weights of the reference architecture)") + " + OU noise"
                        if use_actor else "uniform [0,1) float32") + ", coin Bernoulli(1/2), own state fed back",
            "parallelism": "env-parallel, %d independent shard(s), no collective" % world}


def actor_flops(N, P=1, H=200):
    """multiply-adds x2 of one actor forward for one environment (GEMMs + adjacency products)"""
    gemm = 3 * N * 13 * H + P * 4 * H + 7 * N * H * H + N * H * 5
    adj = 10 * N * N * H + P * P * H + 2 * N * N * 5
    return 2 * (gemm + adj)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def last_step_outputs(env, actions):
    """what a caller of the timed path holds after its last step: the actor's actions (when the actor drives the step;
    the env-step clips them in place) and every output of the env-step, as float32 / float64 numpy arrays.  A batch whose
    arrays exceed DUMP_LIMIT_BYTES is cut to a fixed sample of environments (seed 0, sorted), the same for every run with
    the same --batch."""
    import torch
    names = ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "move_range", "point", "status") + \
        (("y", "y_weak") + env.FP64_FIELDS if env.fp64_outputs else ())
    tensors = dict(zip(("a_geo", "a_topo"), actions or ()))
    tensors.update((k, getattr(env, k)) for k in names)
    per_env = sum(t[0].numel() * (8 if t.dtype == torch.float64 else 4) for t in tensors.values())
    keep = min(env.B, (DUMP_LIMIT_BYTES - 4096 * len(tensors)) // per_env)
    rows = None
    if keep < env.B:
        rows = torch.from_numpy(np.sort(np.random.RandomState(0).choice(env.B, keep, replace=False))).to(env.device)
    out = {}
    for k, t in tensors.items():
        t = t if rows is None else t.index_select(0, rows)
        out[k] = t.to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu().numpy()
    return out


def _max_over_ranks(ms, dev, world):
    if world > 1:
        import torch
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def e2e_piece_schedule(spec, B):
    """--e2e-pieces: "3" -> 3 equal pieces; "512,1536,2048" -> those sizes; "0.125,0.375,0.5" -> fractions of B rounded to 32"""
    if str(spec) == "auto":
        return "auto"
    parts = [p for p in str(spec).split(",") if p]
    if len(parts) == 1 and "." not in parts[0]:
        return int(parts[0])
    vals = [float(p) for p in parts]
    if all(v < 1 for v in vals):
        sizes = [max(32, int(round(v * B / 32)) * 32) for v in vals[:-1]]
        sizes.append(B - sum(sizes))
    else:
        sizes = [int(v) for v in vals]
    if min(sizes) <= 0 or sum(sizes) != B:
        raise SystemExit("--e2e-pieces %s does not add up to the batch %d" % (spec, B))
    return sizes


def fem_leg(family, B, rank, world, dev, flush, what, steps=50, warmup=5):
    """FEM env-step alone (resident uniform actions, own state fed back) at one of BASELINE.json's named shapes"""
    import torch
    import torch.distributed as dist
    from mop_truss_marl_b200 import batched_env
    env = batched_env.BatchedTrussEnv(family, B, device=dev, fp64_outputs=True)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    acts = [(torch.rand(B, env.N, 2, device=dev, generator=gen), torch.rand(B, env.N, 3, device=dev, generator=gen),
             (torch.rand(B, device=dev, generator=gen) >= 0.5).to(torch.uint8)) for _ in range(8)]
    for i in range(8 + warmup):
        env.step(acts[i % 8][0].clone(), acts[i % 8][1].clone(), acts[i % 8][2])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    total = 0.0
    for i in range(steps):
        a_geo, a_topo = acts[i % 8][0].clone(), acts[i % 8][1].clone()     # the step clips its actions in place
        if flush is not None:
            flush.fill_(i & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.step(a_geo, a_topo, acts[i % 8][2])
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    ms = _max_over_ranks(total / steps, dev, world)
    bad = int((env.status != 0).sum().item())
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
    abytes = algorithmic_bytes(env.N, env.E, env.ndof)
    return {"workload": what, "family": family, "envs_per_gpu": B, "n_gpus": world, "value": B * world / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms, "scaling": "strong" if family == "small_roof" else "weak",
            "roofline_fem": {"bound": "hbm", "achieved": abytes * B / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": abytes * B / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_env": abytes},
            "status_nonzero_envs": bad}


def actor_leg(env, pol, P, dev, flush, world, steps=30, warmup=5):
    """the actor stage alone with a Pareto graph of P rows (a chain graph over a full front, truss2D_ENV.py:22-41)"""
    import torch
    from mop_truss_marl_b200.pareto_graph import chain_graph
    B, N = env.B, env.N
    x_p_np, A_p_np = chain_graph(P)
    x_p = torch.from_numpy(x_p_np).to(dev).repeat(B, 1, 1).contiguous()
    A_p = torch.from_numpy(A_p_np).to(dev).repeat(B, 1, 1).contiguous()
    geo, topo = torch.empty(B, N, 2, device=dev), torch.empty(B, N, 3, device=dev)
    for _ in range(warmup):
        pol.act(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p, out=(geo, topo))
    torch.cuda.synchronize()
    total = 0.0
    for i in range(steps):
        if flush is not None:
            flush.fill_(i & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pol.act(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p, out=(geo, topo))
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    pol.check()
    ms = _max_over_ranks(total / steps, dev, world)
    return {"workload": "actor stage (Pareto branch + fused network + OU noise) with a %d-row Pareto graph" % P, "P": P,
            "envs_per_gpu": B, "actor_ms": ms, "actor_forwards_per_s": B * world / (ms * 1e-3)}


def train_leg(args, rank, local_rank, world, dev, steps=10, standalone=False, family="large_roof", B=1024, P=50):
    """BASELINE.json configs[4]: the multi-agent DDPG training loop on the large roof -- per step the three agents' CUDA
    actors act on the batch's parent state, the three child states are evaluated by three env-steps, a slice of the
    transitions enters the device-resident replay, and one MADDPG.train() + update() follows (one update per game step,
    train/code/master_DDPG_truss2D_MO.py:647-649) with the gradients of every model averaged over the ranks by one
    flat-buffer NCCL all-reduce each (learner.allreduce_flat); the updated actors are pushed into the CUDA actor handles.
    Rewards are synthetic (minus the child's two objectives and their sum): the driver's Pareto / hypervolume reward is outside
    the hot path."""
    import torch
    import torch.distributed as dist
    from mop_truss_marl_b200 import actor as actor_mod
    from mop_truss_marl_b200 import batched_env, learner as learner_mod
    from mop_truss_marl_b200.pareto_graph import chain_graph
    parent = batched_env.BatchedTrussEnv(family, B, device=dev, fp64_outputs=False)
    parent.reset()
    children = [batched_env.BatchedTrussEnv(family, B, device=dev, fp64_outputs=False) for _ in range(3)]
    N = parent.N
    lrn = learner_mod.MADDPGLearner(lr=1e-7, batch_size=32, device=dev, seed=20)       # same seed on every rank: identical models
    lrn.keep_losses_on_device = True
    lrn.device_replay = learner_mod.DeviceReplay(4096, N, P, dev, seed=1000 + rank)     # each rank holds its own replay shard
    for k in range(3):
        w = trained_actor_weights(k + 1)
        if w is not None:
            lrn.agents[k].actor.import_weights(w)
        lrn.agents[k].update_init()
    pols = [actor_mod.BatchedActor(lrn.actor_weights(k), N, B, device=dev, seed=20 + 1000 * rank + k) for k in range(3)]
    x_p_np, A_p_np = chain_graph(P)
    x_p = torch.from_numpy(x_p_np).to(dev).repeat(B, 1, 1).contiguous()
    A_p = torch.from_numpy(A_p_np).to(dev).repeat(B, 1, 1).contiguous()
    gen = torch.Generator(device=dev).manual_seed(7 + rank)
    keep = torch.arange(0, B, B // 64, device=dev)[:64]                                   # 64 transitions per step enter the replay
    acts = [(torch.empty(B, N, 2, device=dev), torch.empty(B, N, 3, device=dev)) for _ in range(3)]
    ev = lambda: torch.cuda.Event(enable_timing=True)                                    # noqa: E731
    use_graph = not getattr(args, "train_eager", False)

    def state_of(e):
        return {"x_n": e.x_n, "A_n": e.A_n, "A_s": e.A_s, "A_n_ts": e.A_n_ts, "A_n_cs": e.A_n_cs, "x_p": x_p, "A_p": A_p}

    def one_step(timed):
        t = [ev() for _ in range(5)] if timed else None
        if timed:
            t[0].record()
        coin = (torch.rand(B, device=dev, generator=gen) >= 0.5).to(torch.uint8)
        for k in range(3):
            pols[k].act(parent.x_n, parent.A_n, parent.A_s, parent.A_n_ts, parent.A_n_cs, x_p, A_p, out=acts[k])
            children[k].step(acts[k][0], acts[k][1], coin, parent=parent)
        if timed:
            t[1].record()
        rewards = torch.stack([-children[0].point[:, 0], -children[1].point[:, 1],
                               -(children[2].point[:, 0] + children[2].point[:, 1])], dim=1)
        lrn.device_replay.push(state_of(parent), acts, rewards, [state_of(c) for c in children], 0.0, rows=keep)
        if timed:
            t[2].record()
        trained = lrn.train()
        lrn.update()
        if timed:
            t[3].record()
        if trained:
            for k in range(3):
                pols[k].set_weights_device(lrn.actor_tensors(k))       # weight images rebuilt on the device
        # the game moves on along agent 0's child (the driver keeps a front of candidates; one parent per environment here)
        for name in ("x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "move_range", "point"):
            getattr(parent, name).copy_(getattr(children[0], name))
        if timed:
            t[4].record()
        return t
    for _ in range(3):
        one_step(False)
    if use_graph:
        lrn.capture_graph()          # one MADDPG.train() = one cudaGraphLaunch from here on (the all-reduces are graph nodes)
        for _ in range(2):
            one_step(False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    # elements one update all-reduces (six flat buffers: three critics, three actors)
    sizes = [sum(p.numel() for p in m.parameters()) for a in lrn.agents for m in (a.critic, a.actor)]
    t0 = time.perf_counter()
    stamps = [one_step(True) for _ in range(steps)]
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3 / steps
    seg = lambda a, b: float(np.mean([s[a].elapsed_time(s[b]) for s in stamps]))       # noqa: E731
    # the six all-reduces of one update, timed on their own (inside the update they are nodes of the captured graph)
    ar_ms = 0.0
    if world > 1:
        bufs = [torch.zeros(n, device=dev) for n in sizes]
        for rep_ in range(12):
            e0, e1 = ev(), ev()
            e0.record()
            for b_ in bufs:
                dist.all_reduce(b_)
            e1.record()
            torch.cuda.synchronize()
            if rep_ >= 2:
                ar_ms += e0.elapsed_time(e1) / 10
    step_ms = _max_over_ranks(wall_ms, dev, world)
    for p_ in pols:
        p_.check()
    # every rank must hold the same models after the same all-reduced updates
    chk = torch.cat([p.detach().reshape(-1) for p in lrn.agents[0].actor.parameters()]).double().sum()
    same = True
    if world > 1:
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same = bool(lo.item() == hi.item())
    line = {
        "workload": "%s B=%d per GPU: three-agent DDPG training loop (3 x actor act + 3 x FEM env-step, device replay, "
                    "MADDPG train + update per game step, gradient all-reduce, actor weight images rebuilt on the device)" % (family, B),
        "family": family, "envs_per_gpu": B, "n_gpus": world, "steps": steps,
        "value": 3 * B * world / (step_ms * 1e-3), "unit": UNIT, "ms_per_step": step_ms,
        "updates_per_s": 1e3 / step_ms, "replay_transitions_per_step": int(keep.numel()), "learner_batch": lrn.batch_size,
        "stages_ms": {"rollout_3x_act_3x_env_step": seg(0, 1), "replay_push": seg(1, 2), "learner_train_update": seg(2, 3),
                      "weight_push_and_state_advance": seg(3, 4)},
        "learner_update": "one captured CUDA graph per MADDPG.train()" if use_graph else "eager PyTorch",
        "all_reduce": {"backend": dist.get_backend() if world > 1 else None, "ranks": world,
                       "calls_per_step": 6 if world > 1 else 0,
                       "bytes_per_step": 4 * sum(sizes) if world > 1 else 0,
                       "ms_per_step_standalone": ar_ms, "share_of_step": ar_ms / step_ms},
        "models_identical_across_ranks": same,
        "rewards": "synthetic (minus the child's objectives)", "data": "synthetic",
    }
    if standalone:
        line = {"metric": METRIC + ", training loop", "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64 (FEM) + f32 (actor, learner)", **line}
    return line


# --------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--family", default="small_bridge")
    ap.add_argument("--batch", type=int, default=4096, help="environments per GPU")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-step-seconds", type=float, default=0.0, help="--impl reference: CPU seconds per bench step (default: sized for a ~2 minute run)")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--e2e-pieces", type=str, default="auto",
                    help="end-to-end path: 'auto' (HostRollout's choice: ~5.7 MB of download per piece), the number of equal "
                         "pieces the batch is cut into, or a comma list of piece sizes (fractions of the batch if below 1)")
    ap.add_argument("--no-actor", action="store_true", help="drive the env with resident uniform actions instead of the actor")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra legs (BASELINE configs 3 and 4 shapes, actor at P = 50, training leg)")
    ap.add_argument("--train", action="store_true", help="only the training loop of BASELINE config 5 (large roof, MADDPG update with gradient all-reduce)")
    ap.add_argument("--train-steps", type=int, default=0, help="timed steps of the training leg (default: 10, or --steps with --train)")
    ap.add_argument("--train-eager", action="store_true", help="training leg: run the learner update eagerly instead of as a captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (actions, state tensors, point, status, "
                         "float64 FEM fields) as DIR/<name>.npy, float32 or float64, at most 64 MB in all (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.train or args.impl != "b200"):
        ap.error("--dump-outputs writes the outputs of the B200 env-step path; it does not apply to --train or --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    from mop_truss_marl_b200 import actor as actor_mod
    from mop_truss_marl_b200 import batched_env, capi, tf_checkpoint

    # the CPU baselines run on rank 0 BEFORE the process group exists: the other ranks wait in the TCP rendezvous of
    # init_process_group, not in an NCCL barrier that would keep their GPUs spinning for the 15 s this takes
    cpu_lines = cpu_baselines(args) if (rank == 0 and not args.train) else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(minutes=20))
    if args.train:
        line = train_leg(args, rank, local_rank, world, dev, steps=args.train_steps or args.steps, standalone=True)
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    B, K, W = args.batch, args.steps, max(3, args.warmup)
    env = batched_env.BatchedTrussEnv(args.family, B, device=dev)
    N, E = env.N, env.E
    gen = torch.Generator(device=dev).manual_seed(rank)
    env.reset()
    nact = 16                                   # pre-generated, resident action batches, cycled

    def make_actions():
        return (torch.rand(B, N, 2, device=dev, generator=gen), torch.rand(B, N, 3, device=dev, generator=gen),
                (torch.rand(B, device=dev, generator=gen) >= 0.5).to(torch.uint8))
    acts = [make_actions() for _ in range(nact)]
    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    use_actor = not args.no_actor
    if use_actor:
        # random-init weights of the reference architecture (no checkpoint travels to the GPU box); the
        # Pareto-front graph is the reset-time one-node graph of _game_get_1_state (truss2D_ENV.py:346-352)
        # the trained checkpoint when its fixture travelled with the repository, else random-init weights of the
        # reference architecture; OU-noise seeds differ per rank (the noise field is a function of seed and call index)
        weights = trained_actor_weights(1 + rank % 3) or tf_checkpoint.random_actor_weights(seed=20 + rank)
        pol = actor_mod.BatchedActor(weights, N, B, device=dev, seed=20 + 1000 * rank)
        x_p = torch.tensor([1.0, 1.0, 1.0, 1.0 / 50], device=dev).repeat(B, 1, 1).contiguous()
        A_p = torch.ones(B, 1, 1, device=dev)
        a_geo_buf = torch.empty(B, N, 2, device=dev)
        a_topo_buf = torch.empty(B, N, 3, device=dev)
    stage_ev = []

    def one_step(i, timed=False):
        if use_actor:
            if timed:
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record()
            pol.act(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p, out=(a_geo_buf, a_topo_buf))
            if timed:
                e1.record()
            env.step(a_geo_buf, a_topo_buf, acts[i % nact][2])
            if timed:
                e2.record()
                stage_ev.append((e0, e1, e2))
        else:
            a_geo, a_topo, coin = acts[i % nact]
            env.step(a_geo, a_topo, coin)

    for i in range(8):                          # SURVEY 8d: state after w = 8 warm-up steps of i.i.d. actions
        one_step(i)
    for i in range(W):
        if flush is not None:
            flush.fill_(i & 0xFF)
        one_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = env.launch_count() + (pol.launch_count() if use_actor else 0)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    torch.cuda.synchronize()
    for i in range(K):
        if flush is not None:
            flush.fill_(i & 0xFF)
        starts[i].record()
        one_step(i, timed=True)
        ends[i].record()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:                 # before the e2e legs below step `env` again
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in last_step_outputs(env, (a_geo_buf, a_topo_buf) if use_actor else None).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    launches = env.launch_count() + (pol.launch_count() if use_actor else 0) - launches0
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    total_ms = float(sum(step_ms))
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / K
    value = B * world / (ms_per_step * 1e-3)
    status_bad = int((env.status != 0).sum().item())

    # ---- e2e: HOST buffers in, HOST buffers out, copies inside the timed region ----------------------------
    f32_out = (("x_n", (B, N, 13)), ("A_s", (B, N, N)), ("A_n_ts", (B, N, N)), ("A_n_cs", (B, N, N)),
               ("nN_x_n", (B, N, 12)), ("nN_x_e", (B, E, 21)), ("point", (B, 4)))
    out_host = {k: torch.empty(sh, dtype=torch.float32).pin_memory() for k, sh in f32_out}
    out_host["status"] = torch.zeros(B, dtype=torch.int32).pin_memory()
    coin_host = (torch.rand(B) >= 0.5).to(torch.uint8).pin_memory()
    if use_actor:
        # the caller holds the state tuple on the host (like the reference driver); per step it goes to the
        # device, the actor acts on it, the env steps, and the new state tuple + actions come back
        from mop_truss_marl_b200.host_pipeline import HostRollout, STATE_IN
        roll = HostRollout(env, pol, pieces=e2e_piece_schedule(args.e2e_pieces, B))
        bufs = [roll.alloc_host(), roll.alloc_host()]
        for k in STATE_IN:
            bufs[0][k].copy_(getattr(env, k))
        torch.cuda.synchronize()
        HostRollout.fill_compact(bufs[0])                   # the two live table columns travel as compact arrays
        x_p_host, A_p_host = x_p.cpu().pin_memory(), A_p.cpu().pin_memory()
        torch.cuda.synchronize()
        flip = [0]

        def e2e_step():
            src, dst = bufs[flip[0]], bufs[1 - flip[0]]
            roll.step(src, coin_host, x_p_host, A_p_host, dst)  # returned state tuple = next step's input
            flip[0] = 1 - flip[0]
        h2d, d2h = roll.bytes_per_step()
        e2e_path = ("pinned host state tuple + Pareto graph -> device -> tactor_act + tfem_step -> host (state tuple, point, "
                    "status, actions); trollout_step_host (host_pipeline.HostRollout), %d pieces on 3 streams, %s" % (
                        len(roll.ranges), "copy engines" if os.environ.get("TROLLOUT_ZEROCOPY", "1") == "0" else
                        "one transfer kernel per piece and direction reading / writing the mapped pinned host arrays"))
    else:
        host = {
            "set_node": env.nN_x_n.cpu().pin_memory(), "set_element": env.nN_x_e.cpu().pin_memory(),
            "move_range": env.move_range.cpu().pin_memory(),
            "a_geo": torch.rand(B, N, 2).pin_memory(), "a_topo": torch.rand(B, N, 3).pin_memory(),
        }
        out_np = {k: v.numpy() for k, v in out_host.items()}
        a_geo0, a_topo0 = host["a_geo"].clone(), host["a_topo"].clone()

        def e2e_step():
            host["a_geo"].copy_(a_geo0); host["a_topo"].copy_(a_topo0)      # fresh (unclipped) actions each step
            batched_env.step_host(env.handle, host["set_node"].numpy(), host["set_element"].numpy(),
                                  host["move_range"].numpy(), host["a_geo"].numpy(), host["a_topo"].numpy(),
                                  coin_host.numpy(), want_fp64=False, out=out_np)
            host["set_node"].copy_(out_host["nN_x_n"]); host["set_element"].copy_(out_host["nN_x_e"])
        h2d = sum(v.numel() * v.element_size() for v in host.values()) + B
        d2h = sum(v.numel() * v.element_size() for v in out_host.values()) + sum(
            host[k].numel() * host[k].element_size() for k in ("a_geo", "a_topo", "move_range"))
        e2e_path = "tfem_step_host: pinned host state tables + actions in, all float32 tensors out"
    ke = max(5, min(K, 50))
    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(ke):
        e2e_step()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / ke
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    # ---- e2e with the raw tables travelling as their live columns in BOTH directions (extra key, next to `e2e`) -----------
    e2e_compact = None
    if use_actor:
        cb = [roll.alloc_host(raw_tables=False), roll.alloc_host(raw_tables=False)]
        for k in cb[0]:
            if k in bufs[flip[0]]:
                cb[0][k].copy_(bufs[flip[0]][k])
        cflip = [0]

        def compact_step():
            roll.step(cb[cflip[0]], coin_host, x_p_host, A_p_host, cb[1 - cflip[0]])
            cflip[0] = 1 - cflip[0]
        for _ in range(3):
            compact_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            compact_step()
        torch.cuda.synchronize()
        c_ms = _max_over_ranks((time.perf_counter() - t0) * 1e3 / ke, dev, world)
        ch2d, cd2h = roll.bytes_per_step(raw_tables=False)
        e2e_compact = {"value": B * world / (c_ms * 1e-3), "unit": UNIT, "ms_per_step": c_ms, "h2d_bytes_per_step": ch2d,
                       "d2h_bytes_per_step": cd2h,
                       "path": "as `e2e`, but the host state tuple carries nN_x_n / nN_x_e as the one column of each that "
                               "_game_modify / _set_model read (node_y [B,N], element_section [B,E]) in both directions; "
                               "HostRollout.alloc_host(raw_tables=False)"}
    # ---- e2e, resident state: what a batched driver does when the state tuple lives with the environment object (as it
    # does inside the reference's own Game / gen_model objects): per step the host sends the coins and the Pareto-front
    # graph and receives point + status; only the states it wants to archive would be fetched (not timed here).  Reported
    # next to `e2e`, never instead of it.
    e2e_res = None
    if use_actor:
        point_h = torch.empty(B, 4).pin_memory()
        status_h = torch.empty(B, dtype=torch.int32).pin_memory()
        coin_d = torch.empty(B, dtype=torch.uint8, device=dev)
        x_p_d, A_p_d = torch.empty_like(x_p), torch.empty_like(A_p)

        def resident_step():
            coin_d.copy_(coin_host, non_blocking=True)
            x_p_d.copy_(x_p_host, non_blocking=True)
            A_p_d.copy_(A_p_host, non_blocking=True)
            a_geo, a_topo = pol.act(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p_d, A_p_d)
            env.step(a_geo, a_topo, coin_d)
            point_h.copy_(env.point, non_blocking=True)
            status_h.copy_(env.status, non_blocking=True)
            torch.cuda.current_stream().synchronize()          # the driver reads point / status before the next step
        for _ in range(3):
            resident_step()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            resident_step()
        res_ms = (time.perf_counter() - t0) * 1e3 / ke
        if world > 1:
            t = torch.tensor([res_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res_ms = float(t.item())
        e2e_res = {"value": B * world / (res_ms * 1e-3), "unit": UNIT, "ms_per_step": res_ms,
                   "h2d_bytes_per_step": int(B + x_p_host.numel() * 4 + A_p_host.numel() * 4),
                   "d2h_bytes_per_step": int(B * 16 + B * 4),
                   "path": "state tuple resident in HBM (BatchedTrussEnv); per step: pinned coins + Pareto graph -> device, "
                           "BatchedActor.act + BatchedTrussEnv.step, point + status -> pinned host, stream sync"}
    clocks = sampler.result()
    extra = None
    if not args.no_extras:
        # the shapes BASELINE.json configs 3 and 4 name, FEM env-step only, and the actor with a full Pareto graph
        extra = {
            "config3": fem_leg("small_roof", max(1, 16384 // world), rank, world, dev, flush,
                               "small roof, 16384 environments in TOTAL split over the ranks (strong scaling)"),
            "config4": fem_leg("large_bridge", 1024, rank, world, dev, flush,
                               "large bridge, 1024 environments per GPU (8192 across 8)"),
        }
        if use_actor:
            extra["actor_pareto_P50"] = actor_leg(env, pol, 50, dev, flush, world)
        if world == 8:
            extra["config5"] = train_leg(args, rank, local_rank, world, dev, steps=args.train_steps or 10, standalone=False)

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else {}
        abytes = algorithmic_bytes(N, E, env.ndof)
        if use_actor:
            actor_ms = float(np.mean([e0.elapsed_time(e1) for e0, e1, _ in stage_ev]))
            fem_ms = float(np.mean([e1.elapsed_time(e2) for _, e1, e2 in stage_ev]))
        else:
            actor_ms, fem_ms = 0.0, float(np.mean(step_ms))
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("%s_B%d" % (args.family, B))
        fem_achieved = abytes * B / (fem_ms * 1e-3) / 1e9
        roof_fem = {"bound": "hbm", "achieved": fem_achieved, "peak": peak, "unit": "GB/s", "frac": fem_achieved / peak,
                    "traffic": traffic, "peak_source": peak_src, "kernel": "tfem_step_kernel (1 launch per step)",
                    "algorithmic_bytes_per_env": abytes, "kernel_ms": fem_ms}
        stages = {"actor_ms": actor_ms, "fem_ms": fem_ms,
                  "fem_only_env_steps_per_s": B * world / (fem_ms * 1e-3)}
        if use_actor and actor_ms > fem_ms:
            # dominant stage = actor_pipe_kernel (tcgen05 kind::f16 with the fp16 hi/lo split = float32-equivalent
            # accuracy, three MMAs per product).  achieved counts ALGORITHMIC flops (one multiply-add per
            # product) against the measured bf16 cuBLAS roof; fp16 runs at the bf16 rate and the split costs 3x,
            # so 1/3 of that roof is the ceiling of this formulation.
            tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
            aflops = actor_flops(N) * B
            ach = aflops / (actor_ms * 1e-3) / 1e12
            roofline = {"bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak,
                        "traffic": (json.load(open(tpath)).get("actor_%s_B%d" % (args.family, B))
                                    if os.path.exists(tpath) else None),
                        "kernel": "actor_pipe_kernel (kernel_ms is the whole actor stage: + Pareto embedding and the two "
                                  "OU-noise launches, about 3 % of it)",
                        "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback",
                        "algorithmic_flops_per_env": actor_flops(N), "kernel_ms": actor_ms,
                        "note": "tcgen05 kind::f16, fp16 hi/lo split = 3 MMAs per product (float32-equivalent); algorithmic "
                                "flops vs the bf16 tensor roof (formulation ceiling = roof/3)"}
        else:
            roofline = roof_fem
        cpu_line, c_line = cpu_lines
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 (FEM) + f32 (actor)" if use_actor else "f64", "data": "synthetic",
            "config": bench_config(args, world),
            "roofline": roofline,
            "roofline_fem": roof_fem,
            "stages": stages,
            "cpu_baseline": cpu_line,
            "cpu_baseline_c_env_step": c_line,
            "e2e": {"value": B * world / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "path": e2e_path,
                    "h2d_gbs_per_rank": h2d / (e2e_ms * 1e-3) / 1e9, "d2h_gbs_per_rank": d2h / (e2e_ms * 1e-3) / 1e9},
            "e2e_compact_state": e2e_compact,
            "e2e_resident_state": e2e_res,
            "gpu_launches": launches,
            "clocks": clocks,
            "status_nonzero_envs": status_bad,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
