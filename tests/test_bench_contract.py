"""The JSON lines bench.py prints are what the round driver parses: keep their keys and types pinned.
CPU: the reference arm (oracle port on the host cores).  GPU: the B200 arm with a short run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric": str, "value": float, "unit": str, "n_gpus": int, "steps": int, "warmup": int, "ms_per_step": float,
             "higher_is_better": bool, "scaling": str, "dtype": str, "data": str, "config": dict, "cpu_baseline": dict,
             "e2e": dict, "gpu_launches": int}


def run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]           # exactly ONE JSON line
    return json.loads(lines[0])


def check_base(d):
    for k, t in BASE_KEYS.items():
        assert k in d, k
        assert isinstance(d[k], t) or (t is float and isinstance(d[k], int)), (k, type(d[k]))
    assert d["vs_baseline"] is None                       # BASELINE.md publishes no number for this metric
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in d["cpu_baseline"], k


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--ref-step-seconds", "0.4")
    check_base(d)
    # the same `config` object as the B200 arm prints (the driver compares them)
    assert {"workload", "family", "envs_per_gpu", "nodes", "elements", "free_dofs", "l2", "actions", "parallelism"} <= set(d["config"])
    assert d["impl"] == "reference" and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"] > 0


@pytest.mark.gpu
def test_b200_arm_line():
    d = run_bench("--steps", "6", "--warmup", "3", "--cpu-seconds", "0.5", "--batch", "512")
    check_base(d)
    assert "impl" not in d or d["impl"] == "b200"
    assert d["gpu_launches"] == 6 * 3                     # Pareto branch + fused actor network + env-step per step
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"]
    c = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(c)
    assert d["status_nonzero_envs"] == 0
    # round-2 keys: per-rank link rates, the compact-state end-to-end number, the legs at BASELINE configs 3 / 4 shapes
    assert d["e2e"]["h2d_gbs_per_rank"] > 0 and d["e2e"]["d2h_gbs_per_rank"] > 0
    assert d["e2e_compact_state"]["d2h_bytes_per_step"] < d["e2e"]["d2h_bytes_per_step"]
    ex = d["extra"]
    assert ex["config3"]["family"] == "small_roof" and ex["config3"]["envs_per_gpu"] == 16384 and ex["config3"]["value"] > 0
    assert ex["config4"]["family"] == "large_bridge" and ex["config4"]["envs_per_gpu"] == 1024
    assert 0 < ex["config3"]["roofline_fem"]["frac"] < 1 and ex["actor_pareto_P50"]["P"] == 50
    assert d["config"]["nodes"] == 16 and d["config"]["free_dofs"] == 28


@pytest.mark.gpu
def test_training_leg_line():
    d = run_bench("--train", "--steps", "3")
    assert d["family"] == "large_roof" and d["envs_per_gpu"] == 1024 and d["value"] > 0 and d["n_gpus"] == 1
    assert d["models_identical_across_ranks"] is True and d["learner_update"].startswith("one captured CUDA graph")
    assert set(d["stages_ms"]) >= {"rollout_3x_act_3x_env_step", "replay_push", "learner_train_update"}


@pytest.mark.gpu
def test_dump_outputs_repeat(tmp_path):
    """--dump-outputs: the last timed step's outputs as float32 / float64 .npy files, identical for identical arguments;
    one more timed step (--steps 5) is the oracle's env-step of the --steps 4 state under the dumped actions"""
    import numpy as np
    from oracle.truss_oracle import TrussOracle
    args = ("--warmup", "3", "--cpu-seconds", "0.2", "--batch", "300", "--no-extras")
    dumps = []
    for k, steps in enumerate(("4", "4", "5")):
        run_bench("--steps", steps, *args, "--dump-outputs", str(tmp_path / str(k)))
        dumps.append({f[:-4]: np.load(tmp_path / str(k) / f) for f in sorted(os.listdir(tmp_path / str(k)))})
    a, b, c = dumps
    assert {"a_geo", "a_topo", "x_n", "nN_x_e", "point", "status", "d"} <= set(a) and set(a) == set(b) == set(c)
    for name in a:
        assert a[name].dtype in (np.float32, np.float64) and a[name].shape[0] == 300, name
        assert np.array_equal(a[name], b[name]), name
    assert (a["status"] == 0).all() and (c["status"] == 0).all() and np.isfinite(a["d"]).all()
    assert not np.array_equal(a["nN_x_n"], c["nN_x_n"])
    o = TrussOracle("small_bridge")
    for i in range(0, 300, 37):
        # the coin of a step is not dumped: one of the two must give the dumped state
        outs = [o.step(a["nN_x_n"][i], a["nN_x_e"][i], a["move_range"][i, :, 0], a["move_range"][i, :, 1],
                       c["a_geo"][i].copy(), c["a_topo"][i].copy(), coin) for coin in (False, True)]
        assert any(np.array_equal(out["y"].astype(np.float32), c["nN_x_n"][i, :, 1]) and
                   np.array_equal(out["section"], c["nN_x_e"][i, :, 0].astype(np.int32)) and
                   np.array_equal(out["max_up"], c["move_range"][i, :, 0]) and
                   np.array_equal(out["max_down"], c["move_range"][i, :, 1]) for out in outs), i


def test_dump_outputs_sample():
    """a batch larger than the dump budget is cut to the same sorted sample of environments for every output"""
    import numpy as np
    import torch
    import bench

    class Env:
        FP64_FIELDS = ("d",)
        fp64_outputs, device = True, torch.device("cpu")

        def __init__(self, B):
            self.B = B
            rows = torch.arange(B)
            for k, shape in (("x_n", (13,)), ("A_s", (3, 3)), ("A_n_ts", (3, 3)), ("A_n_cs", (3, 3)), ("nN_x_n", (12,)),
                             ("nN_x_e", (5, 21)), ("move_range", (3, 2)), ("point", (4,)), ("y", (3,))):
                setattr(self, k, rows.reshape(B, *[1] * len(shape)).expand(B, *shape).to(torch.float32).contiguous())
            self.d = rows.to(torch.float64)[:, None].repeat(1, 6)
            self.status = torch.zeros(B, dtype=torch.int32)
            self.y_weak = torch.ones(B, 3, dtype=torch.uint8)

    small = bench.last_step_outputs(Env(50), (torch.rand(50, 3, 2), torch.rand(50, 3, 3)))
    assert all(a.shape[0] == 50 for a in small.values()) and small["d"].dtype == np.float64
    assert small["status"].dtype == np.float32 and small["y_weak"].dtype == np.float32
    B = 200000
    out = bench.last_step_outputs(Env(B), None)
    assert "a_geo" not in out
    rows = out["x_n"][:, 0].astype(np.int64)
    assert 0 < len(rows) < B and (np.diff(rows) > 0).all()
    for name, a in out.items():
        if name not in ("status", "y_weak"):                  # every other fake output carries its row index
            assert np.array_equal(a.reshape(len(rows), -1)[:, 0], rows), name
    assert sum(a.nbytes for a in out.values()) <= bench.DUMP_LIMIT_BYTES
    assert np.array_equal(bench.last_step_outputs(Env(B), None)["d"], out["d"])


def test_e2e_piece_schedule_argument():
    """--e2e-pieces: 'auto' (HostRollout decides), a count of equal pieces, explicit sizes, or fractions of the batch"""
    import bench
    assert bench.e2e_piece_schedule("auto", 4096) == "auto"
    assert bench.e2e_piece_schedule("3", 4096) == 3
    assert bench.e2e_piece_schedule("512,1536,2048", 4096) == [512, 1536, 2048]
    frac = bench.e2e_piece_schedule("0.125,0.375,0.5", 4096)
    assert frac == [512, 1536, 2048] and all(v % 32 == 0 for v in frac[:-1])
    with pytest.raises(SystemExit):
        bench.e2e_piece_schedule("512,512", 4096)
