"""Per-warp wait / work cycle counters of the actor kernel (development build, -DTACTOR_PROF).

    python -m mop_truss_marl_b200.build --prof
    TFEM_LIB=mop_truss_marl_b200/lib/libtfem_prof.so python scripts/actor_prof.py [family] [B] [P]

Prints, for CTA 0 of one forward, what every warp of every role waited on (cycles and share of the kernel)."""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mop_truss_marl_b200 import actor, capi  # noqa: E402
from mop_truss_marl_b200.batched_env import BatchedTrussEnv  # noqa: E402
from mop_truss_marl_b200.families import FAMILIES  # noqa: E402
from mop_truss_marl_b200.tf_checkpoint import random_actor_weights  # noqa: E402

NPH, NEPIW = 2, 4                      # generator phases and epilogue warps of actor_pipe_kernel (tactor_pipe.cuh)


def main():
    family = sys.argv[1] if len(sys.argv) > 1 else "small_bridge"
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
    P = int(sys.argv[3]) if len(sys.argv) > 3 else 1
    env = BatchedTrussEnv(FAMILIES[family], B, device="cuda:0")
    env.reset()
    act = actor.BatchedActor(random_actor_weights(0), env.N, B, device="cuda:0")
    x_p = torch.rand(B, P, 4, device="cuda:0")
    A_p = torch.eye(P, device="cuda:0").repeat(B, 1, 1).contiguous()
    for _ in range(3):
        act.forward(env.x_n, env.A_n, env.A_s, env.A_n_ts, env.A_n_cs, x_p, A_p)
    try:
        act.check()
    except capi.TfemError as e:        # reported; the counters are still read
        print(json.dumps({"status": str(e)}))
    ngen, nepi = 4 * NPH, NEPIW
    nw = ngen + nepi + 2
    buf = (C.c_longlong * (nw * 8))()
    capi.lib.tactor_prof_read.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    rc = capi.lib.tactor_prof_read(act._h, buf, nw * 8)
    assert rc == 0, rc
    a = np.array(buf[:], dtype=np.int64).reshape(nw, 8)
    names = {"gen": ["x_full", "h_ready", "a_empty", "a_empty(dead)", "wait::st", "X build", "mix+split", "total"],
             "epi": ["acc_full", "drain", "-", "-", "-", "-", "-", "total"],
             "iss": ["a_full", "w_full", "acc_empty", "-", "-", "-", "-", "total"],
             "prod": ["w_empty", "-", "-", "-", "-", "-", "-", "total"]}
    out = []
    for w in range(nw):
        role = "gen" if w < ngen else "epi" if w < ngen + nepi else "iss" if w == ngen + nepi else "prod"
        tot = max(int(a[w, 7]), 1)
        row = {"warp": w, "role": role, "total_cycles": tot}
        for k, nm in enumerate(names[role][:7]):
            if nm != "-":
                row[nm] = round(float(a[w, k]) / tot, 3)
        out.append(row)
        print(json.dumps(row))
    if os.environ.get("TACTOR_TRACE"):
        np.save(os.environ["TACTOR_TRACE"], trace(act))
    return out




def trace(act):
    """time line of item 1 of CTA 0 (see PROF_TRACE in tactor_pipe.cuh)"""
    n = 2048 + 4608 + NEPIW * 7 * 2 + 64
    buf = (C.c_longlong * ((n + 1) // 2))()
    capi.lib.tactor_prof_read.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    assert capi.lib.tactor_prof_read(act._h, buf, (n + 1) // 2) == 0
    w = np.frombuffer(buf, dtype=np.uint32)[2048 - 32:]   # tactor_prof_read starts at error_flag + 32 ints
    return w


if __name__ == "__main__":
    main()
