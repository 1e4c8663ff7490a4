"""CPU: the multi-agent rollout ABI -- the ctypes layout of trollout_agents_io matches the C header, and
trollout_create_agents refuses bad agent lists before it touches a device."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

from mop_truss_marl_b200 import capi
from mop_truss_marl_b200.families import FAMILIES, family_desc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_agents_io_layout_matches_header(tmp_path):
    from mop_truss_marl_b200 import host_pipeline as hp
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "trollout.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %d\\n", sizeof(trollout_agents_io), offsetof(trollout_agents_io, P),\n'
                   '         offsetof(trollout_agents_io, child), sizeof(trollout_child), offsetof(trollout_child, a_topo),\n'
                   '         TROLLOUT_MAX_AGENTS);\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(hp._AgentsIO), hp._AgentsIO.P.offset, hp._AgentsIO.child.offset, C.sizeof(hp._Child),
                   hp._Child.a_topo.offset, hp.MAX_AGENTS]


def test_create_agents_refusals():
    from mop_truss_marl_b200.host_pipeline import _lib
    env = capi.Handle(family_desc(FAMILIES["small_bridge"]), device=-1)
    # opaque, never dereferenced: every refusal below comes before the actors are used
    fake = (C.c_void_p * 4)(0x1000, 0x2000, 0x3000, 0x4000)
    out = C.c_void_p()

    def create(actors, n):
        rc = _lib.trollout_create_agents(env.ptr, actors, n, 64, 1, C.byref(out))
        return rc, _lib.trollout_last_error().decode()
    assert create(fake, 0) == (-1, "n_agents must be in 1..3, got 0")
    assert create(fake, 4) == (-1, "n_agents must be in 1..3, got 4")
    assert create((C.c_void_p * 3)(0x1000, 0x2000, 0x1000), 3) == (-1, "the agents must be distinct actor handles")
    assert create((C.c_void_p * 2)(0x1000, None), 2)[0] == -1
    rc, msg = create(fake, 3)
    assert rc == -2 and "tables-only" in msg and not out.value
    env.close()
