"""CPU: a rollout over a mixed-family env handle -- trollout_create_agents no longer refuses a handle of several
families (tfem_create_mixed); a tables-only one still fails with the tables-only error, before it touches a device."""
import ctypes as C

from mop_truss_marl_b200 import capi
from mop_truss_marl_b200.families import FAMILIES, TRAIN_FAMILIES, family_desc


def test_create_agents_on_tables_only_mixed_handle():
    from mop_truss_marl_b200.host_pipeline import _lib
    env = capi.MixedHandle([family_desc(FAMILIES[n]) for n in TRAIN_FAMILIES], -1)
    fake = (C.c_void_p * 3)(0x1000, 0x2000, 0x3000)     # opaque, never dereferenced
    out = C.c_void_p()
    rc = _lib.trollout_create_agents(env.ptr, fake, 3, 64, 1, C.byref(out))
    msg = _lib.trollout_last_error().decode()
    assert rc == -2 and "tables-only" in msg and not out.value, (rc, msg)
    env.close()
