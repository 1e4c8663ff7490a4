"""CPU: mixed-family handles (tfem_create_mixed) on tables-only handles -- which families may share a handle, which
tables such a handle serves, and that it refuses to compute without a GPU."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from mop_truss_marl_b200 import FAMILIES, capi, family_desc
from mop_truss_marl_b200.families import TRAIN_FAMILIES

TOPOLOGY = ("conn", "tnsc", "res", "top", "pair", "A_n", "mask", "nC_e")
PER_FAMILY = ("loaded", "loadvec", "x", "y0", "target", "sym_src", "sym_elem", "int_obj", "scalars")


def descs(names):
    return [family_desc(FAMILIES[n] if isinstance(n, str) else n) for n in names]


def create(specs, device=-1):
    arr = (capi.FamilyDesc * max(1, len(specs)))(*descs(specs))
    h = C.c_void_p()
    rc = capi.lib.tfem_create_mixed(arr, len(specs), device, C.byref(h))
    return rc, h, capi.lib.tfem_last_error().decode()


def test_train_families():
    assert len(TRAIN_FAMILIES) == 10 and len(set(TRAIN_FAMILIES)) == 10
    assert all(n in FAMILIES and FAMILIES[n].num_x == 6 for n in TRAIN_FAMILIES)
    assert {FAMILIES[n].truss_type for n in TRAIN_FAMILIES} == {"roof", "bridge"}
    h = capi.MixedHandle(descs(TRAIN_FAMILIES), device=-1)
    assert h.n_families == 10 and (h.dims.N, h.dims.E, h.dims.device) == (12, 26, -1)
    h.close()


@pytest.mark.parametrize("pair", [("small_bridge", "small_roof"), ("large_bridge", "large_roof")])
def test_same_topology_test_families(pair):
    h = capi.MixedHandle(descs(pair), device=-1)
    h.close()


def test_num_x_mismatch_refused():
    rc, _, err = create(["train0_roof", "small_bridge"])
    assert rc == -3 and "num_x" in err and "family 1" in err


def test_support_case_mismatch_refused():
    other = dataclasses.replace(FAMILIES["train0_roof"], support_case=2)
    rc, _, err = create(["train0_roof", "train1_bridge", other])
    assert rc == -3 and "RES" in err and "family 2" in err


@pytest.mark.parametrize("n", [0, 17])
def test_family_count_bounds(n):
    rc, _, err = create(["train0_roof"] * n)
    assert rc == -1 and "n_families" in err


def test_unsupported_member_refused():
    bad = dataclasses.replace(FAMILIES["train0_roof"], num_x=7, span_x=(5,) * 6, tar_y=(1,) * 7)
    rc, _, err = create(["train0_roof", bad])
    assert rc == -3 and "family 1" in err and "num_x" in err


def test_topology_tables_served_family_tables_refused():
    h = capi.MixedHandle(descs(TRAIN_FAMILIES), device=-1)
    single = capi.Handle(family_desc(FAMILIES[TRAIN_FAMILIES[0]]), device=-1)
    for name in TOPOLOGY:
        assert np.array_equal(h.table(name), single.table(name)), name
    for name in PER_FAMILY:
        with pytest.raises(capi.TfemError, match="tables-only handle of one family"):
            h.table(name)
    with pytest.raises(capi.TfemError, match="unknown table id"):
        tid = 99
        arr = np.empty(8)
        capi.check(capi.lib.tfem_get_table(h.ptr, tid, arr.ctypes.data_as(C.c_void_p), arr.nbytes))


def test_one_family_handle_is_a_single_family_handle():
    h = capi.MixedHandle(descs(["small_roof"]), device=-1)
    single = capi.Handle(family_desc(FAMILIES["small_roof"]), device=-1)
    for name in TOPOLOGY + PER_FAMILY:
        assert np.array_equal(h.table(name), single.table(name)), name
    # the single-family entry points take it (and fail only for want of a device)
    out = capi.StepOut()
    assert capi.lib.tfem_reset(h.ptr, 1, None, C.byref(out), None) == -2


def test_compute_entry_points_need_a_device():
    h = capi.MixedHandle(descs(TRAIN_FAMILIES), device=-1)
    fam = np.zeros(4, np.uint8)
    out = capi.StepOut()
    rc = capi.lib.tfem_reset_mixed(h.ptr, 4, fam.ctypes.data, None, C.byref(out), None)
    assert rc == -2 and "no CPU path" in capi.lib.tfem_last_error().decode()
    buf = np.zeros(4 * 12 * 21, np.float32)
    sin = capi.StepIn()
    sin.set_node = sin.set_element = sin.a_geo = sin.a_topo = sin.move_range = buf.ctypes.data
    rc = capi.lib.tfem_step_mixed(h.ptr, 4, fam.ctypes.data, C.byref(sin), C.byref(out), None)
    assert rc == -2


def test_single_family_entry_points_refuse_several_families():
    h = capi.MixedHandle(descs(["train0_roof", "train0_bridge"]), device=-1)
    out = capi.StepOut()
    sin = capi.StepIn()
    buf = np.zeros(4096)
    p = buf.ctypes.data
    sin.set_node = sin.set_element = sin.a_geo = sin.a_topo = sin.move_range = p
    gout = capi.GenesOut()
    calls = {
        "tfem_reset": lambda: capi.lib.tfem_reset(h.ptr, 1, None, C.byref(out), None),
        "tfem_step": lambda: capi.lib.tfem_step(h.ptr, 1, C.byref(sin), C.byref(out), None),
        "tfem_solve_only": lambda: capi.lib.tfem_solve_only(h.ptr, 1, p, p, None, None, None, None, None, None, None),
        "tfem_read_genes": lambda: capi.lib.tfem_read_genes(h.ptr, 1, p, 1.0, 0.0, 0.0, C.byref(gout), None),
        "tfem_step_host": lambda: capi.lib.tfem_step_host(h.ptr, 1, C.byref(sin), C.byref(out), None),
        "tfem_solve_dense_dmma": lambda: capi.lib.tfem_solve_dense_dmma(h.ptr, 1, p, p, p, None, None),
    }
    for name, call in calls.items():
        assert call() == -1, name
        err = capi.lib.tfem_last_error().decode()
        assert err.startswith(name) and "2 families" in err, (name, err)
    capi.lib.tfem_step(h.ptr, 1, C.byref(sin), C.byref(out), None)
    assert "use tfem_step_mixed" in capi.lib.tfem_last_error().decode()


def test_new_exports():
    for name in ("tfem_create_mixed", "tfem_reset_mixed", "tfem_step_mixed"):
        assert name in capi.EXPORTS and hasattr(capi.lib, name)
    assert capi.STATUS_BAD_FAMILY == 4 and capi.MAX_FAMILIES == 16
