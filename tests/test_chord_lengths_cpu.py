"""CPU: families of every chord length num_x = 3..16 with train/code's ENV (no symmetry step), the shapes a user of the
reference reaches by editing gen_model's arguments (train/code trains on 6 x 2, test/* evaluates on 8 x 2 and 16 x 2).

* tables-only handles of every num_x x truss type x support case against the oracle's build_mesh;
* a tables-only mixed handle of two families of one new num_x;
* what tfem_create and tactor_create refuse, and that a newly accepted node count gets past the argument checks."""
import ctypes as C

import numpy as np
import pytest

from mop_truss_marl_b200 import capi, family_desc
from mop_truss_marl_b200.families import SYM_LARGE, SYM_NONE, SYM_SMALL, FamilySpec
from oracle.truss_oracle import FamilySpec as OracleSpec
from oracle.truss_oracle import TrussOracle

CHORDS = tuple(range(3, 17))


def spec_pair(num_x, truss_type, support_case=1, span_y=5.0, loady=-100000.0):
    """the library's and the oracle's description of one family: mixed 4 / 3 / 5 m spans, targets rising from 1 m at
    mid-span to 3 m at the ends, d_min 0.2 (the training driver's values)"""
    span_x = tuple((4.0, 3.0, 5.0)[i % 3] for i in range(num_x - 1))
    tar_y = tuple(1.0 + 2.0 * abs(2 * i - (num_x - 1)) / (num_x - 1) for i in range(num_x))
    name = "chord%d_%s_sc%d" % (num_x, truss_type, support_case)
    lib = FamilySpec(name, num_x, span_x, (span_y,), tar_y, 0.2, 0, loady, truss_type, support_case, SYM_NONE)
    orc = OracleSpec(name, num_x, list(span_x), [span_y], list(tar_y), 0.2, 0, loady, truss_type, support_case, "none")
    return lib, orc


@pytest.mark.parametrize("support_case", [1, 2, 3, 4])
@pytest.mark.parametrize("truss_type", ["bridge", "roof"])
@pytest.mark.parametrize("num_x", CHORDS)
def test_tables_match_oracle(num_x, truss_type, support_case):
    lib, orc = spec_pair(num_x, truss_type, support_case)
    o = TrussOracle(orc)
    m = o.mesh
    h = capi.Handle(family_desc(lib), device=-1)
    try:
        assert (h.dims.N, h.dims.E, h.dims.ndof, h.dims.num_x) == (m.N, m.E, m.ndof, num_x)
        want = {
            "conn": np.array(m.conn, np.int32), "tnsc": np.array(m.tnsc, np.int32), "res": np.array(m.res, np.int32),
            "top": np.array(m.top, np.int32), "pair": np.array(m.pair, np.int32), "loaded": np.array(m.loaded, np.int32),
            "loadvec": np.array(m.P, np.float64), "x": np.array(m.x, np.float64), "y0": np.array(m.y0, np.float64),
            "target": np.array([0.0 if t is None else t for t in m.target_top], np.float64),
            "A_n": o.A_n, "mask": o.mask, "nC_e": o.nC_e,
            "int_obj": np.array([o.int_obj1, o.int_obj2], np.float32),
            "sym_src": np.array([m.sym_src_false, m.sym_src_true], np.int32),
            "sym_elem": np.arange(m.E, dtype=np.int32),
        }
        for k, v in want.items():
            got = h.table(k)
            assert got.dtype == v.dtype and np.array_equal(got.reshape(v.shape), v), k
        scal = h.table("scalars")
        assert np.array_equal(scal[:4], np.array([m.y_max, m.y_min, m.d_min, m.max_deformation], np.float64))
        assert scal[6] == lib.loady
    finally:
        h.close()


@pytest.mark.parametrize("num_x", [5, 10, 15])
def test_mixed_tables_only_handle(num_x):
    """two families of one new num_x (truss type, spans and targets differing; support case shared) in one handle"""
    import dataclasses
    bridge, _ = spec_pair(num_x, "bridge")
    roof, _ = spec_pair(num_x, "roof", span_y=4.0)
    roof = dataclasses.replace(roof, span_x=tuple(5.0 for _ in roof.span_x), tar_y=tuple(2.0 for _ in roof.tar_y))
    h = capi.MixedHandle([family_desc(bridge), family_desc(roof)], device=-1)
    try:
        for k in ("conn", "tnsc", "res", "top", "pair", "A_n", "mask", "nC_e"):
            single = capi.Handle(family_desc(bridge), device=-1)
            assert np.array_equal(h.table(k), single.table(k)), k
            single.close()
        with pytest.raises(capi.TfemError, match="tables-only handle of one family"):
            h.table("target")
    finally:
        h.close()


def create_error(spec):
    h = C.c_void_p()
    rc = capi.lib.tfem_create(C.byref(family_desc(spec)), -1, C.byref(h))
    return rc, capi.lib.tfem_last_error().decode()


@pytest.mark.parametrize("num_x", [2, 17])
def test_chord_length_out_of_range_refused(num_x):
    import dataclasses
    base, _ = spec_pair(3, "bridge")
    bad = dataclasses.replace(base, num_x=num_x, span_x=(5.0,) * (num_x - 1), tar_y=(2.0,) * num_x)
    if num_x > 16:                                     # the descriptor holds at most 16 columns: set num_x past it directly
        d = family_desc(base)
        d.num_x = num_x
        h = C.c_void_p()
        rc, err = capi.lib.tfem_create(C.byref(d), -1, C.byref(h)), capi.lib.tfem_last_error().decode()
    else:
        rc, err = create_error(bad)
    assert rc == -3
    assert "num_x must be 3..16" in err and ("got %d" % num_x) in err


@pytest.mark.parametrize("symmetry,word", [(SYM_SMALL, "small"), (SYM_LARGE, "large")])
@pytest.mark.parametrize("num_x", [7, 10, 12])
def test_symmetric_convention_of_a_new_chord_length_refused(num_x, symmetry, word):
    import dataclasses
    base, _ = spec_pair(num_x, "bridge")
    rc, err = create_error(dataclasses.replace(base, symmetry=symmetry))
    assert rc == -3
    assert word + " symmetry convention" in err and "num_x = %d" % num_x in err


@pytest.mark.parametrize("num_x", [6, 8, 16])
@pytest.mark.parametrize("symmetry", [SYM_NONE, SYM_SMALL, SYM_LARGE])
def test_chord_lengths_of_the_reference_keep_every_convention(num_x, symmetry):
    import dataclasses
    base, _ = spec_pair(num_x, "roof")
    rc, err = create_error(dataclasses.replace(base, symmetry=symmetry))
    assert rc == 0, err


# ================================================= actor node counts ====================================================
def actor_create(nodes):
    from mop_truss_marl_b200 import actor, tf_checkpoint
    weights = tf_checkpoint.random_actor_weights(seed=1)
    keep, w = [], actor._Weights()
    for i, name in enumerate(tf_checkpoint.ACTOR_LAYERS):
        keep += [np.ascontiguousarray(a, np.float32) for a in weights[name]]
        w.kernel[i], w.bias[i] = keep[-2].ctypes.data, keep[-1].ctypes.data
    h = C.c_void_p()
    rc = capi.lib.tactor_create(C.byref(w), int(nodes), 8, 0, C.byref(h))
    return rc, capi.lib.tactor_last_error().decode(), h


@pytest.mark.parametrize("nodes", [-2, 0, 2, 4, 5, 7, 13, 31, 33, 34, 64])
def test_actor_node_counts_refused_before_the_device_check(nodes):
    rc, err, h = actor_create(nodes)
    assert rc == -3 and "nodes must be even and in 6..32" in err, (rc, err)
    assert not h.value


@pytest.mark.parametrize("nodes", [6, 10, 14, 18, 24, 30])
def test_new_actor_node_counts_reach_the_device_check(nodes):
    """accepted: without a device the call fails at the device check; with one it makes the handle"""
    rc, err, h = actor_create(nodes)
    if rc == 0:
        capi.lib.tactor_destroy(h)
        return
    assert rc == -2 and "no CUDA device" in err, (rc, err)
    assert not h.value
