"""Named geometry families = the constants the reference drivers hard-code
(``*/code/master_DDPG_truss2D_MO.py``; SURVEY.md section 2.1) and the section catalogue
``section_data/01_brace_rod2.csv``.  Host logic only."""
from __future__ import annotations

from dataclasses import dataclass, field

SECTION_AREA_CM2 = (9.085, 20.41, 38.89, 81.23, 164.6)
SECTION_INERTIA_CM4 = (59.5, 300.0, 830.0, 4230.0, 18700.0)
YOUNG = 2 * 1e11
ALLOW_STRESS = 235 * 1e6 / 1.5

BRIDGE, ROOF = 0, 1
SYM_NONE, SYM_SMALL, SYM_LARGE = 0, 1, 2


@dataclass(frozen=True)
class FamilySpec:
    """Arguments of ``gen_model(num_x, num_y, span_x, span_y, tar_y, dmin, loadx, loady, truss_type,
    support_case, topo_code)`` plus which ``truss2D_ENV.py`` symmetry convention applies."""
    name: str
    num_x: int
    span_x: tuple
    span_y: tuple
    tar_y: tuple
    dmin: float
    loadx: float
    loady: float
    truss_type: str
    support_case: int = 1
    symmetry: int = SYM_NONE
    section_area_cm2: tuple = SECTION_AREA_CM2
    section_inertia_cm4: tuple = SECTION_INERTIA_CM4

    @property
    def N(self):
        return 2 * self.num_x

    @property
    def E(self):
        return 5 * self.num_x - 4


_SMALL_TAR = (4, 3, 2.5, 2, 2, 2.5, 3, 4)
_LARGE_TAR = (3, 2.75, 2.5, 2.25, 2.25, 2, 2, 2, 2, 2, 2, 2.25, 2.25, 2.5, 2.75, 3)

FAMILIES = {
    # test/00_small_bridge/code/master_DDPG_truss2D_MO.py:813-830
    "small_bridge": FamilySpec("small_bridge", 8, (5,) * 7, (8,), _SMALL_TAR, 0.3, 0, -75 * 1000, "bridge", 1, SYM_SMALL),
    # test/01_small_roof/code/master_DDPG_truss2D_MO.py:806-823
    "small_roof": FamilySpec("small_roof", 8, (5,) * 7, (8,), _SMALL_TAR, 0.3, 0, -120 * 1000, "roof", 1, SYM_SMALL),
    # test/02_large_bridge/code/master_DDPG_truss2D_MO.py:806-823
    "large_bridge": FamilySpec("large_bridge", 16, (5,) * 15, (6,), _LARGE_TAR, 0.3, 0, -7.5 * 1000, "bridge", 1, SYM_LARGE),
    # test/03_large_roof/code/master_DDPG_truss2D_MO.py:806-823
    "large_roof": FamilySpec("large_roof", 16, (5,) * 15, (6,), _LARGE_TAR, 0.3, 0, -8 * 1000, "roof", 1, SYM_LARGE),
}


# the five 6 x 2 training shapes with mixed spans (train/code/master_DDPG_truss2D_MO.py:787-795: trainChoice; dmin = 0.2,
# gen_load_y = -100000, support_case 1, truss type drawn per episode :809-815).  train/code/truss2D_ENV.py has no symmetry step.
_TRAIN_TAR = ((1.0, 1.5, 2.0, 2.0, 1.5, 1.0), (1.0, 3.0, 3.0, 2.0, 1.5, 1.0), (1.0, 1.5, 2.0, 3.0, 3.0, 1.0),
              (1.0, 3.0, 2.0, 2.0, 3.0, 1.0), (3.0, 2.0, 1.0, 1.0, 2.0, 3.0))
for _i, _tar in enumerate(_TRAIN_TAR):
    for _tt in ("roof", "bridge"):
        FAMILIES["train%d_%s" % (_i, _tt)] = FamilySpec("train%d_%s" % (_i, _tt), 6, (4.0, 3.0, 5.0, 3.0, 5.0), (5,), _tar, 0.2, 0,
                                                        -100000, _tt, 1, SYM_NONE)

# the ten training families (five shapes x two truss types) in a fixed order: the index of a name here is the family id
# of a mixed-family batch built over TRAIN_FAMILIES (batched_env.MixedTrussEnv)
TRAIN_FAMILIES = tuple("train%d_%s" % (_i, _tt) for _i in range(len(_TRAIN_TAR)) for _tt in ("roof", "bridge"))


def family_desc(spec: FamilySpec):
    """FamilySpec -> ctypes ``tfem_family_desc``"""
    from . import capi
    d = capi.FamilyDesc()
    d.num_x = spec.num_x
    d.truss_type = BRIDGE if spec.truss_type == "bridge" else ROOF
    d.support_case = spec.support_case if spec.support_case is not None else 1
    d.symmetry = spec.symmetry
    if len(spec.span_x) != spec.num_x - 1 or len(spec.tar_y) != spec.num_x:
        raise ValueError("span_x must have num_x-1 entries and tar_y num_x entries")
    for i, v in enumerate(spec.span_x):
        d.span_x[i] = float(v)
    d.span_y = float(spec.span_y[0])
    for i, v in enumerate(spec.tar_y):
        d.tar_y[i] = float(v)
    d.d_min = float(spec.dmin)
    d.load_y = float(spec.loady)
    for i in range(5):
        d.section_area_cm2[i] = spec.section_area_cm2[i]
        d.section_inertia_cm4[i] = spec.section_inertia_cm4[i]
    d.young = YOUNG
    d.allow_stress = ALLOW_STRESS
    return d
