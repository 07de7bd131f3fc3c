"""Pins the oracle's wall force / moment integration (and the wall stress tensor the viscous flux stores for it)
against the reference's own wallIntegrationFace (src/solver/surfaceIntegrations.F90:406-881, translated Fortran -> C,
oracle/_ref).  The viscSubface%tau planes fed to the reference come from the oracle's viscous flux, which is itself
pinned against blockette.F90's viscousFlux through the residual tests.  Where the translated library is absent, against
the recorded digests of its outputs (tests/refgold.py)."""
import numpy as np
import pytest

import refgold as gold
from oracle import refblockette as rb
from util import case

IMIN, IMAX, JMIN, JMAX, KMIN, KMAX = 1, 2, 3, 4, 5, 6
SYMM, WALL, FAR, EULERWALL, EXTRAP, ISOWALL = 1, 2, 3, 4, 5, 6


@pytest.mark.parametrize("perm", [
    None,
    {IMIN: WALL, IMAX: FAR, JMIN: FAR, JMAX: SYMM, KMIN: FAR, KMAX: WALL},
    {IMIN: FAR, IMAX: ISOWALL, JMIN: WALL, JMAX: FAR, KMIN: SYMM, KMAX: FAR},
    {IMIN: FAR, IMAX: FAR, JMIN: SYMM, JMAX: WALL, KMIN: WALL, KMAX: FAR},
])
def test_wall_forces_match_reference(perm):
    from oracle.pyoracle import Oracle

    kw = {} if perm is None else {"physical_faces": perm}
    prm, hb = case(10, 9, 8, {"equationType": "RANS"}, **kw)
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    o = Oracle(hb, prm)
    o.apply_turb_bc(True); o.apply_flow_bc(True)
    o.residual_core(8 | 16)                     # stores hb.wallTau
    ref_point = (0.3, -0.2, 0.1)
    mine = o.wall_forces(ref_point, p_ref=2.5)
    ref = gold.run(lambda: rb.wall_forces(hb, prm, ref_point, p_ref=2.5))
    assert np.abs(mine[0]).max() > 0 and np.abs(mine[1]).max() > 0
    gold.same("Fp, Fv, Mp, Mv", ref, lambda ref: ref, mine)


def test_euler_wall_pressure_forces():
    from oracle.pyoracle import Oracle

    perm = {IMIN: FAR, IMAX: FAR, JMIN: SYMM, JMAX: FAR, KMIN: EULERWALL, KMAX: EULERWALL}
    prm, hb = case(9, 8, 10, {"equationType": "Euler"}, physical_faces=perm)
    o = Oracle(hb, prm)
    o.apply_flow_bc(True)
    o.residual_core(8)
    mine = o.wall_forces((0.0, 0.0, 0.0))
    ref = gold.run(lambda: rb.wall_forces(hb, prm, (0.0, 0.0, 0.0)))
    assert np.abs(mine[0]).max() > 0 and np.abs(mine[1]).max() == 0
    gold.same("Fp, Fv, Mp, Mv", ref, lambda ref: ref, mine)
