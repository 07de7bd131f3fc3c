"""Wall force / moment integration on the device (adfb_forces) against the oracle and against the reference's own
wallIntegrationFace (oracle/_ref), incl. the wall stress tensor stored by the viscous flux kernel
(ADFB_RES_STORE_WALL == blocketteRes(useStoreWall))."""
import numpy as np
import pytest

import refgold as gold
from adflow_b200.solver import ADFLOW_B200, RES_FLOW, RES_SKIP_PREAMBLE, RES_STORE_WALL, RES_TURB
from oracle import refblockette as rb
from oracle.pyoracle import Oracle

from util import case

pytestmark = pytest.mark.gpu

IMIN, IMAX, JMIN, JMAX, KMIN, KMAX = 1, 2, 3, 4, 5, 6
SYMM, WALL, FAR, EULERWALL, EXTRAP, ISOWALL = 1, 2, 3, 4, 5, 6


def _cuda_forces(prm, hb, ref_point, p_ref, flags):
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        s.residual(flags | RES_STORE_WALL | RES_SKIP_PREAMBLE)
        return s.getForces(ref_point, p_ref), s
    finally:
        s.close()


@pytest.mark.parametrize("perm,disc", [
    (None, "central plus scalar dissipation"),
    ({IMIN: WALL, IMAX: FAR, JMIN: FAR, JMAX: SYMM, KMIN: FAR, KMAX: WALL}, "central plus matrix dissipation"),
    ({IMIN: FAR, IMAX: ISOWALL, JMIN: WALL, JMAX: FAR, KMIN: SYMM, KMAX: FAR}, "upwind"),
])
def test_forces_match_oracle_and_reference(cuda_lib, perm, disc):
    kw = {} if perm is None else {"physical_faces": perm}
    prm, hb = case(14, 11, 9, {"equationType": "RANS", "discretization": disc}, **kw)
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    o = Oracle(hb, prm)
    o.apply_turb_bc(True); o.apply_flow_bc(True)      # halos consistent on both sides
    ho = hb.copy()
    oo = Oracle(ho, prm)
    oo.residual_core(RES_FLOW | RES_TURB)
    ref_point, p_ref = (0.3, -0.2, 0.1), 2.5
    want = oo.wall_forces(ref_point, p_ref)
    got, _ = _cuda_forces(prm, hb, ref_point, p_ref, RES_FLOW | RES_TURB)
    scale = np.abs(want).max(axis=1, keepdims=True)
    assert (scale > 0).all()
    assert np.abs(got - want).max() <= 1e-12 * scale.max()
    assert (np.abs(got - want) <= 1e-11 * scale).all(), (got - want) / scale
    # the reference's own wallIntegrationFace (recorded digest of its output where the translated library is absent)
    ref = gold.value("Fp, Fv, Mp, Mv", gold.run(lambda: rb.wall_forces(ho, prm, ref_point, p_ref)), lambda ref: ref, want)
    assert (np.abs(got - ref) <= 1e-11 * scale).all()


def test_euler_wall_forces(cuda_lib):
    perm = {IMIN: FAR, IMAX: FAR, JMIN: SYMM, JMAX: FAR, KMIN: EULERWALL, KMAX: EULERWALL}
    prm, hb = case(12, 9, 10, {"equationType": "Euler"}, physical_faces=perm)
    Oracle(hb, prm).apply_flow_bc(True)
    ho = hb.copy()
    oo = Oracle(ho, prm)
    oo.residual_core(RES_FLOW)
    want = oo.wall_forces((0.0, 0.0, 0.0))
    got, _ = _cuda_forces(prm, hb, (0.0, 0.0, 0.0), 1.0, RES_FLOW)
    assert np.abs(got[1]).max() == 0.0
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_lift_and_drag_coefficients(cuda_lib):
    prm, hb = case(14, 11, 9, {"equationType": "RANS"})
    Oracle(hb, prm).apply_turb_bc(True)
    Oracle(hb, prm).apply_flow_bc(True)
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        s.residual(RES_FLOW | RES_TURB | RES_STORE_WALL | RES_SKIP_PREAMBLE)
        a = np.radians(1.8)
        lift, drag = np.array([-np.sin(a), np.cos(a), 0.0]), np.array([np.cos(a), np.sin(a), 0.0])
        f = s.evalFunctions(lift, drag, mach_coef=0.8, surface_ref=1.3)
        F = s.getForces()
    finally:
        s.close()
    fact = 2.0 / (prm.gammaInf * 0.8 * 0.8 * 1.3)
    assert abs(f["cl"] - fact * np.dot(F[0] + F[1], lift)) <= 1e-15 + 1e-13 * abs(f["cl"])
    assert abs(f["cd"] - (f["cdp"] + f["cdv"])) <= 1e-13 * abs(f["cd"])
