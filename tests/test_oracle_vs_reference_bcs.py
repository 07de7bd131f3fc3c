"""Pins the oracle's boundary conditions against the reference's own routines (translated Fortran -> C,
oracle/_ref): applyAllBC_block (src/solver/BCRoutines.F90:57-218) with bcSymm1stHalo/2ndHalo, bcNSWallAdiabatic,
bcFarfield, bcEulerWall, extrapolate2ndHalo, computeEtot and setBCPointers (src/utils/utils.F90:881-1174).
Bit-exact on every array the BCs write (w, p, rlv, rev incl. both halo layers); where the translated library is absent,
against the recorded digests of its outputs (tests/refgold.py)."""
import numpy as np
import pytest

import refgold as gold
from oracle import refblockette as rb
from util import case

IMIN, IMAX, JMIN, JMAX, KMIN, KMAX = 1, 2, 3, 4, 5, 6
SYMM, WALL, FAR, EULERWALL, EXTRAP, ISOWALL = 1, 2, 3, 4, 5, 6
SUBOUT, SUBIN, SUPIN, SUPOUT = 7, 8, 9, 10


def _check(prm, hb, second_halo=True):
    from oracle.pyoracle import Oracle

    ho = hb.copy()
    Oracle(ho, prm).apply_flow_bc(second_halo)
    r = gold.run(lambda: rb.call(hb, prm, "bcroutines_applyallbc_block", int(second_halo)))
    changed = 0
    for ref, mine in (("w", "w"), ("p", "p"), ("rlv", "rlv"), ("rev", "rev")):
        b = getattr(ho, mine)
        gold.same(ref, r, lambda r: r.a[ref], b)
        changed += int(not np.array_equal(b, getattr(hb, mine)))
    assert changed > 0  # the BCs did something


@pytest.mark.parametrize("eq", ["Euler", "laminar NS", "RANS"])
@pytest.mark.parametrize("second", [True, False])
def test_default_faces(eq, second):
    """synthetic default: wall kMin (Euler wall for Euler), symmetry jMin, far field elsewhere"""
    prm, hb = case(9, 8, 7, {"equationType": eq})
    _check(prm, hb, second)


@pytest.mark.parametrize("perm", [
    {IMIN: WALL, IMAX: FAR, JMIN: FAR, JMAX: SYMM, KMIN: FAR, KMAX: FAR},
    {IMIN: FAR, IMAX: WALL, JMIN: SYMM, JMAX: FAR, KMIN: FAR, KMAX: SYMM},
    {IMIN: SYMM, IMAX: SYMM, JMIN: WALL, JMAX: FAR, KMIN: FAR, KMAX: WALL},
    {IMIN: FAR, IMAX: FAR, JMIN: FAR, JMAX: WALL, KMIN: SYMM, KMAX: FAR},
])
def test_every_face_orientation(perm):
    prm, hb = case(8, 7, 9, {"equationType": "RANS"}, physical_faces=perm)
    _check(prm, hb, True)


@pytest.mark.parametrize("perm", [
    {IMIN: EXTRAP, IMAX: FAR, JMIN: SYMM, JMAX: FAR, KMIN: ISOWALL, KMAX: EXTRAP},
    {IMIN: ISOWALL, IMAX: EXTRAP, JMIN: EXTRAP, JMAX: ISOWALL, KMIN: FAR, KMAX: SYMM},
])
@pytest.mark.parametrize("treat", ["constant pressure extrapolation", "linear pressure extrapolation"])
def test_isothermal_wall_and_extrapolation(perm, treat):
    """bcNSWallIsoThermal :579-691 (BCData%TNS_Wall) and bcExtrap :1479-1570"""
    prm, hb = case(8, 7, 9, {"equationType": "RANS", "viscWallTreatment": treat}, physical_faces=perm)
    _check(prm, hb, True)
    _check(prm, hb, False)


@pytest.mark.parametrize("perm", [
    {IMIN: SUBIN, IMAX: SUBOUT, JMIN: SYMM, JMAX: FAR, KMIN: WALL, KMAX: SUPOUT},      # iMin: total conditions
    {IMIN: SUPIN, IMAX: SUPOUT, JMIN: SUBOUT, JMAX: SUBIN, KMIN: FAR, KMAX: WALL},     # jMax: mass flow
    {IMIN: SUBOUT, IMAX: SUBIN, JMIN: WALL, JMAX: SUPOUT, KMIN: SUBIN, KMAX: SUPIN},   # iMax mass flow, kMin total
])
@pytest.mark.parametrize("eq", ["Euler", "RANS"])
@pytest.mark.parametrize("flagset", [(0, 0), (1, 1)])
def test_inflow_outflow(perm, eq, flagset):
    """bcSubsonicOutflow :693-802, bcSubsonicInflow :804-1061 (totalConditions and massFlow, cpConstant),
    bcSupersonicInflow :1411-1477, bcExtrap for SupersonicOutflow with outflowTreatment"""
    prm, hb = case(8, 7, 9, {"equationType": eq}, physical_faces=perm)
    prm.hScalingInlet, prm.outflowLinearExtrapol = flagset
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    _check(prm, hb, True)
    _check(prm, hb, False)


@pytest.mark.parametrize("treat", ["constant pressure extrapolation", "linear pressure extrapolation"])
def test_wall_pressure_treatment(treat):
    prm, hb = case(8, 7, 9, {"equationType": "RANS", "viscWallTreatment": treat})
    _check(prm, hb, True)


@pytest.mark.parametrize("const_p", [0, 1])
def test_euler_wall(const_p):
    perm = {IMIN: FAR, IMAX: FAR, JMIN: SYMM, JMAX: FAR, KMIN: EULERWALL, KMAX: EULERWALL}
    prm, hb = case(8, 7, 9, {"equationType": "Euler"}, physical_faces=perm)
    prm.reserved = const_p
    _check(prm, hb, True)


@pytest.mark.parametrize("perm", [
    None,
    {IMIN: WALL, IMAX: FAR, JMIN: FAR, JMAX: SYMM, KMIN: FAR, KMAX: FAR},
    {IMIN: FAR, IMAX: WALL, JMIN: SYMM, JMAX: FAR, KMIN: FAR, KMAX: SYMM},
    {IMIN: SYMM, IMAX: FAR, JMIN: WALL, JMAX: FAR, KMIN: FAR, KMAX: WALL},
    {IMIN: EXTRAP, IMAX: FAR, JMIN: SYMM, JMAX: ISOWALL, KMIN: ISOWALL, KMAX: EXTRAP},
    {IMIN: SUBIN, IMAX: SUBOUT, JMIN: SUPIN, JMAX: SUPOUT, KMIN: WALL, KMAX: FAR},
    {IMIN: 11, IMAX: FAR, JMIN: SYMM, JMAX: 11, KMIN: WALL, KMAX: 11},   # polar symmetry: bcTurbSymm
])
@pytest.mark.parametrize("second", [True, False])
def test_turbulence_bcs(perm, second):
    """bcTurbTreatment + applyAllTurbBCThisBlock (src/turbulence/turbBCRoutines.F90:49-236, 662-797) with
    bcTurbWall / bcTurbSymm / bcTurbFarfield, bcEddyWall / bcEddyNoWall and turb2ndHalo"""
    from oracle.pyoracle import Oracle

    kw = {} if perm is None else {"physical_faces": perm}
    prm, hb = case(8, 7, 9, {"equationType": "RANS"}, **kw)
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)  # reference: viscous subfaces first
    ho = hb.copy()
    Oracle(ho, prm).apply_turb_bc(second)
    r = gold.run(lambda: (rb.call(hb, prm, "turbbcroutines_bcturbtreatment"),
                          rb.again("turbbcroutines_applyallturbbcthisblock", int(second)))[1])
    gold.same("w[5]", r, lambda r: r.a["w"][..., 5], ho.w[..., 5])
    gold.same("rev", r, lambda r: r.a["rev"], ho.rev)
    assert not np.array_equal(ho.w[..., 5], hb.w[..., 5])


@pytest.mark.parametrize("right_handed", [True, False])
def test_metrics_and_volumes(right_handed):
    """volume_block / metric_block (src/adjoint/adjointExtra.F90:5-298): cell volumes incl. halo cells and
    the face-normal arrays si/sj/sk from the node coordinates"""
    from oracle.pyoracle import Oracle

    prm, hb = case(9, 7, 8, {"equationType": "RANS"})
    if not right_handed:
        hb.x[..., 0] *= -1.0
        hb.right_handed = False
    ho = hb.copy()
    for n in ("vol", "si", "sj", "sk"):
        getattr(ho, n)[...] = 0.0
    o = Oracle(ho, prm)
    o.volume(); o.metrics()
    h2 = hb.copy()
    for n in ("vol", "si", "sj", "sk"):
        getattr(h2, n)[...] = 0.0
    r = gold.run(lambda: (rb.call(h2, prm, "adjointextra_volume_block"), rb.again("adjointextra_metric_block"))[1])
    d = hb.d
    c1 = (slice(1, d.ie + 1), slice(1, d.je + 1), slice(1, d.ke + 1))
    gold.same("vol", r, lambda r: r.a["vol"][c1], ho.vol[c1])
    for n in ("si", "sj", "sk"):
        sl = d.ref_slices(n) + (slice(None),)
        gold.same(n, r, lambda r: r.a[n][sl], getattr(ho, n)[sl])
        assert np.abs(getattr(ho, n)[sl]).max() > 0


@pytest.mark.parametrize("opt", [{"equationType": "Euler"}, {"equationType": "RANS"},
                                 {"equationType": "RANS", "discretization": "central plus matrix dissipation"},
                                 {"equationType": "laminar NS", "discretization": "upwind"}])
def test_reference_shock_sensor(opt):
    """referenceShockSensor (src/adjoint/adjointUtils.F90:1909-1969): pressure for Euler and matrix dissipation,
    entropy otherwise; compared on the cells the reference fills in every variant: those with at most one index in a
    halo (the pressure variants also fill the edge and corner halos)"""
    from oracle.pyoracle import Oracle

    prm, hb = case(9, 8, 7, opt)
    ho = hb.copy()
    Oracle(ho, prm).reference_shock_sensor()
    hb.shock[...] = -7.0
    r = gold.run(lambda: rb.call(hb, prm, "adjointutils_referenceshocksensor"))
    d = hb.d
    halo = [np.isin(np.arange(n + 1), (0, 1, n - 1, n)) for n in (d.ib, d.jb, d.kb)]
    one_halo = halo[0][:, None, None].astype(int) + halo[1][None, :, None] + halo[2][None, None, :] <= 1
    gold.same("shock sensor", r, lambda r: r.a["shocksensor"][one_halo], ho.shock[one_halo])   # -7.0 where not filled
    if r is not None:
        filled = r.a["shocksensor"] != -7.0
        assert np.array_equal(r.a["shocksensor"][filled], ho.shock[filled])


def test_residual_norms():
    """sumResiduals / sumAllResiduals (src/utils/utils.F90:6364-6459): the two monitored sums of getCurrentResidual"""
    import ctypes as C

    from oracle.pyoracle import Oracle

    prm, hb = case(9, 8, 7, {"equationType": "RANS"})
    o = Oracle(hb, prm)
    o.residual_core(8 | 16)
    want = o.norms()

    def reference():
        mon0 = (C.c_double * 16).in_dll(rb.lib(), "monloc")
        for q in range(16):
            mon0[q] = 0.0                            # monLoc accumulates
        rb.call(hb, prm, "sumresiduals", 1, 1)      # (nn = irho, mm = 1)
        rb.again("sumallresiduals", 2)
        return list((C.c_double * 16).in_dll(rb.lib(), "monloc"))[:2]

    gold.same("monLoc(1:2)", gold.run(reference), lambda mon: mon, want[:2])


SYMMPOLAR = 11


@pytest.mark.parametrize("perm", [
    {IMIN: SYMMPOLAR, IMAX: FAR, JMIN: SYMM, JMAX: FAR, KMIN: WALL, KMAX: FAR},
    {IMIN: FAR, IMAX: FAR, JMIN: FAR, JMAX: SYMMPOLAR, KMIN: FAR, KMAX: SYMMPOLAR},
    {IMIN: WALL, IMAX: SYMMPOLAR, JMIN: SYMMPOLAR, JMAX: FAR, KMIN: SYMMPOLAR, KMAX: FAR},
])
@pytest.mark.parametrize("second", [True, False])
def test_polar_symmetry(perm, second):
    """bcSymmPolar1stHalo / bcSymmPolar2ndHalo (BCRoutines.F90:332-486): mirror direction from the face diagonal
    xx(i+1,j+1) - xx(i,j) (setBCPointers with spatial pointers)"""
    prm, hb = case(8, 7, 9, {"equationType": "RANS"}, physical_faces=perm)
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    _check(prm, hb, second)
