"""Pins the CPU oracle (oracle/adflow_oracle*.c) against the REFERENCE'S OWN ROUTINES.

oracle/_ref/libblockette_ref.so is `src/NKSolver/blockette.F90` of /root/reference
(blocketteResCore :299-753 and every routine it calls, :854-6890), translated Fortran -> C by
oracle/f90toc.py from the source where it lies and compiled with gcc -O2 -ffp-contract=off.
The translation is statement for statement, so the comparison below is (and is asserted to be)
BIT-EXACT: same inputs, same operation order, IEEE double.

Runs without a GPU.  Where the library was not built, the oracle is held to the recorded digests of the reference's
outputs instead (tests/refgold.py).
"""
import numpy as np
import pytest

import refgold as gold
from oracle import refblockette as rb
from util import case

FLOW, TURB, INTERMED, DISS_APPROX, VISC_APPROX = 8, 16, 4, 1, 2


def _oracle(prm, hb, flags, rfil=1.0):
    from oracle.pyoracle import Oracle

    ho = hb.copy()
    Oracle(ho, prm).residual_core(flags, rfil)
    return ho


def _prepare(nx, ny, nz, options, **kw):
    from oracle.pyoracle import Oracle

    prm, hb = case(nx, ny, nz, options, **kw)
    # frozen shock sensor of the approximate-dissipation paths (blockette.F90:199-226): an INPUT
    # of blocketteResCore (bShockSensor), produced here by the oracle for both sides
    Oracle(hb, prm).reference_shock_sensor()
    return prm, hb


def _compare_dw(prm, hb, flags, rfil=1.0, lset=None):
    ho = _oracle(prm, hb, flags, rfil)
    r = gold.run(lambda: rb.residual_core(hb, prm, flags, rfil))
    ow = hb.d.owned()
    b = ho.dw[ow]
    if lset is None:
        lset = range(hb.nw)
    for l in lset:
        assert np.abs(b[..., l]).max() > 0.0
        gold.same("dw[%d]" % l, r, lambda r: r.a["dw"][ow][..., l], b[..., l])
    return r, ho


EQS = [("Euler", 5), ("laminar NS", 5), ("RANS", 6)]
DISCS = ["central plus scalar dissipation", "central plus matrix dissipation", "upwind"]


@pytest.mark.parametrize("eq,nw", EQS)
@pytest.mark.parametrize("disc", DISCS)
def test_exact_residual_matches_reference(eq, nw, disc):
    """full residual, every discretisation x equation set; block not a multiple of the 8^3 tile"""
    prm, hb = _prepare(13, 10, 9, {"equationType": eq, "discretization": disc})
    assert hb.nw == nw
    _compare_dw(prm, hb, FLOW | TURB)


@pytest.mark.parametrize("shape", [(8, 8, 8), (16, 8, 8), (17, 9, 8), (3, 2, 1), (1, 1, 1), (24, 5, 11)])
def test_tile_shapes(shape):
    """tile-boundary handling of blocketteResCore: exact multiples, ragged last tiles, tiny blocks"""
    prm, hb = _prepare(*shape, {"equationType": "RANS"})
    _compare_dw(prm, hb, FLOW | TURB)


@pytest.mark.parametrize("limiter", ["first order", "no limiter", "van Albada", "minmod"])
@pytest.mark.parametrize("eq", ["Euler", "RANS"])
def test_upwind_limiters(limiter, eq):
    """inviscidUpwindFlux :3341-4365 (leftRightState + riemannFlux, Roe, no preconditioner)"""
    prm, hb = _prepare(12, 9, 10, {"equationType": eq, "discretization": "upwind", "limiter": limiter})
    _compare_dw(prm, hb, FLOW | TURB)


@pytest.mark.parametrize("kappa", [-1.0, 0.0, 1.0 / 3.0])
def test_upwind_kappa(kappa):
    prm, hb = _prepare(9, 9, 9, {"equationType": "Euler", "discretization": "upwind", "kappaCoef": kappa})
    _compare_dw(prm, hb, FLOW | TURB)


@pytest.mark.parametrize("disc", DISCS)
@pytest.mark.parametrize("flags", [DISS_APPROX, VISC_APPROX, DISS_APPROX | VISC_APPROX])
def test_approximate_paths(disc, flags):
    """*Approx routines used by the ANK/NK preconditioner assembly (:4367-5166, :6467-6837)"""
    prm, hb = _prepare(11, 10, 9, {"equationType": "RANS", "discretization": disc})
    _compare_dw(prm, hb, FLOW | TURB | flags)


@pytest.mark.parametrize("opt", [
    {"turbulenceProduction": "vorticity"},
    {"useQCR": True},
    {"useRotationSA": True},
    {"useft2SA": False},
    {"useApproxSA": True},
    {"turbulenceOrder": "second order"},
    {"turbResScale": 1.0},
    {"vis2": 0.5, "vis4": 0.03},
    {"acousticScaleFactor": 0.7, "discretization": "central plus matrix dissipation"},
    {"dissipationScalingExponent": 0.5},
])
def test_sa_and_dissipation_options(opt):
    o = {"equationType": "RANS"}
    o.update(opt)
    prm, hb = _prepare(10, 9, 11, o)
    _compare_dw(prm, hb, FLOW | TURB)


def test_flow_only_and_turb_only():
    prm, hb = _prepare(10, 9, 9, {"equationType": "RANS"})
    _compare_dw(prm, hb, FLOW, lset=range(5))
    _compare_dw(prm, hb, TURB, lset=[5])


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_other_states(seed):
    prm, hb = _prepare(9, 10, 8, {"equationType": "RANS"}, seed=seed)
    _compare_dw(prm, hb, FLOW | TURB)


def test_left_handed_block():
    prm, hb = _prepare(9, 8, 10, {"equationType": "RANS"})
    # mirror the block: x -> -x makes it left handed; metrics/volumes are recomputed by make_block's
    # helpers so that si/sj/sk/vol stay consistent with x
    from adflow_b200 import synthetic as syn

    hb.x[..., 0] *= -1.0
    hb.right_handed = False
    syn.compute_metrics(hb)
    syn.compute_volumes(hb)
    _compare_dw(prm, hb, FLOW | TURB)


def test_intermediates_match_reference():
    """updateIntermed (:698-748): dtl, spectral radii, aa and the 12 nodal gradients"""
    prm, hb = _prepare(13, 10, 9, {"equationType": "RANS"})
    r, ho = _compare_dw(prm, hb, FLOW | TURB | INTERMED)
    d = hb.d
    ow = d.owned()
    c1 = (slice(1, d.ie + 1), slice(1, d.je + 1), slice(1, d.ke + 1))
    nd = (slice(1, d.il + 1), slice(1, d.jl + 1), slice(1, d.kl + 1))
    gold.same("dtl", r, lambda r: r.a["dtl"][ow], ho.dtl[ow])
    # radii / aa: the reference writes every tile's (1:ie) range, later tiles overwrite the overlap; the
    # values are point functions of the state so the overlap is consistent
    for ref, mine in (("radi", "radI"), ("radj", "radJ"), ("radk", "radK"), ("aa", "aa")):
        gold.same(ref, r, lambda r: r.a[ref][c1], getattr(ho, mine)[c1])
    for q, n in enumerate(["ux", "uy", "uz", "vx", "vy", "vz", "wx", "wy", "wz", "qx", "qy", "qz"]):
        gold.same(n, r, lambda r: r.a[n][nd], ho.grad[nd + (q,)])


@pytest.mark.parametrize("rfil", [0.56, 0.25])
@pytest.mark.parametrize("disc", DISCS)
def test_runge_kutta_dissipation_fraction(rfil, disc):
    """rFil (iteration module): fraction of new dissipation / viscous flux at intermediate RK stages"""
    prm, hb = _prepare(10, 9, 11, {"equationType": "RANS", "discretization": disc})
    _compare_dw(prm, hb, FLOW | TURB, rfil=rfil)


@pytest.mark.parametrize("disc", DISCS)
def test_iblank_holes_fringes_and_porosities(disc):
    """overset blanking (iblank 0 = hole, -1 = fringe: residual multiplied by max(iblank, 0)) and the three face
    porosities (normalFlux / boundFlux / noFlux) in the flux routines"""
    prm, hb = _prepare(12, 10, 9, {"equationType": "RANS", "discretization": disc})
    hb.iblank[4:7, 4:6, 3:5] = 0
    hb.iblank[8, 8, 6] = -1
    hb.iblank[2:4, 9, 2:5] = -1
    hb.porI[5, 3:6, 4:7] = -1     # noFlux
    hb.porJ[3:8, 6, 5] = 0        # boundFlux in the interior
    hb.porK[6, 7, 2:9] = -1
    _compare_dw(prm, hb, FLOW | TURB)
    _compare_dw(prm, hb, FLOW | TURB | DISS_APPROX | VISC_APPROX)
