"""CUDA residual (through the C ABI) against the REFERENCE'S OWN blockette routines.

oracle/_ref/libblockette_ref.so = the reference's src/NKSolver/blockette.F90 translated to C
(oracle/f90toc.py) and compiled where the reference's source lies.  Where that library is absent,
the reference's residual is the oracle's once it matches the recorded digest of the reference's
output bit for bit (tests/refgold.py).  Tolerance as in test_residual_parity (north_star: 1e-10
relative; held to 1e-12)."""
import numpy as np
import pytest

import refgold as gold
from adflow_b200.solver import ADFLOW_B200, RES_FLOW, RES_SKIP_PREAMBLE, RES_TURB
from oracle import refblockette as rb

from util import case, rel_l2, rel_max

pytestmark = pytest.mark.gpu

TOL = 1e-12
DISS_APPROX, VISC_APPROX = 1, 2


def _cuda_dw(prm, hb, flags):
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        if flags & (DISS_APPROX | VISC_APPROX):
            s.referenceShockSensor()
        s.residual(flags | RES_SKIP_PREAMBLE)
        return s.downloadResidual(0)
    finally:
        s.close()


def _check(options, shape, flags=RES_FLOW | RES_TURB):
    from oracle.pyoracle import Oracle

    prm, hb = case(*shape, options)
    Oracle(hb, prm).reference_shock_sensor()
    r = gold.run(lambda: rb.residual_core(hb, prm, flags))
    ow = hb.d.owned()

    def oracle_dw():
        ho = hb.copy()
        Oracle(ho, prm).residual_core(flags)
        return ho.dw[ow]

    ref = gold.value("dw", r, lambda r: r.a["dw"][ow], oracle_dw)
    dw = _cuda_dw(prm, hb, flags)
    for l in range(hb.nw):
        a, b = dw[ow + (l,)], ref[..., l]
        assert np.isfinite(a).all()
        assert rel_l2(a, b) < TOL, "dw[%d] rel L2 %.3e" % (l, rel_l2(a, b))
        assert rel_max(a, b) < 10 * TOL, "dw[%d] rel max %.3e" % (l, rel_max(a, b))


@pytest.mark.parametrize("eq", ["Euler", "laminar NS", "RANS"])
@pytest.mark.parametrize("disc", ["central plus scalar dissipation", "central plus matrix dissipation", "upwind"])
def test_residual_vs_reference(cuda_lib, eq, disc):
    _check({"equationType": eq, "discretization": disc}, (21, 12, 10))


@pytest.mark.parametrize("shape", [(8, 8, 8), (17, 9, 8), (1, 1, 1), (40, 6, 5)])
def test_shapes_vs_reference(cuda_lib, shape):
    _check({"equationType": "RANS"}, shape)


@pytest.mark.parametrize("limiter", ["first order", "no limiter", "van Albada", "minmod"])
def test_upwind_limiters_vs_reference(cuda_lib, limiter):
    _check({"equationType": "RANS", "discretization": "upwind", "limiter": limiter}, (12, 9, 10))


@pytest.mark.parametrize("disc", ["central plus scalar dissipation", "central plus matrix dissipation"])
@pytest.mark.parametrize("flags", [DISS_APPROX, VISC_APPROX, DISS_APPROX | VISC_APPROX])
def test_approx_vs_reference(cuda_lib, disc, flags):
    _check({"equationType": "RANS", "discretization": disc}, (11, 10, 9), RES_FLOW | RES_TURB | flags)


@pytest.mark.parametrize("opt", [{"turbulenceProduction": "vorticity"}, {"useQCR": True}, {"useRotationSA": True},
                                 {"useft2SA": False}, {"useApproxSA": True}, {"turbulenceOrder": "second order"}])
def test_sa_options_vs_reference(cuda_lib, opt):
    o = {"equationType": "RANS"}
    o.update(opt)
    _check(o, (10, 9, 11))
