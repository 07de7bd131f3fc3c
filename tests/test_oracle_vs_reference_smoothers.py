"""Pins the oracle's state preparation and smoother stages against the reference's own routines
(translated Fortran -> C, oracle/_ref, see test_oracle_vs_reference.py):

  flowUtils.F90   computePressureSimple, computeLamViscosity, computeEtotBlock
  turbUtils.F90   computeEddyViscosity / saEddyViscosity
  residuals.F90   residualAveraging :1785-2080, computeDwDADI :1038-1755 (+ tridiagSolve)
  smoothers.F90   executeRkStage :90-382, executeDADIStep :425-693

The stages end with the reference's own applyAllBC (BCRoutines.F90, also translated); setPointers and the
halo exchange whalo1/2 are no-op stubs (one block, no neighbours; oracle/ref_env.c).  Bit-exact; where the translated
library is absent, against the recorded digests of its outputs (tests/refgold.py).
"""
import numpy as np
import pytest

import refgold as gold
from oracle import refblockette as rb
from util import case


def _oracle(hb, prm):
    from oracle.pyoracle import Oracle

    ho = hb.copy()
    return ho, Oracle(ho, prm)


def _residual_state(shape, options, seed=314):
    """block with a freshly computed residual, time step and spectral radii (what the smoothers see)"""
    from oracle.pyoracle import Oracle

    prm, hb = case(*shape, options, seed=seed)
    o = Oracle(hb, prm)
    o.time_step(True)
    o.residual_block(1.0)
    hb.wn[...] = hb.w[..., :5]
    hb.pn[...] = hb.p
    return prm, hb


@pytest.mark.parametrize("eq", ["Euler", "laminar NS", "RANS"])
@pytest.mark.parametrize("halos", [0, 1])
def test_state_preparation(eq, halos):
    prm, hb = case(11, 9, 10, {"equationType": eq})
    d = hb.d
    ho, o = _oracle(hb, prm)
    o.pressure(bool(halos)); o.lam_viscosity(bool(halos)); o.eddy_viscosity(bool(halos))
    r = gold.run(lambda: rb.call(hb, prm, "flowutils_computepressuresimple", halos))
    gold.same("p", r, lambda r: r.a["p"], ho.p)
    hb2 = hb.copy(); hb2.p[...] = ho.p
    r = gold.run(lambda: rb.call(hb2, prm, "flowutils_computelamviscosity", halos))
    gold.same("rlv", r, lambda r: r.a["rlv"], ho.rlv)
    hb2.rlv[...] = ho.rlv
    r = gold.run(lambda: rb.call(hb2, prm, "turbutils_computeeddyviscosity", halos))
    gold.same("rev", r, lambda r: r.a["rev"], ho.rev)
    # computeEtotBlock over the owned range
    import ctypes as C
    o.L.orc_etot(C.byref(o.ob), C.byref(prm), 2, d.il, 2, d.jl, 2, d.kl)
    r = gold.run(lambda: rb.call(hb2, prm, "flowutils_computeetotblock", 2, d.il, 2, d.jl, 2, d.kl, 0))
    gold.same("rhoE", r, lambda r: r.a["w"][..., 4], ho.w[..., 4])


@pytest.mark.parametrize("shape", [(12, 9, 10), (5, 17, 6), (3, 3, 3)])
def test_residual_averaging(shape):
    prm, hb = _residual_state(shape, {"equationType": "RANS", "resAveraging": "always"})
    ho, o = _oracle(hb, prm)
    o.residual_averaging()
    r = gold.run(lambda: rb.call(hb, prm, "residuals_residualaveraging"))
    ow = hb.d.owned()
    gold.same("dw", r, lambda r: r.a["dw"][ow][..., :5], ho.dw[ow][..., :5])


@pytest.mark.parametrize("eq", ["Euler", "RANS"])
@pytest.mark.parametrize("stage", [1, 2, 5])
@pytest.mark.parametrize("avg", ["never", "alternate"])
def test_rk_stage(eq, stage, avg):
    prm, hb = _residual_state((12, 9, 10), {"equationType": eq, "resAveraging": avg})
    ho, o = _oracle(hb, prm)
    o.rk_stage(stage)
    r = gold.run(lambda: rb.call(hb, prm, "smoothers_executerkstage", rkstage=stage))
    for l in range(5):
        gold.same("w[%d]" % l, r, lambda r: r.a["w"][..., l], ho.w[..., l])  # whole box: owned cells and BC halos
    gold.same("p", r, lambda r: r.a["p"], ho.p)
    gold.same("rlv", r, lambda r: r.a["rlv"], ho.rlv)
    gold.same("rev", r, lambda r: r.a["rev"], ho.rev)


@pytest.mark.parametrize("eq", ["Euler", "laminar NS", "RANS"])
def test_compute_dw_dadi(eq):
    prm, hb = _residual_state((11, 10, 9), {"equationType": eq})
    ow = hb.d.owned()
    # executeDADIStep scales the residual by -cfl*dtl*vol before computeDwDADI
    hb.dw[ow + (slice(0, 5),)] *= (-prm.cfl * hb.dtl[ow] * hb.vol[ow])[..., None]
    ho, o = _oracle(hb, prm)
    o.compute_dw_dadi()
    r = gold.run(lambda: rb.call(hb, prm, "residuals_computedwdadi"))
    for l in range(5):
        gold.same("dw[%d]" % l, r, lambda r: r.a["dw"][ow][..., l], ho.dw[ow][..., l])


@pytest.mark.parametrize("eq", ["Euler", "RANS"])
@pytest.mark.parametrize("avg", ["never", "always"])
def test_dadi_step(eq, avg):
    prm, hb = _residual_state((10, 12, 9), {"equationType": eq, "resAveraging": avg, "smoother": "DADI"})
    ho, o = _oracle(hb, prm)
    o.dadi_step()
    r = gold.run(lambda: rb.call(hb, prm, "smoothers_executedadistep", rkstage=0))
    for l in range(5):
        gold.same("w[%d]" % l, r, lambda r: r.a["w"][..., l], ho.w[..., l])
    gold.same("p", r, lambda r: r.a["p"], ho.p)


@pytest.mark.parametrize("shape", [(12, 9, 10), (4, 15, 7)])
@pytest.mark.parametrize("opt", [{}, {"turbulenceOrder": "second order"}, {"turbulenceProduction": "vorticity"},
                                 {"useApproxSA": True}, {"useRotationSA": True}])
def test_sa_block_ddadi(shape, opt):
    """sa_block (src/turbulence/sa.F90:16-86): saSource, turbAdvection (turbUtils.F90:828-1553), saViscous,
    saResScale, saSolve (DD-ADI, :717-1267), saEddyViscosity, and the turbulence BC treatment around them
    (bcTurbTreatment / applyAllTurbBCThisBlock, src/turbulence/turbBCRoutines.F90)."""
    o_ = {"equationType": "RANS"}
    o_.update(opt)
    prm, hb = case(*shape, o_)
    from oracle.pyoracle import Oracle

    # the reference numbers the viscous-wall subfaces first (1..nViscBocos) and applies the turbulence BCs in
    # subface order, which decides the values of halo cells on block edges shared by two subfaces
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    ho = hb.copy()
    Oracle(ho, prm).sa_block()
    r = gold.run(lambda: rb.call(hb, prm, "sa_sa_block", 0))
    ow = hb.d.owned()
    gold.same("dw(itu1) after saResScale", r, lambda r: r.a["dw"][ow][..., 5], ho.dw[ow][..., 5])
    gold.same("nuTilde after the DD-ADI update and the turbulence BCs (whole box)", r, lambda r: r.a["w"][..., 5], ho.w[..., 5])
    gold.same("rev", r, lambda r: r.a["rev"], ho.rev)
    assert np.abs(ho.w[ow][..., 5] - hb.w[ow][..., 5]).max() > 0.0


@pytest.mark.parametrize("opt", [{"equationType": "Euler"}, {"equationType": "RANS"},
                                 {"equationType": "RANS", "discretization": "central plus matrix dissipation"},
                                 {"equationType": "laminar NS", "discretization": "upwind"}])
def test_block_residual_with_persistent_fw(opt):
    """initres_block + residual_block (src/solver/residuals.F90:4-346, 427-955) with the block flux routines of
    src/solver/fluxes.F90 over three Runge-Kutta stages: rFil = cdisRK(rkStage+1) = 1, 0, 0.56 -- the dissipative /
    viscous part fw persists between the stages and is blended with (1 - rFil)"""
    prm, hb = case(11, 9, 10, opt)
    from oracle.pyoracle import Oracle

    Oracle(hb, prm).time_step(True)        # spectral radii: inputs of the dissipation
    assert np.abs(hb.radI).max() > 0
    ho, o = _oracle(hb, prm)
    ho.fw[...] = 0.0
    first = True
    ow = hb.d.owned()
    for stage in (0, 1, 2):
        o.residual_block(prm.cdisRK[stage])

        def reference():
            if first:
                rb.call(hb, prm, "residuals_initres_block", 1, 5, 1, 1, rkstage=stage)
            else:
                rb.set_int("rkstage", stage)
                rb.again("residuals_initres_block", 1, 5, 1, 1)
            return rb.again("residuals_residual_block")

        r = gold.run(reference)
        first = False
        for l in range(5):
            gold.same("stage %d dw[%d]" % (stage, l), r, lambda r: r.a["dw"][ow][..., l], ho.dw[ow][..., l])
            gold.same("stage %d fw[%d]" % (stage, l), r, lambda r: r.a["fw"][ow][..., l], ho.fw[ow][..., l])


@pytest.mark.parametrize("opt", [{"equationType": "Euler", "nRKStages": 3}, {"equationType": "RANS"},
                                 {"equationType": "RANS", "resAveraging": "never", "nRKStages": 4},
                                 {"equationType": "laminar NS", "discretization": "central plus matrix dissipation"}])
def test_full_runge_kutta_cycle(opt):
    """RungeKuttaSmoother (src/solver/smoothers.F90:4-86) end to end: stage updates, residual averaging, the
    reference's own applyAllBC after every stage, initres + residual with the stage's cdisRK between the stages.
    Everything in the loop is the translated reference; only the halo exchange is a no-op (one block)."""
    prm, hb = _residual_state((12, 9, 10), opt)
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    hb.fw[...] = 0.0
    from oracle.pyoracle import Oracle

    Oracle(hb, prm).residual_block(prm.cdisRK[0])     # entry state of the smoother: residual of stage 0 incl. fw
    ho, o = _oracle(hb, prm)
    o.rk_smoother()
    r = gold.run(lambda: rb.call(hb, prm, "smoothers_rungekuttasmoother"))
    for l in range(5):
        gold.same("w[%d]" % l, r, lambda r: r.a["w"][..., l], ho.w[..., l])
    gold.same("p", r, lambda r: r.a["p"], ho.p)
    ow = hb.d.owned()
    gold.same("dw of the last residual", r, lambda r: r.a["dw"][ow][..., :5], ho.dw[ow][..., :5])
    assert np.abs(ho.w[ow][..., :5] - hb.w[ow][..., :5]).max() > 0


@pytest.mark.parametrize("opt", [{"equationType": "Euler"}, {"equationType": "RANS"}])
def test_full_dadi_smoother(opt):
    """DADISmoother (src/solver/smoothers.F90:383-421) with nSubiterations = 2: step, initres + residual (rFil = 1
    for smoother == DADI), step -- everything inside is the translated reference"""
    o_ = dict(opt)
    o_["smoother"] = "DADI"
    prm, hb = _residual_state((10, 12, 9), o_)
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    ho, o = _oracle(hb, prm)
    o.dadi_step(); o.residual_block(1.0); o.dadi_step()

    def reference():
        rb.set_params(prm, hb.nw)
        rb.set_int("smoother", 2); rb.set_int("nsubiterations", 2); rb.set_int("rkstage", 0)
        r = rb.RefBlock(hb, prm)
        r.bind()
        r.keep = rb.bind_bcs(hb, prm)
        rb._BOUND = r
        rb.lib().smoothers_dadismoother()
        rb.set_int("smoother", 1); rb.set_int("nsubiterations", 1)
        return r

    r = gold.run(reference)
    for l in range(5):
        gold.same("w[%d]" % l, r, lambda r: r.a["w"][..., l], ho.w[..., l])
    gold.same("p", r, lambda r: r.a["p"], ho.p)


@pytest.mark.parametrize("disc", ["central plus scalar dissipation", "central plus matrix dissipation", "upwind"])
@pytest.mark.parametrize("eq", ["Euler", "RANS"])
def test_time_step_block(disc, eq):
    """timeStep_block (src/solver/solverUtils.F90:43-355), the block twin used by the smoother loops: local time
    step for every discretisation; the spectral radii are stored only where the reference needs them (scalar
    dissipation, inputParamRoutines.F90:2824-2833)"""
    from oracle.pyoracle import Oracle

    prm, hb = case(9, 8, 7, {"equationType": eq, "discretization": disc})
    ho = hb.copy()
    Oracle(ho, prm).time_step(True)
    r = gold.run(lambda: rb.call(hb, prm, "solverutils_timestep_block", 0))
    d = hb.d
    gold.same("dtl", r, lambda r: r.a["dtl"][d.owned()], ho.dtl[d.owned()])
    if disc.startswith("central plus scalar"):
        c1 = (slice(1, d.ie + 1), slice(1, d.je + 1), slice(1, d.ke + 1))
        for ref, mine in (("radi", "radI"), ("radj", "radJ"), ("radk", "radK")):
            gold.same(ref, r, lambda r: r.a[ref][c1], getattr(ho, mine)[c1])


def test_smoothers_with_iblank():
    """blanked cells in the smoother stages: residual averaging (epz * max(iblank,0)), DADI (dual_dt * max(iblank,0))
    and the SA solve (rblank)"""
    from oracle.pyoracle import Oracle

    prm, hb = _residual_state((12, 9, 10), {"equationType": "RANS", "resAveraging": "always"})
    hb.iblank[4:7, 4:6, 3:5] = 0
    hb.iblank[8, 8, 6] = -1
    hb.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    Oracle(hb, prm).residual_block(1.0)
    ho, o = _oracle(hb, prm)
    o.rk_stage(1)
    r = gold.run(lambda: rb.call(hb, prm, "smoothers_executerkstage", rkstage=1))
    gold.same("w after the RK stage", r, lambda r: r.a["w"], ho.w)
    ho, o = _oracle(hb, prm)
    o.dadi_step()
    r = gold.run(lambda: rb.call(hb, prm, "smoothers_executedadistep", rkstage=0))
    gold.same("w after the DADI step", r, lambda r: r.a["w"], ho.w)
    ho, o = _oracle(hb, prm)
    o.sa_block()
    r = gold.run(lambda: rb.call(hb, prm, "sa_sa_block", 0))
    gold.same("nuTilde after sa_block", r, lambda r: r.a["w"][..., 5], ho.w[..., 5])
