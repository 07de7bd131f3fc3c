"""Pin the oracle's multigrid pieces (oracle/adflow_oracle_mg.c + the coarse-level branches of the smoother path)
BIT FOR BIT against the reference's own routines: transferToCoarseGrid, transferToFineGrid, setCornerRowHalos,
setCorrectionsCoarseHalos (src/solver/multiGrid.F90), inviscidDissFluxScalarCoarse (src/solver/fluxes.F90), the coarse
branches of initRes_block / residual_block / timeStep_block / executeRkStage / the wall BCs, translated to C where the
source lies (oracle/_ref).  Where the translated library is absent, against the recorded digests of its outputs
(tests/refgold.py)."""
import numpy as np
import pytest

import refgold as gold
from adflow_b200 import synthetic as syn
from oracle import refblockette as rb
from oracle.pyoracle import Oracle

from util import case

CASES = [((12, 8, 10), None), ((9, 7, 6), None), ((8, 6, 6), {"equationType": "Euler"}),
         ((6, 9, 5), {"equationType": "laminar NS"}),
         ((10, 8, 6), {"coarseDiscretization": "central plus matrix dissipation"}),
         ((10, 8, 6), {"coarseDiscretization": "upwind"}),
         ((8, 6, 6), {"equationType": "Euler", "discretization": "upwind", "coarseDiscretization": "upwind"})]


def two_levels(shape, options, seed=314):
    prm, fine = case(*shape, options, seed=seed)
    # the reference numbers the viscous wall subfaces first (nViscBocos); where subfaces share edge halos the order
    # of application matters (setCorrectionsCoarseHalos), so both sides use that order
    fine.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    coarse = syn.make_coarse_block(fine, prm)
    # halos of the fine block as the smoother leaves them
    o = Oracle(fine, prm)
    o.apply_turb_bc(True); o.apply_flow_bc(True)
    return prm, fine, coarse


def oracle_transfer_to_coarse(prm, fine, coarse):
    """transferToCoarseGrid (multiGrid.F90:5-324) composed from the oracle's pieces, one block per level"""
    of, oc = Oracle(fine, prm), Oracle(coarse, prm)
    of.time_step(False)                      # timeStep(.true.): only the spectral radii
    of.residual_block(prm.cdisRK[0])         # rkStage = 0 -> rFil = cdisRK(1); initres + residual
    oc.mg_restrict(of)
    oc.apply_flow_bc(False)                  # applyAllBC(.false.); whalo1: no neighbours
    oc.time_step(True)                       # timeStep(.false.)
    oc.mg_store_w1()
    oc.residual_block_coarse(prm.cdisRK[0], init=0)
    oc.mg_forcing()
    return of, oc


def eq(a, mg, pick, name):
    """a (the oracle's) against pick(mg), the reference's RefMG after the run"""
    assert np.isfinite(a).all(), name
    gold.same(name, mg, pick, a)


def run_mg(fine, coarse, prm, steps, **kw):
    """the translated reference on two (or more) grid levels: steps(mg), then the RefMG; None where it is absent"""
    def reference():
        mg = rb.RefMG(fine, coarse, prm, **kw)
        try:
            steps(mg)
        finally:
            mg.close()
        return mg

    return gold.run(reference)


@pytest.mark.parametrize("shape,options", CASES)
def test_transfer_to_coarse_grid(shape, options):
    prm, fine, coarse = two_levels(shape, options)
    f2, c2 = fine.copy(), coarse.copy()
    mg = run_mg(f2, c2, prm, lambda mg: mg.transfer_to_coarse())
    oracle_transfer_to_coarse(prm, fine, coarse)
    d, df = coarse.d, fine.d
    ow, owf = d.owned(), df.owned()
    c1 = (slice(1, d.ie + 1), slice(1, d.je + 1), slice(1, d.ke + 1))
    # dw, fw, dtl, radI/J/K, rlv of every level ARE the finest level's arrays in the reference (setPointers):
    # the coarse values sit in the fine arrays at the coarse indices
    eq(coarse.wr[ow], mg, lambda mg: mg.lv[2].a["wr"][ow], "wr (forcing term)")
    eq(coarse.dw[ow][..., :5], mg, lambda mg: mg.lv[1].a["dw"][ow][..., :5], "coarse dw")
    eq(coarse.w[c1][..., :5], mg, lambda mg: mg.lv[2].a["w"][c1][..., :5], "coarse w incl. first halos")
    eq(coarse.p[c1], mg, lambda mg: mg.lv[2].a["p"][c1], "coarse p")
    eq(coarse.w1[c1], mg, lambda mg: mg.lv[2].a["w1"][c1], "w1")
    eq(coarse.p1[c1], mg, lambda mg: mg.lv[2].a["p1"][c1], "p1")
    eq(coarse.dtl[ow], mg, lambda mg: mg.lv[1].a["dtl"][ow], "coarse dtl")
    for n, m in (("radI", "radi"), ("radJ", "radj"), ("radK", "radk")):
        eq(getattr(coarse, n)[c1], mg, lambda mg: mg.lv[1].a[m][c1], n)
    if prm.equations != 1:
        eq(coarse.rlv[c1], mg, lambda mg: mg.lv[1].a["rlv"][c1], "coarse rlv")
    if prm.equations == 3:
        eq(coarse.rev[c1], mg, lambda mg: mg.lv[2].a["rev"][c1], "coarse rev")


@pytest.mark.parametrize("shape,options", CASES[:3] + CASES[5:])
def test_coarse_level_rk_smoother(shape, options):
    """RungeKuttaSmoother on level 2: dw = wr start, cflCoarse, first-order dissipation, no second halos"""
    prm, fine, coarse = two_levels(shape, options)
    oracle_transfer_to_coarse(prm, fine, coarse)
    f2, c2 = fine.copy(), coarse.copy()
    mg = run_mg(f2, c2, prm, lambda mg: (mg.seed_coarse_shared(), mg.call(2, "smoothers_rungekuttasmoother")))
    Oracle(coarse, prm).rk_smoother()
    d = coarse.d
    c1 = (slice(1, d.ie + 1), slice(1, d.je + 1), slice(1, d.ke + 1))
    assert np.abs(coarse.w[d.owned()][..., :5] - c2.w[d.owned()][..., :5]).max() > 0
    eq(coarse.w[c1][..., :5], mg, lambda mg: mg.lv[2].a["w"][c1][..., :5], "coarse w after the RK cycle")
    eq(coarse.p[c1], mg, lambda mg: mg.lv[2].a["p"][c1], "coarse p after the RK cycle")
    eq(coarse.dw[d.owned()][..., :5], mg, lambda mg: mg.lv[1].a["dw"][d.owned()][..., :5], "coarse dw")


@pytest.mark.parametrize("shape,options", CASES)
@pytest.mark.parametrize("neumann", [0, 1])
def test_transfer_to_fine_grid(shape, options, neumann):
    prm, fine, coarse = two_levels(shape, options)
    prm.mgBoundCorr = neumann
    oracle_transfer_to_coarse(prm, fine, coarse)
    Oracle(coarse, prm).rk_smoother()        # something to interpolate
    f2, c2 = fine.copy(), coarse.copy()
    mg = run_mg(f2, c2, prm, lambda mg: mg.transfer_to_fine())
    of, oc = Oracle(fine, prm), Oracle(coarse, prm)
    of.mg_prolong(oc)
    of.apply_flow_bc(True)                   # applyAllBC(secondHalo = .true.); whalo2: no neighbours
    d, dc = fine.d, coarse.d
    c1c = (slice(1, dc.ie + 1), slice(1, dc.je + 1), slice(1, dc.ke + 1))
    eq(coarse.w[c1c][..., :5], mg, lambda mg: mg.lv[2].a["w"][c1c][..., :5], "corrections on the coarse block (incl. boundary halos)")
    eq(fine.dw[d.owned()][..., :5], mg, lambda mg: mg.lv[1].a["dw"][d.owned()][..., :5], "interpolated corrections")
    assert np.abs(fine.w[d.owned()][..., :5] - f2.w[d.owned()][..., :5]).max() > 0
    eq(fine.w[..., :5], mg, lambda mg: mg.lv[1].a["w"][..., :5], "fine w (whole box)")
    eq(fine.p, mg, lambda mg: mg.lv[1].a["p"], "fine p")
    if prm.equations != 1:
        eq(fine.rlv, mg, lambda mg: mg.lv[1].a["rlv"], "fine rlv")
    if prm.equations == 3:
        eq(fine.rev, mg, lambda mg: mg.lv[1].a["rev"], "fine rev")


@pytest.mark.parametrize("shape,options", CASES[:4])
def test_full_multigrid_start_up_transfer(shape, options):
    """transferToFineGrid(corrections = .false.), multiGrid.F90:326-654 with extrapolateSolution / extrapolateViscosities:
    the solution of the coarse ground level interpolated to the next finer level, halos extrapolated, turbulence + flow
    BCs (the flow BCs three times, as the reference does)"""
    prm, fine, coarse = two_levels(shape, options)
    oracle_transfer_to_coarse(prm, fine, coarse)
    Oracle(coarse, prm).rk_smoother()        # a coarse solution that differs from the restricted one
    rng = np.random.default_rng(5)
    fine.w[...] = fine.w * (1.0 + 0.05 * rng.standard_normal(fine.w.shape))   # the fine state is overwritten entirely
    f2, c2 = fine.copy(), coarse.copy()
    mg = run_mg(f2, c2, prm, lambda mg: mg.transfer_to_fine(corrections=False))
    of, oc = Oracle(fine, prm), Oracle(coarse, prm)
    of.mg_prolong_solution(oc)
    if prm.equations == 3:
        of.apply_turb_bc(True)
    of.apply_flow_bc(True); of.apply_flow_bc(True); of.apply_flow_bc(True)
    d, dc = fine.d, coarse.d
    c1c = (slice(1, dc.ie + 1), slice(1, dc.je + 1), slice(1, dc.ke + 1))
    eq(coarse.w[c1c], mg, lambda mg: mg.lv[2].a["w"][c1c], "coarse w with the pressure in place of rho*E (incl. boundary halos)")
    eq(fine.w, mg, lambda mg: mg.lv[1].a["w"], "fine w (whole box)")
    eq(fine.p, mg, lambda mg: mg.lv[1].a["p"], "fine p")
    if prm.equations != 1:
        eq(fine.rlv, mg, lambda mg: mg.lv[1].a["rlv"], "fine rlv")
    if prm.equations == 3:
        eq(fine.rev, mg, lambda mg: mg.lv[1].a["rev"], "fine rev")


@pytest.mark.parametrize("shape,options", CASES[:4])
def test_rk_smoother_on_a_coarse_ground_level(shape, options):
    """Full-multigrid start-up: RungeKuttaSmoother with currentLevel = groundLevel = 2.  The reference then runs the
    FINE-grid routines on the coarse block (second-order dissipation, dw = 0 start, second halos, eddy viscosity updated) with
    cflCoarse; the oracle does the same when the block carries level 1 and the parameters cfl = cflCoarse."""
    prm, fine, coarse = two_levels(shape, options)
    oracle_transfer_to_coarse(prm, fine, coarse)
    cfl = prm.cfl
    try:
        prm.cfl = prm.cflCoarse
        coarse.level = 1
        og = Oracle(coarse, prm)
        if prm.equations == 3:
            og.apply_turb_bc(True)
        og.apply_flow_bc(True)
        og.time_step(True)
        coarse.fw[...] = 0
        og.residual_block(prm.cdisRK[0])
        f2, c2 = fine.copy(), coarse.copy()
        c2.level = 2
        prm.cfl = cfl
        mg = run_mg(f2, c2, prm, lambda mg: (mg.seed_coarse_shared(), mg.call(2, "smoothers_rungekuttasmoother", ground=2)))
        prm.cfl = prm.cflCoarse
        w0 = coarse.w.copy()
        og.rk_smoother()
    finally:
        prm.cfl = cfl
        coarse.level = 2
    d = coarse.d
    assert np.abs(coarse.w[d.owned()][..., :5] - w0[d.owned()][..., :5]).max() > 0
    eq(coarse.w[..., :5], mg, lambda mg: mg.lv[2].a["w"][..., :5], "coarse-ground-level w after the RK cycle (whole box, second halos)")
    eq(coarse.p, mg, lambda mg: mg.lv[2].a["p"], "p")
    eq(coarse.dw[d.owned()][..., :5], mg, lambda mg: mg.lv[1].a["dw"][d.owned()][..., :5], "dw")
    if prm.equations == 3:
        eq(coarse.rev, mg, lambda mg: mg.lv[2].a["rev"], "rev")


def test_coarse_dissipation_and_corner_row_halos():
    prm, fine, coarse = two_levels((10, 8, 6), None)
    oracle_transfer_to_coarse(prm, fine, coarse)
    rng = np.random.default_rng(1)
    coarse.fw[...] = 1e-3 * rng.standard_normal(coarse.fw.shape)
    c2 = coarse.copy()

    def steps(mg):
        mg.seed_coarse_shared()
        rb._setd("rfil", 0.56)
        mg.call(2, "fluxes_invisciddissfluxscalarcoarse")
        mg.call(2, "multigrid_setcornerrowhalos", 5)

    mg = run_mg(fine.copy(), c2, prm, steps)
    oc = Oracle(coarse, prm)
    oc.diss_scalar_coarse(0.56)
    oc.mg_corner_row_halos()
    ow = coarse.d.owned()
    eq(coarse.fw[ow], mg, lambda mg: mg.lv[1].a["fw"][ow], "fw")
    eq(coarse.w[..., :5], mg, lambda mg: mg.lv[2].a["w"][..., :5], "w after the momentum round trip + corner row halos")
    eq(coarse.p, mg, lambda mg: mg.lv[2].a["p"], "p")


@pytest.mark.parametrize("shape,options", [((12, 8, 10), None), ((8, 6, 6), {"equationType": "Euler", "resAveraging": "always"})])
def test_coarse_level_dadi_smoother(shape, options):
    """DADISmoother on level 2: nSubiterations executeDADIStep with the coarse residual (dw = wr start) in between,
    cflCoarse, first halos only"""
    prm, fine, coarse = two_levels(shape, options)
    oracle_transfer_to_coarse(prm, fine, coarse)
    f2, c2 = fine.copy(), coarse.copy()

    def steps(mg):
        mg.seed_coarse_shared()
        rb.set_int("smoother", 2); rb.set_int("nsubiterations", 3); rb.set_int("rkstage", 0)
        try:
            mg.call(2, "smoothers_dadismoother")
        finally:
            rb.set_int("smoother", 1); rb.set_int("nsubiterations", 1)

    mg = run_mg(f2, c2, prm, steps)
    oc = Oracle(coarse, prm)
    for _ in range(2):
        oc.dadi_step()
        oc.residual_block(1.0)
    oc.dadi_step()
    d = coarse.d
    c1 = (slice(1, d.ie + 1), slice(1, d.je + 1), slice(1, d.ke + 1))
    assert np.abs(coarse.w[d.owned()][..., :5] - c2.w[d.owned()][..., :5]).max() > 0
    eq(coarse.w[c1][..., :5], mg, lambda mg: mg.lv[2].a["w"][c1][..., :5], "coarse w after the DADI step")
    eq(coarse.p[c1], mg, lambda mg: mg.lv[2].a["p"][c1], "coarse p after the DADI step")


def test_coarse_matrix_dissipation():
    """inviscidDissFluxMatrixCoarse (coarseDiscretization = matrix dissipation)"""
    prm, fine, coarse = two_levels((10, 8, 6), {"coarseDiscretization": "central plus matrix dissipation"})
    oracle_transfer_to_coarse(prm, fine, coarse)
    rng = np.random.default_rng(1)
    coarse.fw[...] = 1e-3 * rng.standard_normal(coarse.fw.shape)
    c2 = coarse.copy()

    def steps(mg):
        mg.seed_coarse_shared()
        rb._setd("rfil", 0.56)
        mg.call(2, "fluxes_invisciddissfluxmatrixcoarse")

    mg = run_mg(fine.copy(), c2, prm, steps)
    Oracle(coarse, prm).diss_matrix_coarse(0.56)
    ow = coarse.d.owned()
    assert np.abs(coarse.fw[ow] - c2.fw[ow]).max() > 0
    eq(coarse.fw[ow], mg, lambda mg: mg.lv[1].a["fw"][ow], "fw")


@pytest.mark.parametrize("shape,options,cycle,dadi_sub", [
    ((12, 8, 10), {"equationType": "laminar NS"}, "2v", 0),
    ((16, 12, 8), {"equationType": "Euler", "nRKStages": 3, "resAveraging": "never"}, "3w", 0),
    ((12, 8, 8), None, "2v", 0),                                   # RANS: turbSolveDDADI at the end of the cycle
    ((12, 12, 8), None, "3v", 0),
    ((12, 8, 8), {"equationType": "Euler", "smoother": "DADI", "resAveraging": "never"}, "2v", 2),
])
def test_execute_mg_cycle_driven_by_the_reference(shape, options, cycle, dadi_sub):
    """the reference's own driver executeMGCycle (multiGrid.F90:825-955, translated) runs the whole cycle -- its
    transferToCoarseGrid / RungeKuttaSmoother or DADISmoother / transferToFineGrid on every level, then turbSolveDDADI,
    timeStep and the residual -- and the composition of the oracle's pieces that tests/test_mg_gpu.py holds the device to
    (oracle_mg_cycle) has to reproduce it bit for bit: the ORDER of operations of adfb_mg_cycle is the reference's"""
    from adflow_b200.solver import ADFLOW_B200
    from test_mg_gpu import oracle_mg_cycle, prepare_fine

    nlev = int(cycle[0])
    prm, fine = case(*shape, options)
    fine.subfaces.sort(key=lambda s_: 0 if s_["bcType"] in (2, 6) else 1)
    o = Oracle(fine, prm)
    o.apply_turb_bc(True); o.apply_flow_bc(True)
    levels = [fine]
    for _ in range(nlev - 1):
        levels.append(syn.make_coarse_block(levels[-1], prm))
    prepare_fine(Oracle(fine, prm))
    cyc = ADFLOW_B200.cycleStrategy(cycle)
    ref_levels = [l.copy() for l in levels]
    mg = run_mg(ref_levels[0], ref_levels[1], prm,
                lambda mg: mg.execute_mg_cycle(cyc, smoother="DADI" if dadi_sub else "RK", n_subiterations=max(dadi_sub, 1)),
                more_levels=ref_levels[2:])
    w0 = fine.w.copy()
    oracle_mg_cycle(prm, levels, cyc, dadi_subiter=dadi_sub)
    ow = fine.d.owned()
    assert np.abs(fine.w[ow] - w0[ow]).max() > 0
    nv = fine.nw
    eq(fine.w[..., :nv], mg, lambda mg: mg.lv[1].a["w"][..., :nv], "fine state after the cycle (whole box)")
    eq(fine.p, mg, lambda mg: mg.lv[1].a["p"], "fine p")
    eq(fine.dw[ow][..., :5], mg, lambda mg: mg.lv[1].a["dw"][ow][..., :5], "fine residual after the cycle")
    if prm.equations == 3:
        eq(fine.rev, mg, lambda mg: mg.lv[1].a["rev"], "eddy viscosity")
