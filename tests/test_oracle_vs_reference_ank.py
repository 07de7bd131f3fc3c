"""Pin the oracle's ANK pieces (oracle/adflow_oracle_ank.c) BIT FOR BIT against the reference's computeTimeStepBlock
and physicalityCheckANK (module ANKSolver, src/NKSolver/NKSolvers.F90), translated to C where the source lies
(oracle/_ref/anksolver_ref.c; PETSc vector access and the MPI reduction are replaced by plain arrays / a copy).  Where
the translated library is absent, against the recorded digests of its outputs (tests/refgold.py)."""
import ctypes as C

import numpy as np
import pytest

import refgold as gold
from adflow_b200.params import make_ank_params
from oracle import refblockette as rb
from oracle.pyoracle import Oracle

from util import case


def bind_ank(ank, nstate):
    L = rb.lib()
    for name, v in (("anksolver_ank_cfl", ank.cfl), ("anksolver_ank_cfllimit", ank.cflLimit), ("anksolver_ank_turbcflscale", ank.turbCFLScale),
                    ("anksolver_ank_physlstol", ank.physLSTol), ("anksolver_ank_physlstolturb", ank.physLSTolTurb),
                    ("anksolver_ank_stepmin", ank.stepMin), ("anksolver_ank_stepfactor", ank.stepFactor), ("ank_machinf", ank.machInf)):
        C.c_double.in_dll(L, name).value = v
    for name, v in (("anksolver_ank_coupled", ank.coupled), ("anksolver_nstate", nstate), ("ank_chartimestepcode", ank.charTimeStepType)):
        C.c_int.in_dll(L, name).value = v


@pytest.mark.parametrize("kind", ["None", "VLR", "Turkel"])
@pytest.mark.parametrize("options,coupled", [(None, False), (None, True), ({"equationType": "Euler"}, False)])
def test_time_step_block(kind, options, coupled):
    prm, hb = case(9, 8, 7, options)
    o = Oracle(hb, prm)
    o.time_step(True)
    o.call("orc_speed_of_sound", C.byref(prm))
    ank = make_ank_params(cfl=7.5, coupled=coupled, char_time_step=kind, mach=0.8, cflLimit=30.0, turbCFLScale=2.0)
    n = hb.nw if coupled else 5
    d = hb.d
    cells = [(2, 2, 2), (d.il, d.jl, d.kl), (5, 4, 3), (3, 7, 6)]

    def reference():
        rb.set_params(prm, hb.nw)
        r = rb.RefBlock(hb, prm)
        r.bind()
        bind_ank(ank, n)
        out = []
        for (i, j, k) in cells:
            ref = np.zeros((n, n), order="F")
            rb.lib().anksolver_computetimestepblock(C.byref(C.c_int(i)), C.byref(C.c_int(j)), C.byref(C.c_int(k)), ref.ctypes.data_as(C.c_void_p))
            out.append(ref)
        return out

    refs = gold.run(reference)
    for q, (i, j, k) in enumerate(cells):
        mine = o.ank_time_step_block(ank, i, j, k)
        assert np.isfinite(mine).all() and np.abs(mine).max() > 0
        gold.same("block %s" % ((i, j, k),), refs, lambda refs: refs[q], mine)


@pytest.mark.parametrize("coupled", [False, True])
def test_physicality_check(coupled):
    prm, hb = case(8, 7, 6)
    n = hb.nw if coupled else 5
    ow = hb.d.owned()
    ank = make_ank_params(coupled=coupled, physLSTol=0.2, physLSTolTurb=0.99, stepMin=0.01, stepFactor=1.0)
    wv = np.ascontiguousarray(np.transpose(hb.w[ow][..., :n], (2, 1, 0, 3)).reshape(-1))
    rng = np.random.default_rng(11)
    dv = rng.standard_normal(wv.size) * np.abs(wv) * 0.4
    if coupled:   # a few turbulence updates that would be more limiting than stepFactor * stepMin (clipped instead)
        dv[5::6][:40] = wv[5::6][:40] * 500.0
    for lam0 in (1.0, 0.05):
        d_mine = dv.copy()

        def reference():
            d_ref = dv.copy()
            rb.set_params(prm, hb.nw)
            r = rb.RefBlock(hb, prm)
            r.bind()
            bind_ank(ank, n)
            L = rb.lib()
            C.c_void_p.in_dll(L, "ank_wvec").value = wv.ctypes.data
            C.c_void_p.in_dll(L, "ank_dvec").value = d_ref.ctypes.data
            C.c_int.in_dll(L, "ank_nvec").value = wv.size
            lam = C.c_double(lam0)
            L.anksolver_physicalitycheckank(C.byref(lam))
            return lam.value, d_ref

        ref = gold.run(reference)
        mine = Oracle(hb, prm).ank_physicality_check(ank, wv, d_mine, lam0)
        gold.same("step", ref, lambda ref: ref[0], mine)
        assert 0.0 < mine <= lam0
        gold.same("update", ref, lambda ref: ref[1], d_mine)
        if coupled:
            assert np.abs(d_mine - dv).max() > 0   # the clip was exercised


def test_physicality_check_turb():
    """physicalityCheckANKTurb (NKSolvers.F90:3212-3335): the oracle against the translated routine, bit for bit"""
    prm, hb = case(8, 7, 6)
    ow = hb.d.owned()
    ank = make_ank_params(coupled=False, physLSTol=0.2, physLSTolTurb=0.99, stepMin=0.01, stepFactor=1.0)
    wv = np.ascontiguousarray(np.transpose(hb.w[ow][..., 5], (2, 1, 0)).reshape(-1))
    rng = np.random.default_rng(12)
    dv = rng.standard_normal(wv.size) * np.abs(wv) * 0.4
    dv[:40] = wv[:40] * 500.0     # updates more limiting than stepFactor * stepMin: clipped instead
    for lam0 in (1.0, 0.05):
        d_mine = dv.copy()

        def reference():
            d_ref = dv.copy()
            rb.set_params(prm, hb.nw)
            r = rb.RefBlock(hb, prm)
            r.bind()
            bind_ank(ank, 1)
            L = rb.lib()
            C.c_void_p.in_dll(L, "ank_wvec").value = wv.ctypes.data
            C.c_void_p.in_dll(L, "ank_dvec").value = d_ref.ctypes.data
            C.c_int.in_dll(L, "ank_nvec").value = wv.size
            lam = C.c_double(lam0)
            L.anksolver_physicalitycheckankturb(C.byref(lam))
            return lam.value, d_ref

        ref = gold.run(reference)
        f = Oracle(hb, prm).L.orc_ank_physicality_check_turb
        f.restype = C.c_double
        mine = f(C.byref(ank), C.c_long(wv.size), wv.ctypes.data_as(C.c_void_p), d_mine.ctypes.data_as(C.c_void_p), C.c_double(lam0))
        gold.same("step", ref, lambda ref: ref[0], mine)
        assert 0.0 < mine <= lam0
        gold.same("update", ref, lambda ref: ref[1], d_mine)
        assert np.abs(d_mine - dv).max() > 0
