"""The CUDA path at BASELINE.json's full single-GPU size (configs[1]: 96 x 72 x 64 = 442,368 cells).

The oracle still finishes this size in seconds, so the residual, one Runge-Kutta cycle, one DADI step, one
sa_block solve and one matrix-free product are compared with it directly; on top of that the size-independent
properties of the path are checked where no oracle is needed: free-stream preservation on the warped mesh,
partition independence (1 block == 2x2x2 blocks + halo exchange), and the residual norm reduced on the device
against the same norm recomputed on the host from the downloaded residual (checksum of checksums).

Tolerances: north_star's 1e-10 relative is the bar against the reference; the CUDA path keeps the oracle's
per-cell summation order and is held to 1e-12 on the residual, 1e-10 on state changes over a smoother cycle
(which divide by small differences), see test_residual_parity.py / test_smoother_parity.py."""
import numpy as np
import pytest

from adflow_b200 import make_params
from adflow_b200.halo import BlockGrid, build_cartesian_pattern, make_grid_blocks
from adflow_b200.solver import ADFLOW_B200, RES_FLOW, RES_TURB
from oracle.pyoracle import Oracle

from util import case, rel_l2, rel_max

pytestmark = pytest.mark.gpu

C2 = (96, 72, 64)


def _oracle_full_residual(prm, hb):
    ho = hb.copy()
    o = Oracle(ho, prm)
    o.pressure(False); o.lam_viscosity(False); o.eddy_viscosity(False)
    o.apply_turb_bc(True); o.apply_flow_bc(True)
    o.residual_core(RES_FLOW | RES_TURB)
    return ho, o


def test_c2_residual_matches_oracle_and_reference(cuda_lib):
    prm, hb = case(*C2)
    ho, o = _oracle_full_residual(prm, hb)
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        s.residual(RES_FLOW | RES_TURB)
        dw = s.downloadResidual(0)
        norms = s.getResNorms()
    finally:
        s.close()
    ow = hb.d.owned()
    for l in range(6):
        assert rel_l2(dw[ow + (l,)], ho.dw[ow + (l,)]) < 1e-12, l
        assert rel_max(dw[ow + (l,)], ho.dw[ow + (l,)]) < 1e-11, l
    rn = o.norms()
    assert abs(norms[0] - rn[0]) <= 1e-11 * rn[0] and abs(norms[1] - rn[1]) <= 1e-11 * rn[1]
    # checksum of checksums: the device reduction against the host reduction of the downloaded residual
    # (getCurrentResidual / setRVec scaling: dw / volRef, SA row * turbResScale)
    r = dw[ow] / hb.volRef[ow][..., None]
    host_rho = np.sum(r[..., 0] ** 2)      # the norms are returned squared (getCurrentResidual takes the root)
    r[..., 5] *= prm.turbResScale
    host_tot = np.sum(r ** 2)
    assert abs(norms[0] - host_rho) <= 1e-12 * host_rho
    assert abs(norms[1] - host_tot) <= 1e-12 * host_tot
    # the reference's own routines (where the translated library is absent: the oracle's residual, once it matches the
    # recorded digest of the reference's bit for bit)
    import refgold as gold
    from oracle import refblockette as rb

    def reference():
        hr = hb.copy()
        orr = Oracle(hr, prm)
        orr.pressure(False); orr.lam_viscosity(False); orr.eddy_viscosity(False)
        orr.apply_turb_bc(True); orr.apply_flow_bc(True)
        return rb.residual_core(hr, prm)

    rdw = gold.value("dw", gold.run(reference), lambda r: r.a["dw"][ow], ho.dw[ow])
    for l in range(6):
        assert rel_l2(dw[ow + (l,)], rdw[..., l]) < 1e-10, l


def test_c2_free_stream_preservation(cuda_lib):
    from test_oracle_invariants import freestream_block
    prm, hb = freestream_block(*C2)
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        from adflow_b200.solver import RES_SKIP_PREAMBLE
        s.residual(RES_FLOW | RES_TURB | RES_SKIP_PREAMBLE)
        dw = s.downloadResidual(0)
    finally:
        s.close()
    ow = hb.d.owned()
    scale = np.abs(hb.si[ow]).max() * prm.wInf[1] * prm.wInf[4]
    for l in range(5):
        assert np.abs(dw[ow + (l,)]).max() < 1e-13 * scale, l


def test_c2_partition_independence(cuda_lib):
    """The same global mesh and state as ONE block and as 2 x 2 x 2 blocks joined by the 1-to-1 exchange: every
    owned cell sees the same stencil values, so the residuals agree to round-off."""
    prm = make_params()
    res = {}
    # the synthetic state carries per-block noise: build the 8 blocks first and assemble the single block's owned
    # cells from theirs (the mesh is generated globally consistent)
    g8 = BlockGrid((2, 2, 2), tuple(c // 2 for c in C2), nranks=1)
    b8 = make_grid_blocks(g8, 0, prm)
    g1 = BlockGrid((1, 1, 1), C2, nranks=1)
    b1 = make_grid_blocks(g1, 0, prm)
    for q, b in enumerate(g8.local_blocks(0)):
        c = g8.coords[b]
        sl = tuple(slice(2 + c[a] * g8.n[a], 2 + (c[a] + 1) * g8.n[a]) for a in range(3))
        b1[0].w[sl] = b8[q].w[b8[q].d.owned()]
    for nb, grid, blocks in (((1, 1, 1), g1, b1), ((2, 2, 2), g8, b8)):
        n = grid.n
        s = ADFLOW_B200(prm)
        try:
            for hb in blocks:
                s.addBlock(hb)
            s.setCommPattern(build_cartesian_pattern(grid, 0))
            # blocketteRes applies the BCs before the exchange (like the reference): the BC halos on the edge between
            # a physical face and a block interface are computed from the interface halos of the PREVIOUS evaluation,
            # so the comparison is made on the second evaluation, when those hold the neighbour's current values
            s.residual(RES_FLOW | RES_TURB)
            s.residual(RES_FLOW | RES_TURB)
            g = np.zeros(C2 + (6,))
            for q, b in enumerate(grid.local_blocks(0)):
                c = grid.coords[b]
                sl = tuple(slice(c[a] * n[a], (c[a] + 1) * n[a]) for a in range(3))
                g[sl] = s.downloadResidual(q)[blocks[q].d.owned()]
            res[nb] = (g, s.getResNorms())
        finally:
            s.close()
    a, na = res[(1, 1, 1)]
    b, nb_ = res[(2, 2, 2)]
    for l in range(6):
        assert rel_max(b[..., l], a[..., l]) < 1e-12, (l, rel_max(b[..., l], a[..., l]))
    assert abs(na[1] - nb_[1]) <= 1e-12 * na[1]


@pytest.mark.parametrize("smoother", ["rk", "dadi"])
def test_c2_smoother_cycle_matches_oracle(cuda_lib, smoother):
    opts = {"nRKStages": 5, "resAveraging": "alternate"} if smoother == "rk" else {"smoother": "DADI", "resAveraging": "never"}
    prm, hb = case(*C2, opts)
    ho = hb.copy()
    o = Oracle(ho, prm)
    o.apply_turb_bc(True); o.apply_flow_bc(True)
    o.time_step(True)
    ho.fw[...] = 0
    o.residual_block(prm.cdisRK[0])
    if smoother == "rk":
        o.rk_smoother()
    else:
        o.dadi_step()
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        s.applyBCs(True, True)
        s.timeStep(False)
        s.smootherResidual(0)
        if smoother == "rk":
            s.rkCycle()
        else:
            s.dadiStep()
        w, p, rlv, rev = s.downloadState(0)
    finally:
        s.close()
    ow = hb.d.owned()
    dwv = w[ow] - hb.w[ow]
    dwo = ho.w[ow] - hb.w[ow]
    for l in range(5):
        assert np.abs(dwo[..., l]).max() > 0
        assert rel_l2(dwv[..., l], dwo[..., l]) < (1e-10 if smoother == "rk" else 1e-9), (l, rel_l2(dwv[..., l], dwo[..., l]))
    assert rel_max(p, ho.p) < 1e-11


def test_c2_sa_block_matches_oracle(cuda_lib):
    prm, hb = case(*C2)
    ho = hb.copy()
    o = Oracle(ho, prm)
    o.apply_turb_bc(True); o.apply_flow_bc(True)
    o.sa_block()
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        s.applyBCs(True, True)
        s.turbSolveDDADI(1)
        w, p, rlv, rev = s.downloadState(0)
    finally:
        s.close()
    ow = hb.d.owned()
    dv = w[ow + (5,)] - hb.w[ow + (5,)]
    do = ho.w[ow + (5,)] - hb.w[ow + (5,)]
    assert np.abs(do).max() > 0
    assert rel_l2(dv, do) < 1e-9, rel_l2(dv, do)
    assert rel_max(w[..., 5], ho.w[..., 5]) < 1e-10
    assert rel_max(rev[ow], ho.rev[ow]) < 1e-10


def test_c2_matrix_free_product_matches_oracle(cuda_lib):
    """MatMult of the NK shell matrix (NKSolvers.F90:295-302, PETSc MatMFFD) at full size: with a given h the
    product is the difference quotient of two FormFunction_mf evaluations of the oracle."""
    from test_mffd import state_vec
    from util import oracle_form_function
    prm, hb = case(*C2)
    U = state_vec(hb)
    a = np.random.default_rng(314).standard_normal(U.size) * np.abs(U).clip(1e-6)
    h = 1e-6
    F0 = oracle_form_function(prm, hb, U)
    yref = (oracle_form_function(prm, hb, U + h * a) - F0) / h
    s = ADFLOW_B200(prm)
    try:
        s.addBlock(hb)
        r = s.formFunction(U)
        s.mffdSetBase(U)
        y = s.mffdApply(a, h)
    finally:
        s.close()
    assert rel_l2(r, F0) < 1e-12
    assert rel_l2(y, yref) < 1e-6, rel_l2(y, yref)
