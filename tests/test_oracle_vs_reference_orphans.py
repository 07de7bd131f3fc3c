"""orphanAverage (src/utils/haloExchange.F90:201-354): the oracle's restatement against the reference's own routine
(translated where it lies, oracle/_ref), bit for bit -- including orphans on the block boundary, orphans next to other
blanked cells and an orphan without any valid neighbour (free-stream fall-back).  Where the translated library is absent,
against the recorded digests of its outputs (tests/refgold.py)."""
import ctypes as C

import numpy as np
import pytest

import refgold as gold
from oracle import refblockette as rb
from oracle.pyoracle import Oracle

from util import case


def orphan_case(seed=3):
    prm, hb = case(9, 8, 7, seed=seed)
    rng = np.random.default_rng(seed)
    d = hb.d
    orph = set()
    while len(orph) < 25:
        orph.add((int(rng.integers(0, d.ib + 1)), int(rng.integers(0, d.jb + 1)), int(rng.integers(0, d.kb + 1))))
    orph = sorted(orph)
    # one orphan whose six neighbours are all blanked: free-stream fall-back
    lone = (5, 4, 4)
    if lone not in orph:
        orph.append(lone)
    for (i, j, k) in orph:
        hb.iblank[i, j, k] = -1
    for di, dj, dk in ((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)):
        hb.iblank[lone[0] + di, lone[1] + dj, lone[2] + dk] = 0
    # a few more holes next to orphans
    for (i, j, k) in orph[:8]:
        if i + 1 <= d.ib and (i + 1, j, k) not in orph:
            hb.iblank[i + 1, j, k] = 0
    return prm, hb, np.array(orph, dtype=np.int32)


@pytest.mark.parametrize("args", [(1, 6, 1, 1, 1), (1, 5, 1, 1, 0), (6, 6, 0, 0, 1), (1, 5, 0, 0, 0)])
def test_orphan_average_matches_reference(args):
    w_start, w_end, calc_p, calc_lam, calc_eddy = args
    prm, hb, orph = orphan_case()
    mu_inf, ratio = 1.7e-3, 0.009
    ho = hb.copy()
    o = Oracle(ho, prm)
    flat = np.ascontiguousarray(orph.reshape(-1))
    o.L.orc_orphan_average(C.byref(o.ob), C.byref(prm), len(orph), flat.ctypes.data_as(C.c_void_p), w_start, w_end, calc_p, calc_lam,
                           calc_eddy, C.c_double(mu_inf), C.c_double(ratio))
    r = gold.run(lambda: rb.orphan_average(hb.copy(), prm, orph, w_start, w_end, calc_p, calc_lam, calc_eddy, mu_inf, ratio))
    for n in ("w", "p", "rlv", "rev"):
        gold.same(n, r, lambda r: r.a[n], getattr(ho, n))
    assert np.abs(ho.w - hb.w).max() > 0
    # the lone orphan took the free stream
    assert ho.w[5, 4, 4, w_start - 1] == prm.wInf[w_start - 1]
