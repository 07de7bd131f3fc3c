#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (contract in the task brief).

Metric (BASELINE.json): Mcells/s of the RANS-SA residual.  A "step" is one full
residual evaluation (blocketteRes core: SA source/advection/diffusion, central +
scalar-JST + viscous fluxes, spectral radii/time step) of every local block.

Workload at N=1: BASELINE configs[1] -- one 96x72x64 = 442 368-cell RANS-SA
block ("MDO tutorial wing RANS-SA, 450k cells, 1 block"), synthetic mesh/state
(adflow_b200/synthetic.py, seed 314).  N>1 (weak scaling): one such block per
GPU in a Cartesian arrangement with 2-layer 1-to-1 halos exchanged by NCCL
send/recv over NVLink inside every step.

  step  : adfb_residual = blocketteRes (p/rlv/rev, turbulence+flow BCs, halo exchange, core)
  value : whole-job Mcells/s with inputs resident in HBM, timed per step with CUDA
          events on the library's stream; L2 is flushed (256 MiB memset) before
          every timed step.
  e2e   : same metric through the public vector API with HOST buffers
          (setStates -> residual incl. p/rlv/rev preamble -> getRes): pinned host
          state vector H2D and residual vector D2H inside the timed region.
  roofline : HBM; achieved = 176 B/cell (SURVEY 8d, RANS-SA residual, algorithmic)
          x cells / summed duration of the residual's kernels (CUDA events around
          each launch, separate pass); peak from MEASURED_PEAKS.json.
  cpu_baseline : the oracle port (C restatement of the reference algorithm,
          -O3 -march=native -ffast-math like the reference's gfortran flags) on 1 core.

--impl reference times that same CPU restatement using all host cores (one
sub-block per process, the reference's MPI-rank-per-block model); the reference
Fortran itself cannot be built in this image (no Fortran/MPI/PETSc/CGNS).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2 = (96, 72, 64)
# DRAM traffic of one residual step on C2 measured by ncu (profiles/r02_ncu_summary.md: sum over the four residual kernels
# k_state_prep + k_sa + k_prep + k_flowres; round 1 had 568.1e6 over six kernels)
NCU_TRAFFIC_BYTES = 403.6e6
NCU_TRAFFIC_NOTE = ("dram__bytes_read.sum + dram__bytes_write.sum summed over the residual kernels of one step, ncu --set full capture "
                    "(profiles/)")
# the second roof (SURVEY section 7 'report both'): the path is FP64-issue bound long before it is HBM bound
FP64_ROOF = {"note": "B200 FP64 pipe: 64 DFMA lanes / SM / clk x 148 SMs x 1.965 GHz = 18.6 T FP64 instructions/s (37 TFLOP/s); "
                     "percentages of the dominant kernel k_flowres from the ncu --set full capture profiles/r02_ncu_summary.md", "fp64_pipe_pct": 23.9, "issue_active_pct": 27.9}
BYTES_PER_CELL = 176.0  # SURVEY.md 8(d): RANS-SA residual, metrics from x, algorithmic
METRIC = "Mcells/s RANS-SA residual"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.lines, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


KIND_NOTE = {
    "reference": "oracle/_ref: the reference's src/NKSolver/blockette.F90 translated to C, gcc -O3 -ffast-math",
    "port": "oracle port (C restatement), gcc -O3 -march=native -ffast-math",
}


def _cpu_core_runner(hb, prm):
    """callable running the reference's blocketteResCore once on `hb`, and its kind:
    "reference" = oracle/_ref (the reference's own blockette.F90 translated to C and built with
    -O3 -ffast-math like config.LINUX_GFORTRAN.mk), else "port" = the oracle restatement."""
    from oracle import refblockette as rb

    if rb.available(fast=True):
        rb.use_fast(True)
        rb.residual_core(hb, prm, 8 | 16)
        return (lambda: rb.call_core(8 | 16)), "reference"
    from oracle.pyoracle import Oracle

    o = Oracle(hb, prm, fast=True)
    return (lambda: o.residual_core(8 | 16)), "port"


def cpu_baseline_single(shape, reps_budget_s=12.0):
    """Reference CPU path on ONE core over the full C2 block; returns (Mcells/s, reps, kind)."""
    from adflow_b200 import make_params
    from adflow_b200 import synthetic as syn

    prm = make_params()
    hb = syn.make_block(*shape, prm)
    run, kind = _cpu_core_runner(hb, prm)
    run()  # warm-up
    t0 = time.perf_counter()
    reps = 0
    while True:
        run()
        reps += 1
        if time.perf_counter() - t0 > reps_budget_s or reps >= 20:
            break
    dt = time.perf_counter() - t0
    return hb.d.ncells * reps / dt / 1e6, reps, kind


def _ref_worker(args):
    shape, origin, gshape, reps, tag = args
    os.environ["OMP_NUM_THREADS"] = "1"
    from adflow_b200 import make_params
    from adflow_b200 import synthetic as syn

    prm = make_params()
    hb = syn.make_block(*shape, prm, origin=origin, global_n=gshape, origin_tag=tag)
    run, kind = _cpu_core_runner(hb, prm)
    run()
    t0 = time.perf_counter()
    for _ in range(reps):
        run()
    return time.perf_counter() - t0, hb.d.ncells, kind


def _split_parts(ncores, ny, nz):
    """(pj, pk): sub-block grid of the C2 block over the host cores, at least 4 cells per sub-block and direction"""
    best = (1, 1)
    for pk in range(1, nz // 4 + 1):
        for pj in range(1, ny // 4 + 1):
            if pj * pk <= ncores and pj * pk > best[0] * best[1]:
                best = (pj, pk)
    return best


def run_reference(args):
    """--impl reference: the reference's own blocketteResCore (oracle/_ref; else the oracle port) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp

    from oracle import refblockette as rb

    if rb.available(fast=True):
        rb.use_fast(True)   # the parent maps the library too: it is what the workers run (driver-side .so record)
    ncores = len(os.sched_getaffinity(0))
    nx, ny, nz = C2
    # the block is split along j and k into one sub-block per core, like the reference's load balancer splits a block
    # over MPI ranks (loadBalance.F90:2790); an N-GPU job is compared with N such blocks on the same host cores
    nblocks = max(1, args.gpus)
    reps = max(1, 3 // nblocks) if nblocks > 1 else 3
    ctx = mp.get_context("spawn")

    def jobs_for(pj, pk, r):
        js = [ny * q // pj for q in range(pj + 1)]
        ks = [nz * q // pk for q in range(pk + 1)]
        return [((nx, js[a + 1] - js[a], ks[q + 1] - ks[q]), (0, js[a], ks[q]), C2, r, q * pj + a) for q in range(pk) for a in range(pj)]

    # one process per sub-block; more sub-blocks use more cores but carry more halo cells (2 layers per cut) and more
    # memory traffic per owned cell, so the split is calibrated on this host: candidates up to one process per core, one
    # step each, the fastest is measured
    cands = []
    for want in (16, 32, 64, ncores):
        c = _split_parts(min(want, ncores), ny, nz)
        if c not in cands:
            cands.append(c)
    calib = {}
    for (pj, pk) in cands:
        pool = ctx.Pool(pj * pk)
        try:
            pool.map(_ref_worker, jobs_for(pj, pk, 1))          # start-up + warm-up
            out = pool.map(_ref_worker, jobs_for(pj, pk, 1))
            calib[(pj, pk)] = max(o[0] for o in out)
        finally:
            pool.close()
            pool.join()
    pj, pk = min(calib, key=calib.get)
    parts = pj * pk
    jobs = jobs_for(pj, pk, reps * nblocks)
    step_ms = []
    pool = ctx.Pool(parts)
    try:
        for _ in range(args.warmup):
            pool.map(_ref_worker, jobs)
        for _ in range(args.steps):
            out = pool.map(_ref_worker, jobs)
            wall = max(o[0] for o in out)  # slowest rank, like an MPI barrier
            step_ms.append(wall * 1e3 / reps)   # one step = one residual of all nblocks blocks
    finally:
        pool.close()
        pool.join()
    cells = nx * ny * nz * nblocks
    ms = sum(step_ms) / len(step_ms)
    val = cells / (ms * 1e-3) / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mcells/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(C2, nblocks), "cells": cells,
                   "note": "CPU arm: residual core (blocketteResCore) of %d C2 block(s), each split %d x %d (j x k) over the host cores; "
                           "the host does not grow with --gpus; split calibrated over %s (s per step)" % (nblocks, pj, pk, {"%dx%d" % k: round(v, 3) for k, v in calib.items()})},
        "cpu_baseline": {"value": val, "unit": "Mcells/s", "cores": parts, "kind": out[0][2],
                         "sample": "%d residual evaluations (blocketteResCore) of %d C2 block(s) per step, %d sub-blocks "
                                   "(1 per core, one process each, %d host cores visible), %s" % (reps, nblocks, parts, ncores, KIND_NOTE[out[0][2]])},
        "e2e": {"value": val, "unit": "Mcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, s, blocks, block_ids, nblocks_total, with_norms, np):
    """What the timed step hands its caller: the residual dw of every owned cell of each block (float64, layout
    (i, j, k, variable)) and the two residual norms.  A block whose dw exceeds its share of the 64 MiB budget is
    written as a fixed sample: flat indices drawn with seed 0, sorted; the same sample for every build."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BUDGET_BYTES // nblocks_total - 4096
    for q, (hb, b) in enumerate(zip(blocks, block_ids)):
        dw = np.ascontiguousarray(s.downloadResidual(q)[hb.d.owned()], dtype=np.float64)
        if dw.nbytes > share:
            pick = np.sort(np.random.default_rng(0).choice(dw.size, share // 8, replace=False))
            np.save(os.path.join(out_dir, "residual_block%d_sample.npy" % b), dw.reshape(-1)[pick])
        else:
            np.save(os.path.join(out_dir, "residual_block%d.npy" % b), dw)
    norms = np.asarray(s.getResNorms(), dtype=np.float64)   # every rank: the norms are reduced over the job
    if with_norms:
        np.save(os.path.join(out_dir, "residual_norms.npy"), norms)


def workload_name(shape, nblocks):
    return "C2 %dx%dx%d RANS-SA residual (blocketteRes), %d block(s)" % (tuple(shape) + (nblocks,))


def _event_ms(torch, stream, fn, n):
    """mean device time of fn over n calls: CUDA events on the library stream"""
    with torch.cuda.stream(stream):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        e1.synchronize()
    return e0.elapsed_time(e1) / n


def _gather_ms(torch, dist, world, ms):
    """per-rank values and their max"""
    if world == 1:
        return [ms], ms
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    v = [float(x[0]) for x in out]
    return v, max(v)


def halo_data_check(s, blocks, pat, np, torch=None, dist=None):
    """Data-plane check of the 1-to-1 exchange (NCCL between ranks, copies inside a rank): every listed halo cell is
    poisoned on the device, the library exchanges, and each halo cell must then hold exactly the donor cell's value.
    The expected values travel independently of the library: same-rank donors are read from the host copy, other ranks'
    donors are sent with torch.distributed point-to-point in the order of the send lists.  Returns (checked, bad)."""
    saved = []
    for q, hb in enumerate(blocks):
        w0, p0 = hb.w.copy(), hb.p.copy()
        saved.append((w0, p0))
        ow = hb.d.owned()
        wp = np.full_like(hb.w, -7.5e3); pp = np.full_like(hb.p, -7.5e3)
        wp[ow] = w0[ow]; pp[ow] = p0[ow]
        hb.w[...] = wp; hb.p[...] = pp
        s.uploadState(q, hb, with_visc=False)
    s.haloExchange(comm_viscous=False)
    got = [s.downloadState(q)[:2] for q in range(len(blocks))]

    def values(src, lst):   # (n, nw+1): w(1:nw), p of the listed cells, list order
        out = np.empty((len(lst), blocks[0].nw + 1))
        for q in np.unique(lst[:, 0]):
            sel = lst[:, 0] == q
            i, j, k = lst[sel, 1], lst[sel, 2], lst[sel, 3]
            out[sel, :-1] = src[q][0][i, j, k, :]
            out[sel, -1] = src[q][1][i, j, k]
        return out

    checked = bad = 0
    dl, hl = pat["donorList"].reshape(-1, 4), pat["haloList"].reshape(-1, 4)
    if len(hl):
        checked += len(hl)
        bad += int((values(got, hl) != values(saved, dl)).any(axis=1).sum())
    sl, rl = pat["sendList"].reshape(-1, 4), pat["recvList"].reshape(-1, 4)
    if len(pat["nbrRank"]):
        send_all = torch.from_numpy(values(saved, sl)).cuda()
        recv_all = torch.empty((len(rl), blocks[0].nw + 1), dtype=torch.float64, device="cuda")
        ops, so, ro = [], 0, 0
        for m, peer in enumerate(pat["nbrRank"]):
            ns, nr = int(pat["sendCount"][m]), int(pat["recvCount"][m])
            if ns:
                ops.append(dist.P2POp(dist.isend, send_all[so:so + ns].contiguous(), int(peer)))
            if nr:
                ops.append(dist.P2POp(dist.irecv, recv_all[ro:ro + nr], int(peer)))
            so += ns; ro += nr
        for r in dist.batch_isend_irecv(ops):
            r.wait()
        torch.cuda.synchronize()
        checked += len(rl)
        bad += int((values(got, rl) != recv_all.cpu().numpy()).any(axis=1).sum())
    for q, hb in enumerate(blocks):
        hb.w[...], hb.p[...] = saved[q]
        s.uploadState(q, hb)
    return checked, bad


# residual norms of the C3 8-block case after one 5-stage RK cycle from the synthetic state, measured at N = 1 (all
# eight blocks on one GPU): every other distribution of the same blocks must reproduce them (partition independence,
# the reference's analogue: tests/reg_tests/test_functionals.py:24-58).  None = not recorded yet.
C3_REF_NORMS = (1233939870.9755895, 26154234242.979332)   # measured at N = 1 (8 blocks on one B200), round 2


def strong_scaling_c3(args, torch, dist, rank, world, local, fresh_uid, np):
    """BASELINE config 3: 8 blocks x 128x128x64 (2x2x2 arrangement, 1-to-1 halos), 8/N blocks per GPU; a step is one
    5-stage Runge-Kutta cycle (RungeKuttaSmoother, src/solver/smoothers.F90:4-86) incl. the halo exchanges of every stage."""
    from adflow_b200 import make_params
    from adflow_b200.halo import BlockGrid, build_cartesian_pattern, make_grid_blocks
    from adflow_b200.solver import ADFLOW_B200, RES_FLOW, RES_TURB

    shape = (128, 128, 64)
    if 8 % world:
        return {"skipped": "8 blocks do not divide over %d ranks" % world}
    prm = make_params()
    grid = BlockGrid((2, 2, 2), shape, nranks=world)
    blocks = make_grid_blocks(grid, rank, prm)
    pat = build_cartesian_pattern(grid, rank)
    s = ADFLOW_B200(prm, device=local, rank=rank, nranks=world, unique_id=fresh_uid())
    out = {}
    try:
        for hb in blocks:
            s.addBlock(hb)
        s.setCommPattern(pat)
        stream = torch.cuda.ExternalStream(s.L.adfb_stream(), device=local)
        checked, bad = halo_data_check(s, blocks, pat, np, torch, dist)
        if world > 1:
            t = torch.tensor([checked, bad], dtype=torch.int64, device="cuda")
            dist.all_reduce(t)
            checked, bad = int(t[0]), int(t[1])
        # partition independence of the result: one cycle from the synthetic state, then the residual norms
        s.applyBCs(True, True)
        s.haloExchange()
        s.timeStep(False)
        s.smootherResidual(0)
        s.rkCycle()
        s.residual(RES_FLOW | RES_TURB)
        norms = [float(x) for x in s.getResNorms()]
        ok = bad == 0
        rel = None
        if C3_REF_NORMS is not None:
            rel = max(abs(a - b) / b for a, b in zip(norms, C3_REF_NORMS))
            ok = ok and rel < 1e-10
        # timing
        nrep = max(3, min(10, args.steps))
        for _ in range(3):
            s.rkCycle()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = _event_ms(torch, stream, lambda: s.rkCycle(), nrep)
        per_rank, ms_max = _gather_ms(torch, dist, world, ms)
        msx = _event_ms(torch, stream, lambda: s.haloExchange(), nrep)
        per_rank_x, msx_max = _gather_ms(torch, dist, world, msx)
        cells = 8 * shape[0] * shape[1] * shape[2]
        out = {
            "workload": "C3: 8 blocks x 128x128x64 RANS-SA (2x2x2), one 5-stage RK cycle per step incl. 5 halo exchanges",
            "scaling": "strong", "n_gpus": world, "blocks_per_gpu": 8 // world, "cells": cells,
            "ms_per_cycle": ms_max, "Mcells/s": cells / (ms_max * 1e-3) / 1e6, "ms_per_rank": per_rank,
            "exchange_only_ms": msx_max, "exchange_only_ms_per_rank": per_rank_x,
            "exchange_share_of_cycle": 5.0 * msx_max / ms_max,
            "halo_check": "ok" if ok else "FAILED",
            "halo_cells_checked": checked, "halo_cells_wrong": bad,
            "res_norms_after_one_cycle": norms, "norms_rel_diff_vs_n1": rel,
            "timing": "CUDA events on the library stream, max over ranks; blocks (1.4 GB each) exceed L2",
        }
    finally:
        s.close()
    return out


def nk_matvec_c5(args, torch, dist, rank, world, local, fresh_uid, np, peak):
    """BASELINE config 5 (per-GPU share): one 160x160x144 block per GPU (N = 8: the 29.5 M-cell case), matrix-free
    Jacobian-vector products y = (F(U + h a) - F(U)) / h of the NK solver (FormFunction_mf, NKSolvers.F90:437) with
    device-resident vectors; a sweep of 60 products, halo exchange inside every residual."""
    from adflow_b200 import make_params
    from adflow_b200.halo import BlockGrid, build_cartesian_pattern, make_grid_blocks
    from adflow_b200.solver import ADFLOW_B200

    shape = (160, 160, 144)
    prm = make_params()
    nb = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}.get(world, (world, 1, 1))
    grid = BlockGrid(nb, shape, nranks=world)
    blocks = make_grid_blocks(grid, rank, prm)
    s = ADFLOW_B200(prm, device=local, rank=rank, nranks=world, unique_id=fresh_uid())
    try:
        for hb in blocks:
            s.addBlock(hb)
        s.setCommPattern(build_cartesian_pattern(grid, rank))
        stream = torch.cuda.ExternalStream(s.L.adfb_stream(), device=local)
        U = s.getStates()
        s.mffdSetBase(U)
        da = torch.from_numpy(np.random.default_rng(7 + rank).standard_normal(U.size)).cuda()
        dy = torch.empty_like(da)
        for _ in range(3):
            s.mffdApplyDevice(da.data_ptr(), dy.data_ptr(), da.numel(), 1e-7)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        nmv = 60
        ms = _event_ms(torch, stream, lambda: s.mffdApplyDevice(da.data_ptr(), dy.data_ptr(), da.numel(), 1e-7), nmv)
        per_rank, ms_max = _gather_ms(torch, dist, world, ms)
        finite = bool(torch.isfinite(dy).all())
        cells = shape[0] * shape[1] * shape[2] * world
        gbs = 464.0 * cells / (ms_max * 1e-3) / 1e9
        return {
            "workload": "C5 share: one 160x160x144 RANS-SA block per GPU, sweep of %d matrix-free Jacobian-vector products, vectors on the GPU" % nmv,
            "scaling": "weak", "n_gpus": world, "cells": cells, "ms_per_matvec": ms_max, "ms_per_rank": per_rank,
            "Mcells/s": cells / (ms_max * 1e-3) / 1e6, "GB/s": gbs, "algorithmic_bytes_per_cell": 464.0,
            "frac_of_hbm_peak": gbs / (peak * world),
            "frac_of_hbm_peak_fused_272B": 272.0 * cells / (ms_max * 1e-3) / 1e9 / (peak * world),
            "result_finite": finite,
        }
    finally:
        s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shape", type=int, nargs=3, default=list(C2))
    ap.add_argument("--no-scaling-sections", action="store_true", help="skip the C3 strong-scaling and C5 matvec sections")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)

    from adflow_b200 import make_params
    from adflow_b200 import synthetic as syn
    from adflow_b200.solver import ADFLOW_B200, RES_FLOW, RES_SKIP_PREAMBLE, RES_TURB

    from adflow_b200.halo import BlockGrid, build_cartesian_pattern, make_grid_blocks

    shape = tuple(args.shape)
    prm = make_params()
    # one C2-sized block per GPU in a (2,2,2)-style Cartesian arrangement; physical BCs
    # (wall kMin, symmetry jMin, far field) on the outer faces, 1-to-1 halos inside
    nb = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}.get(world, (world, 1, 1))
    grid = BlockGrid(nb, shape, nranks=world)
    def fresh_uid():
        """NCCL unique id of a new communicator: rank 0 creates it, torch.distributed carries the 128 bytes"""
        if world == 1:
            return None
        L0 = __import__("adflow_b200._lib", fromlist=["load"]).load()
        t = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            buf = (C.c_char * 128)()
            assert L0.adfb_get_unique_id(buf) == 0
            t = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).cuda()
        dist.broadcast(t, 0)
        return bytes(t.cpu().numpy().tobytes())

    uid = fresh_uid()
    blocks = make_grid_blocks(grid, rank, prm)
    s = ADFLOW_B200(prm, device=local, rank=rank, nranks=world, unique_id=uid)
    for hb in blocks:
        s.addBlock(hb)
    s.setCommPattern(build_cartesian_pattern(grid, rank))
    hb = blocks[0]
    cells = sum(b.d.ncells for b in blocks)
    stream = torch.cuda.ExternalStream(s.L.adfb_stream(), device=local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    flags_core = RES_FLOW | RES_TURB | RES_SKIP_PREAMBLE
    flags_full = RES_FLOW | RES_TURB

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(fn, n):
        """n steps, each bracketed by CUDA events on the library stream, L2 flushed before each."""
        tot = 0.0
        with torch.cuda.stream(stream):
            for _ in range(n):
                flush.zero_()
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                e1.synchronize()
                tot += e0.elapsed_time(e1)
        return tot

    # ---- device-resident value ------------------------------------------------
    step = lambda: s.residual(flags_full)  # noqa: E731
    timed_steps(step, args.warmup)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    n0 = s.launchCount()
    ms_total = timed_steps(step, args.steps)
    launches = s.launchCount() - n0
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, s, blocks, grid.local_blocks(rank), grid.nblocks, rank == 0, np)
        barrier()
    # ---- e2e through the vector API with pinned host buffers -------------------
    nvec = s.getStateSize()
    h_state = torch.empty(nvec, dtype=torch.float64).pin_memory()
    h_res = torch.empty(nvec, dtype=torch.float64).pin_memory()
    h_state.numpy()[:] = s.getStates()

    def e2e_three_calls():
        s.L.adfb_set_states(C.c_void_p(h_state.data_ptr()), nvec)
        s.L.adfb_residual(1, flags_full)
        s.L.adfb_get_res(C.c_void_p(h_res.data_ptr()), nvec)

    def e2e_step():
        # FormFunction_mf (NKSolvers.F90:437-461) = setW(wVec); blocketteRes; setRVec(rVec) with host vectors: ONE C-ABI call.  On one
        # GPU (no exchange partners) it runs as a slab pipeline: copy in, kernels and copy out of the call overlap.
        if s.L.adfb_form_function(C.c_void_p(h_state.data_ptr()), C.c_void_p(h_res.data_ptr()), nvec) != 0:
            raise RuntimeError("adfb_form_function failed")

    def wall_ms(fn):
        for _ in range(args.warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        barrier()
        return ms

    e2e_three_ms = wall_ms(e2e_three_calls)
    res_three = h_res.numpy().copy()
    e2e_ms = wall_ms(e2e_step)
    e2e_maxdiff = float(np.abs(h_res.numpy() - res_three).max() / max(np.abs(res_three).max(), 1e-300))
    # nvidia-smi answers every 100 ms and needs a few hundred ms for its first line; a short timed region (K steps of 0.3 ms) can end
    # before it.  The same step keeps running, untimed, for a fixed number of launches on every rank (the step holds a collective
    # at N > 1), so that the clocks and throttle reasons reported are those of this workload under load.
    for _ in range(60):
        for _ in range(25):
            step()
        torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-kernel timing pass (roofline) --------------------------------------
    s.L.adfb_set_timing(1)
    for _ in range(args.steps):
        with torch.cuda.stream(stream):
            flush.zero_()
        s.residual(flags_full)
    ms_k = (C.c_double * 16)(); cnt_k = (C.c_longlong * 16)()
    s.L.adfb_kernel_times.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    s.L.adfb_kernel_name.restype = C.c_char_p
    nk = s.L.adfb_kernel_times(ms_k, cnt_k, 16)
    s.L.adfb_set_timing(0)
    kernels = {s.L.adfb_kernel_name(i).decode(): {"ms_per_launch": ms_k[i] / cnt_k[i], "launches": int(cnt_k[i])}
               for i in range(nk) if cnt_k[i] > 0}
    res_ms = sum(ms_k[i] for i in range(nk)) / args.steps  # every kernel of the step (preamble, BCs, halo, core)
    dom = max(kernels.items(), key=lambda kv: kv[1]["ms_per_launch"] * kv[1]["launches"]) if kernels else None
    _ = flags_core

    # ---- the other operators of the metric (smoothers, SA solve, matrix-free matvec): N = 1 only --------
    others = None
    if world == 1:
        others = {}
        nrep = max(3, min(10, args.steps))

        def ev_time(fn):
            fn()  # warm-up (graph capture, lazy allocations)
            return timed_steps(fn, nrep) / nrep

        s.timeStep(False)
        s.smootherResidual(0)
        for name, fn, bpc in (
            ("rk_cycle_5stage", lambda: s.rkCycle(), 5 * 272.0),
            ("dadi_step", lambda: s.dadiStep(), 236.0 + 160.0),
            ("sa_ddadi_3subiter", lambda: s.turbSolveDDADI(3), 3 * 156.0),
        ):
            ms = ev_time(fn)
            others[name] = {"ms": ms, "Mcells/s": cells / (ms * 1e-3) / 1e6, "algorithmic_bytes_per_cell": bpc,
                            "GB/s": bpc * cells / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": bpc * cells / (ms * 1e-3) / 1e9 / peaks()[0]}
        # matrix-free matvec y = (F(U + h a) - F(U)) / h through the vector API (host vectors, so PCIe included)
        s.uploadState(0, hb)
        U = s.getStates()
        s.mffdSetBase(U)
        ha = torch.empty(U.size, dtype=torch.float64).pin_memory()
        hy = torch.empty(U.size, dtype=torch.float64).pin_memory()
        a, y = ha.numpy(), hy.numpy()
        a[:] = np.random.default_rng(7).standard_normal(U.size)
        s.mffdApply(a, 1e-7, out=y)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(nrep):
            s.mffdApply(a, 1e-7, out=y)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / nrep
        da = torch.from_numpy(a.copy()).cuda()
        dy = torch.empty_like(da)
        s.mffdApplyDevice(da.data_ptr(), dy.data_ptr(), da.numel(), 1e-7)
        torch.cuda.synchronize()
        same = bool(torch.equal(dy.cpu(), torch.from_numpy(y)))   # same product as through host vectors
        t0 = time.perf_counter()
        for _ in range(nrep):
            s.mffdApplyDevice(da.data_ptr(), dy.data_ptr(), da.numel(), 1e-7)
        torch.cuda.synchronize()
        msd = (time.perf_counter() - t0) * 1e3 / nrep
        others["mffd_matvec_device_vectors"] = {
            "ms": msd, "Mcells/s": cells / (msd * 1e-3) / 1e6, "algorithmic_bytes_per_cell": 464.0,
            "GB/s": 464.0 * cells / (msd * 1e-3) / 1e9, "frac_of_hbm_peak": 464.0 * cells / (msd * 1e-3) / 1e9 / peaks()[0],
            "bitwise_equal_to_host_vector_product": same,
            "note": "a and y resident on the GPU (adfb_mffd_apply_device, the PETSc VECCUDA path): perturb + full residual "
                    "(blocketteRes incl. BCs) + difference, no PCIe"}
        others["mffd_matvec_host_vectors"] = {
            "ms": ms, "Mcells/s": cells / (ms * 1e-3) / 1e6, "algorithmic_bytes_per_cell": 464.0,
            "GB/s": 464.0 * cells / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": 464.0 * cells / (ms * 1e-3) / 1e9 / peaks()[0],
            "note": "unfused form: perturb + residual + difference (464 B/cell); a and y are pinned host vectors, "
                    "so the time includes 2 x %d MB over PCIe" % (a.nbytes >> 20)}

        # the two extra operators must never cost the headline line: a failure is recorded, not raised
        try:
            # ANK matrix-free product (approximate fluxes + time-step term), vectors resident on the device
            from adflow_b200.params import make_ank_params
            s.uploadState(0, hb)
            s.ankSetParams(make_ank_params(cfl=5.0, coupled=False))
            s.referenceShockSensor()
            s.residual(flags_full | 4)
            s.ankTimeStepMat()
            Ua = np.ascontiguousarray(np.transpose(hb.w[hb.d.owned()][..., :5], (2, 1, 0, 3)).reshape(-1))
            s.ankMffdSetBase(Ua)
            dka = torch.from_numpy(np.random.default_rng(9).standard_normal(Ua.size)).cuda()
            dky = torch.empty_like(dka)
            s.ankMffdApplyDevice(dka.data_ptr(), dky.data_ptr(), dka.numel(), 1e-7)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(nrep):
                s.ankMffdApplyDevice(dka.data_ptr(), dky.data_ptr(), dka.numel(), 1e-7)
            torch.cuda.synchronize()
            msa = (time.perf_counter() - t0) * 1e3 / nrep
            others["ank_mffd_matvec_device_vectors"] = {
                "ms": msa, "Mcells/s": cells / (msa * 1e-3) / 1e6,
                "note": "ANKSolver FormFunction_mf product (decoupled, nState = 5): perturb + blocketteRes with the approximate "
                        "dissipation (flow rows only) + timeStepMat term + difference, vectors on the GPU"}
            # one multigrid cycle (the smoother of config C3: 4W, Runge-Kutta) on the same block: 4 grid levels
            from adflow_b200 import synthetic as syn
            lv = [hb]
            for _ in range(3):
                lv.append(syn.make_coarse_block(lv[-1], prm))
            for q in range(1, 4):
                s.addCoarseBlock(lv[q], q - 1)
            s.uploadState(0, hb)
            s.applyBCs(True, True)
            s.timeStep(False)
            s.smootherResidual(0)
            cyc = ADFLOW_B200.cycleStrategy("4w")
            msg = ev_time(lambda: s.mgCycle(cyc))
            others["mg_4w_rk_cycle"] = {
                "ms": msg, "Mcells/s": cells / (msg * 1e-3) / 1e6,
                "levels": ["%dx%dx%d" % (b_.d.nx, b_.d.ny, b_.d.nz) for b_ in lv], "steps_in_cycle": len(cyc),
                "note": "executeMGCycle: %d smoothing steps (5-stage RK each), %d restrictions, %d prolongations, then "
                        "turbSolveDDADI + timeStep + residual on the fine level" % (cyc.count(0), cyc.count(1), cyc.count(-1))}
        except Exception as ex:  # noqa: BLE001
            others["extra_operators_error"] = "%s: %s" % (type(ex).__name__, ex)

    # max over ranks
    ms_step = ms_total / args.steps
    if world > 1:
        t = torch.tensor([ms_step, e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, e2e_ms = float(t[0]), float(t[1])
    value = cells * world / (ms_step * 1e-3) / 1e6
    e2e_val = cells * world / (e2e_ms * 1e-3) / 1e6

    # ---- self-check of the multi-block data plane of THIS run (N > 1: NCCL) ---------------------------------------
    pat_main = build_cartesian_pattern(grid, rank)
    checked, bad = halo_data_check(s, blocks, pat_main, np, torch, dist if world > 1 else None)
    s.residual(flags_full)
    norms_main = [float(x) for x in s.getResNorms()]
    if world > 1:
        t = torch.tensor([checked, bad], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        checked, bad = int(t[0]), int(t[1])
    s.close()

    peak, peak_src = peaks()
    strong = matvec = None
    if not args.no_scaling_sections:
        try:
            strong = strong_scaling_c3(args, torch, dist if world > 1 else None, rank, world, local, fresh_uid, np)
        except Exception as ex:  # noqa: BLE001
            strong = {"error": "%s: %s" % (type(ex).__name__, ex)}
        try:
            matvec = nk_matvec_c5(args, torch, dist if world > 1 else None, rank, world, local, fresh_uid, np, peak)
        except Exception as ex:  # noqa: BLE001
            matvec = {"error": "%s: %s" % (type(ex).__name__, ex)}

    if rank == 0:
        achieved = BYTES_PER_CELL * cells / (res_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "Mcells/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(shape, world), "cells": cells * world,
                       "detail": "full residual = blocketteRes: p/rlv/rev + BCs + halo exchange + flow+SA rows with exact fluxes; "
                                 "1 block per GPU, %s block arrangement" % "x".join(map(str, nb)),
                       "cells_per_gpu": cells, "l2": "flushed before every timed step (256 MiB memset)",
                       "timing": "CUDA events on the library stream around each step"},
            "e2e": {"value": e2e_val, "unit": "Mcells/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(nvec * 8), "d2h_bytes_per_step": int(nvec * 8),
                    "path": "adfb_form_function(pinned host wVec, pinned host rVec) = FormFunction_mf: setW, blocketteRes (p/rlv/rev preamble, BCs, "
                            "core), setRVec in one C-ABI call; without exchange partners (N = 1) the call is a slab pipeline over k planes "
                            "(H2D, kernels and D2H overlap), with partners the one-shot sequence",
                    "three_call_ms_per_step": e2e_three_ms,
                    "three_call_path": "adfb_set_states -> adfb_residual -> adfb_get_res (round-1 e2e path, unpipelined)",
                    "max_rel_diff_vs_three_call_path": e2e_maxdiff},
            "gpu_launches": int(launches),
            "halo_check": {"status": "ok" if bad == 0 else "FAILED", "halo_cells_checked": checked, "halo_cells_wrong": bad,
                           "res_norms": norms_main,
                           "how": "listed halo cells poisoned on the device, exchanged (NCCL between ranks), compared bit for bit with the "
                                  "donor cells' values, which travel to the checking rank independently (torch point-to-point)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_from_step_time": BYTES_PER_CELL * cells / (ms_step * 1e-3) / 1e9 / peak,
                         "frac_note": "frac: 176 B/cell x cells / SUM of the per-kernel event times of one step (separate timing pass, "
                                      "side-stream overlap counted twice: conservative); frac_from_step_time: same bytes / ms_per_step",
                         "traffic": NCU_TRAFFIC_BYTES if tuple(shape) == tuple(C2) else None,
                         "traffic_note": NCU_TRAFFIC_NOTE,
                         "peak_source": peak_src,
                         "kernel": "whole residual step: all launches (state prep, BCs, halo pack/unpack, k_prep, k_flowres tile kernel, "
                                   "k_sa) charged against 176 B/cell",
                         "algorithmic_bytes_per_cell": BYTES_PER_CELL, "kernels": kernels,
                         "dominant_kernel": None if dom is None else {
                             "name": dom[0], "ms_per_launch": dom[1]["ms_per_launch"],
                             "share_of_summed_kernel_time": dom[1]["ms_per_launch"] * dom[1]["launches"] / (res_ms * args.steps),
                             "GB/s_if_charged_the_whole_176_B_per_cell": BYTES_PER_CELL * cells / (dom[1]["ms_per_launch"] * 1e-3) / 1e9,
                             "note": "the tile kernel k_flowres (flow rows of the residual); its own ncu numbers are in profiles/r02_ncu_summary.md"},
                         "second_roof": FP64_ROOF},
            "clocks": clocks,
        }
        if others:
            line["other_operators"] = others
        if strong is not None:
            line["strong_scaling_c3"] = strong
        if matvec is not None:
            line["nk_matvec_c5"] = matvec
        if not args.no_cpu_baseline:
            v, reps, kind = cpu_baseline_single(shape)
            line["cpu_baseline"] = {"value": v, "unit": "Mcells/s", "cores": 1, "kind": kind,
                                    "sample": "%d residual evaluations (blocketteResCore) of the same block, 1 core, %s"
                                              % (reps, KIND_NOTE[kind])}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
