"""Throughput of the batched fixed-theta LP (K9, ppopt_b200.ThetaLPSolver) on env_lp_w3, the bench-shaped synthetic mpLP
(oracle/problems.random_mpqp(30, 6, 100, 0, kind='lp')) and transport_mplp, with HiGHS on one core beside it.

    python scripts/solve_theta_lp_bench.py [--points 4000000] [--out results.json]

Device rate: CUDA events around one ppgpu_solve_theta_lp_batch launch over preallocated buffers, after a warm-up launch of
the same size (4 M theta points and their outputs are larger than L2, so the timed pass does not run from a warm cache).
Pivots per point (mean, p95, max) and the Phase 1 share come from the kernel's own counts.  Models, over kernel time:
    FLOP   = sum over points of pivots x 2 (mi + 1) (np + 2)        (one FMA per dictionary entry and pivot)
    smem B = sum over points of (pivots x 16 + 8) (mi + 1) (np + 2)  (each entry read and written per pivot, written once
                                                                      when the start dictionary is copied in)
against the measured FP64 DFMA rate and a shared-memory bandwidth of 128 B per clock per SM at the card's maximum SM clock.
CPU comparison: scipy.optimize.linprog(method='highs') point by point in this process (HiGHS, not the reference: the
reference's LP backends are not dependencies of this project).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy
import torch
from scipy.optimize import linprog

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))

import problems  # noqa: E402
from ppopt_b200 import _lib, engine  # noqa: E402
from ppopt_b200.mplp_program import MPLP_Program, load_presolved  # noqa: E402
from ppopt_b200.solve_theta import ThetaLPSolver  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clk = [s.strip() for s in q.split(',')]
    return dict(name=name, power_limit=power, max_sm_clock=clk, sm_count=torch.cuda.get_device_properties(0).multi_processor_count)


def programs():
    g = problems.random_mpqp(30, 6, 100, 0, kind='lp')
    synth = MPLP_Program(g['A'], g['b'], g['c'], g['H'], g['A_t'], g['b_t'], g['F'], presolved=True)
    return [('env_lp_w3', load_presolved(os.path.join(GOLDEN, 'envelope', 'env_lp_w3.npz'))),
            ('random_mplp_30_6_100_s0', synth),
            ('transport_mplp', load_presolved(os.path.join(GOLDEN, 'transport_mplp.npz')))]


def thetas_in_theta(solver, k, seed=0):
    out = numpy.zeros((0, solver.t))
    s = seed
    while out.shape[0] < k:
        out = numpy.vstack([out, solver.sample_thetas(max(k, 1000) * 2, s)])
        s += 1
    return numpy.ascontiguousarray(out[:k])


def time_kernel(solver, d_th):
    e = solver.eng
    k = d_th.shape[0]
    st = e.empty((k,), torch.uint8)
    x, dual = e.empty((k, solver.n), torch.float64), e.empty((k, solver.m), torch.float64)
    act, it = e.empty((k, solver.W), torch.int64), e.empty((k, 2), torch.int32)
    args = lambda: (e.h, d_th.data_ptr(), k, st.data_ptr(), x.data_ptr(), dual.data_ptr(), act.data_ptr(), it.data_ptr(), e._stream())  # noqa: E731
    _lib.check(e.lib.ppgpu_solve_theta_lp_batch(*args()), 'warm-up')
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    _lib.check(e.lib.ppgpu_solve_theta_lp_batch(*args()), 'timed')
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), st, it


def highs_rate(prog, th):
    A, b, F = numpy.asarray(prog.A), numpy.asarray(prog.b).ravel(), numpy.asarray(prog.F)
    c, H, ne = numpy.asarray(prog.c).ravel(), numpy.asarray(prog.H), len(prog.equality_indices)
    t0 = time.perf_counter()
    for p in th:
        rhs = b + F @ p
        linprog(c + H @ p, A_ub=A[ne:], b_ub=rhs[ne:], A_eq=A[:ne] if ne else None, b_eq=rhs[:ne] if ne else None,
                bounds=[(None, None)] * A.shape[1], method='highs')
    return len(th) / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--points', type=int, default=4_000_000)
    ap.add_argument('--highs-points', type=int, default=1000)
    ap.add_argument('--out', default=None, help='also write the results as JSON to this file')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    torch.cuda.set_device(0)
    info = card()
    fp64 = engine.measure_fp64_peak()
    smem_bw = info['sm_count'] * 128 * float(info['max_sm_clock'].split()[0]) * 1e6
    res = dict(card=info, fp64_dfma_tflops_measured=fp64, smem_bytes_per_s_model=smem_bw, points=args.points, programs={})
    print(f"{info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}; measured FP64 {fp64:.1f} TFLOP/s")
    for name, prog in programs():
        solver = ThetaLPSolver(prog)
        th = thetas_in_theta(solver, args.points)
        d_th = torch.from_numpy(th).cuda()
        ms, st, it = time_kernel(solver, d_th)
        st, it = st.cpu().numpy(), it.cpu().numpy().astype(numpy.float64)
        mi, npr = solver.eng.mi, solver.n - solver.n_eq
        cells = (mi + 1) * (npr + 2)
        piv = it[:, 0]
        flop = float(piv.sum() * 2.0 * cells)
        smem = float((piv * 16.0 + 8.0).sum() * cells)
        t_flop, t_smem = flop / (fp64 * 1e12), smem / smem_bw
        r = dict(n=solver.n, t=solver.t, m=solver.m, mi=mi, n_eq=solver.n_eq, kernel_ms=ms,
                 device_points_per_s=args.points / ms * 1e3,
                 status_counts={int(k): int(v) for k, v in zip(*numpy.unique(st, return_counts=True))},
                 pivots_mean=float(piv.mean()), pivots_p95=float(numpy.percentile(piv, 95)), pivots_max=int(piv.max()),
                 phase1_share=float(it[:, 1].sum() / max(1.0, piv.sum())),
                 points_with_phase1=float((it[:, 1] > 0).mean()),
                 flop_model=flop, smem_bytes_model=smem, achieved_tflops=flop / ms * 1e-9,
                 achieved_smem_tb_per_s=smem / ms * 1e-9, fp64_bound_ms=1e3 * t_flop, smem_bound_ms=1e3 * t_smem,
                 bound='shared memory' if t_smem > t_flop else 'fp64', share_of_bound=1e3 * max(t_flop, t_smem) / ms)
        r['highs_points_per_s_one_core'] = highs_rate(prog, th[:args.highs_points])
        res['programs'][name] = r
        print(f"{name}: n {r['n']} t {r['t']} m {r['m']}; {args.points} points: kernel {ms:.1f} ms = "
              f"{r['device_points_per_s']:.3e} points/s; status {r['status_counts']}; pivots mean {r['pivots_mean']:.1f} "
              f"p95 {r['pivots_p95']:.0f} max {r['pivots_max']}, Phase 1 {100 * r['phase1_share']:.1f} % of them "
              f"({100 * r['points_with_phase1']:.1f} % of points need it); model {r['achieved_tflops']:.3f} TFLOP/s, "
              f"{r['achieved_smem_tb_per_s']:.3f} TB/s smem, bound {r['bound']} ({100 * r['share_of_bound']:.1f} % of it); "
              f"HiGHS {r['highs_points_per_s_one_core']:.3e} points/s (one core)")
        solver.close()
    res['cpu_comparison'] = "HiGHS through scipy.optimize.linprog(method='highs'), one point per call, one process"
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
