"""Throughput of the batched fixed-theta QP (K8, ppopt_b200.ThetaSolver) on the bench program, mpc_n10 and ctrl_alloc_n5,
with K7 explicit evaluation of the same points for two full solutions and the CPU twin's rate on one core beside it.

    python scripts/solve_theta_bench.py [--points 4000000] [--out results.json]

Device rate: CUDA events around one ppgpu_solve_theta_batch launch over preallocated buffers, after a warm-up launch of
the same size (the 4 M theta points are 4e6 x t x 8 B and outputs larger than L2, so the timed pass does not run from
a warm cache).  End-to-end rate: host numpy thetas in, host status / x out, through ThetaSolver.solve_batch.
Models (counted from each point's step count and final working set, an upper bound on what the iteration did):
    FLOP   = sum over points of iters x (2 mi (|W| + 1) + 2 |W|^2)      (slack update + the two triangular solves)
    smem B = sum over points of iters x 8 mi (|W| + 1)                   (G columns read by the slack update)
over kernel time, against the measured FP64 DFMA rate and a shared-memory bandwidth of 128 B per clock per SM at the
card's maximum SM clock.  The reference's QP backends (daqp, gurobi) are not dependencies of this project: no reference rate is reported.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from ppopt_b200 import _lib, engine, mpqp_algorithm, solve_mpqp  # noqa: E402
from ppopt_b200.mplp_program import load_presolved  # noqa: E402
from ppopt_b200.point_location import PointLocation  # noqa: E402
from ppopt_b200.solve_theta import ThetaSolver  # noqa: E402
from twin_theta_qp import ThetaQpTwin  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clk = [s.strip() for s in q.split(',')]
    return dict(name=name, power_limit=power, max_sm_clock=clk, sm_count=torch.cuda.get_device_properties(0).multi_processor_count)


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
    act, it = e.empty((k, solver.W), torch.int64), e.empty((k,), torch.int32)
    args = lambda: (e.h, d_th.data_ptr(), k, st.data_ptr(), x.data_ptr(), dual.data_ptr(), act.data_ptr(), it.data_ptr(), e._stream())  # noqa: E731
    _lib.check(e.lib.ppgpu_solve_theta_batch(*args()), 'warm-up')
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    _lib.check(e.lib.ppgpu_solve_theta_batch(*args()), 'timed')
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), st, act, it


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--points', type=int, default=4_000_000)
    ap.add_argument('--out', default=None, help='also write the results as JSON to this file')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    torch.cuda.set_device(0)
    info = card()
    fp64 = engine.measure_fp64_peak()
    smem_bw = info['sm_count'] * 128 * float(info['max_sm_clock'].split()[0]) * 1e6
    res = dict(card=info, fp64_dfma_tflops_measured=fp64, smem_bytes_per_s_model=smem_bw, points=args.points, programs={})
    print(f"{info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}; measured FP64 {fp64:.1f} TFLOP/s")
    for name in ('synthetic_30_6_40_s0', 'mpc_n10', 'ctrl_alloc_n5'):
        solver = ThetaSolver(load_presolved(os.path.join(GOLDEN, name + '.npz')))
        th = thetas_in_theta(solver, args.points)
        d_th = torch.from_numpy(th).cuda()
        ms, st, act, it = time_kernel(solver, d_th)
        st, it = st.cpu().numpy(), it.cpu().numpy()
        wsz = numpy.unpackbits(act.cpu().numpy().view(numpy.uint8), axis=1).sum(1).astype(numpy.float64)
        mi = solver.eng.mi
        flop = float((it * (2.0 * mi * (wsz + 1) + 2.0 * wsz ** 2)).sum())
        smem = float((it * 8.0 * mi * (wsz + 1)).sum())
        t_flop, t_smem = flop / (fp64 * 1e12), smem / smem_bw
        solver.solve_batch(th[:100000])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = solver.solve_batch(th)
        host_st, host_x = out['status'].cpu().numpy(), out['x'].cpu().numpy()
        t1 = time.perf_counter()
        assert numpy.array_equal(host_st, st)
        hist = numpy.bincount(it)
        r = dict(n=solver.n, t=solver.t, m=solver.m, mi=mi, kernel_ms=ms, device_points_per_s=args.points / ms * 1e3,
                 host_e2e_ms=1e3 * (t1 - t0), host_e2e_points_per_s=args.points / (t1 - t0),
                 status_counts={int(k): int(v) for k, v in zip(*numpy.unique(st, return_counts=True))},
                 iters_mean=float(it.mean()), iters_p95=float(numpy.percentile(it, 95)), iters_max=int(it.max()),
                 iters_hist={i: int(c) for i, c in enumerate(hist) if c},
                 working_set_mean=float(wsz.mean()), working_set_max=int(wsz.max()),
                 flop_model=flop, smem_bytes_model=smem, achieved_tflops=flop / ms * 1e-9, achieved_smem_tb_per_s=smem / ms * 1e-9,
                 fp64_bound_ms=1e3 * t_flop, smem_bound_ms=1e3 * t_smem, bound='shared memory' if t_smem > t_flop else 'fp64',
                 share_of_bound=1e3 * max(t_flop, t_smem) / ms)
        tw = ThetaQpTwin.from_npz(os.path.join(GOLDEN, name + '.npz'))
        k_cpu = 20000 if mi < 64 else 5000
        t2 = time.perf_counter()
        tw.theta_qp(th[:k_cpu])
        r['twin_points_per_s_one_core'] = k_cpu / (time.perf_counter() - t2)
        res['programs'][name] = r
        print(f"{name}: n {r['n']} t {r['t']} m {r['m']}; {args.points} points: kernel {ms:.1f} ms = {r['device_points_per_s']:.3e} points/s, "
              f"host arrays {r['host_e2e_ms']:.0f} ms = {r['host_e2e_points_per_s']:.3e} points/s; status {r['status_counts']}; "
              f"iters mean {r['iters_mean']:.1f} p95 {r['iters_p95']:.0f} max {r['iters_max']}; |W| mean {r['working_set_mean']:.1f}; "
              f"model {r['achieved_tflops']:.2f} TFLOP/s, {r['achieved_smem_tb_per_s']:.2f} TB/s smem, bound {r['bound']} "
              f"({100 * r['share_of_bound']:.1f} % of it); CPU twin {r['twin_points_per_s_one_core']:.3e} points/s (1 core)")
        solver.close()
    for name in ('mpc_n7', 'rand_6_3_12_s1'):
        prog = load_presolved(os.path.join(GOLDEN, name + '.npz'))
        sol = solve_mpqp(prog, mpqp_algorithm.combinatorial)
        solver = ThetaSolver(prog)
        th = thetas_in_theta(solver, args.points)
        d_th = torch.from_numpy(th).cuda()
        ms_qp = time_kernel(solver, d_th)[0]
        pl = PointLocation(sol)
        pl._run(d_th, sol.point_location_tolerance, True)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pl._run(d_th, sol.point_location_tolerance, True)
        b.record()
        torch.cuda.synchronize()
        ms_pl = a.elapsed_time(b)
        res['programs'][name] = dict(regions=len(sol.critical_regions), k8_kernel_ms=ms_qp, k8_points_per_s=args.points / ms_qp * 1e3,
                                     k7_explicit_ms=ms_pl, k7_points_per_s=args.points / ms_pl * 1e3)
        print(f"{name}: {len(sol.critical_regions)} regions; {args.points} points: implicit (K8) {ms_qp:.1f} ms = "
              f"{args.points / ms_qp * 1e3:.3e} points/s, explicit (K7 locate + evaluate) {ms_pl:.1f} ms = {args.points / ms_pl * 1e3:.3e} points/s")
        solver.close()
    res['reference_backends'] = 'daqp / gurobi are not dependencies of this project: no reference rate'
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
