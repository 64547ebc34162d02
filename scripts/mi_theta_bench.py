"""Throughput of the fixed-theta mixed-integer solves (MixedIntegerThetaSolver: K8 / K9 in pair mode, the winner, pass 2).

    python scripts/mi_theta_bench.py [--points 100000] [--out FILE]

For an mpMIQP and an mpMILP (tests/mi_programs.objective_program) at nb ~ 10 and nb ~ 40 binaries: the assignments (the
relaxation tree's leaves), the pairs per batch (points x assignments), and pairs/s and points/s of solve_batch over
--points points of Theta (CUDA events, after a warm-up batch, median of --reps).  For the mpMILPs also scipy.optimize.milp
(HiGHS MIP) one point per call on one core, over --milp-points points.  The card's name and power limit are read in the
same run (nvidia-smi) and written beside the numbers.  One JSON object per line; --out also writes them to a file."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]

CASES = [('mpMIQP', 'qp', 10, None), ('mpMILP', 'lp', 10, None), ('mpMIQP', 'qp', 40, 2), ('mpMILP', 'lp', 40, 2)]


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [v.strip() for v in q.split(',')]
        return dict(gpu=name, power_limit=power)
    except Exception as e:   # the numbers are still written, marked as such
        return dict(gpu='unknown', power_limit='unknown', card_query_error=str(e))


def milp_rate(prog, th):
    from scipy.optimize import Bounds, LinearConstraint, milp
    n = prog.A.shape[1]
    eq = numpy.zeros(prog.A.shape[0], bool)
    eq[list(prog.equality_indices)] = True
    integ = numpy.zeros(n)
    integ[prog.binary_indices] = 1
    lb, ub = numpy.full(n, -numpy.inf), numpy.full(n, numpy.inf)
    lb[prog.binary_indices], ub[prog.binary_indices] = 0.0, 1.0
    t0 = time.perf_counter()
    for p in th:
        h = prog.b.ravel() + prog.F @ p
        milp(prog.c.ravel() + prog.H @ p, constraints=LinearConstraint(prog.A, numpy.where(eq, h, -numpy.inf), h),
             integrality=integ, bounds=Bounds(lb, ub), options=dict(mip_rel_gap=0.0))
    return len(th) / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--points', type=int, default=100000)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--milp-points', type=int, default=300)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch
    from mi_programs import objective_program
    from ppopt_b200 import MixedIntegerThetaSolver
    if not torch.cuda.is_available():
        raise SystemExit('mi_theta_bench needs a CUDA device')
    info = card()
    lines = []
    for label, kind, nb, at_most in CASES:
        prog = objective_program(nb, 0, kind=kind, at_most=at_most)
        s = MixedIntegerThetaSolver(prog)
        th = torch.from_numpy(s.sample_thetas(int(a.points * 1.05) + 16, seed=1)[:a.points]).cuda()
        s.solve_batch(th[:1024])
        times = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = s.solve_batch(th)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
        sec = float(numpy.median(times))
        k = th.shape[0]
        st = out['status'].cpu().numpy()
        rec = dict(program=label, nb=nb, n_cont=len(prog.cont_indices), t=prog.F.shape[1], rows=prog.A.shape[0],
                   assignments=s.n_assign, points=k, pairs=k * s.n_assign, seconds=sec, pairs_per_s=k * s.n_assign / sec,
                   points_per_s=k / sec, optimal=int((st == 0).sum()), infeasible=int((st == 1).sum()),
                   failed=int((st == 2).sum()), unbounded=int((st == 4).sum()), **info)
        if kind == 'lp':
            rec['highs_milp_points_per_s_one_core'] = milp_rate(prog, th[:a.milp_points].cpu().numpy())
        s.close()
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
