"""Whole solve_mpqp calls with the geometric, combinatorial and combinatorial_graph algorithms on five programs.

Timing starts from the program object and ends after a device synchronise; every (program, algorithm) pair is run once as
warm-up first.  Also reported: regions, waves and QP solves, and the GPU time of K10 (facet_cheb_kernel) and K8
(k8_theta_qp_kernel) as a share of the geometric call, from torch.profiler in a separate run (K10 is stateless and K8 is not
one of the handle's profile_read families).  Writes profiles/r11_geometric_bench.jsonl with the GPU name and power limit read
in the same call; a line is written as soon as its (program, algorithm) pair is measured.

    python scripts/geometric_bench.py [--reps 3] [--out profiles/r11_geometric_bench.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PROGRAMS = ['ctrl_alloc_n2', 'rand_6_3_12_s1', 'mpc_n7', 'mpc_n10', 'ctrl_alloc_n5']


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else 'unknown'
    except Exception as e:   # the measurement itself still needs the GPU; only the label is missing
        return f'unknown ({e})'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r11_geometric_bench.jsonl'))
    args = ap.parse_args()
    import torch
    from ppopt_b200 import mpqp_algorithm, solve_mpqp
    from ppopt_b200.mplp_program import load_presolved
    if not torch.cuda.is_available():
        raise SystemExit('geometric_bench needs a GPU')
    gpu = gpu_info()
    algos = [mpqp_algorithm.geometric, mpqp_algorithm.combinatorial, mpqp_algorithm.combinatorial_graph]
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    fh = open(args.out, 'w')
    for name in PROGRAMS:
        prog = load_presolved(os.path.join(ROOT, 'tests', 'golden', name + '.npz'))
        for algo in algos:
            solve_mpqp(prog, algo)
            torch.cuda.synchronize()
            times = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                sol = solve_mpqp(prog, algo)
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t0)
            rec = dict(gpu=gpu, program=name, algorithm=algo.name, seconds=sorted(times), regions=len(sol.critical_regions))
            if algo is mpqp_algorithm.geometric:
                rec.update(waves=sol.waves, qp_solves=sol.qp_solves, facets=sol.facets, facets_thin=sol.facets_thin,
                           retries=sol.retries, unresolved=len(sol.unresolved))
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    solve_mpqp(prog, algo)
                    torch.cuda.synchronize()
                tot, k10, k8 = 0.0, 0.0, 0.0
                for ev in prof.key_averages():
                    us = getattr(ev, 'device_time_total', None)
                    us = ev.cuda_time_total if us is None else us
                    tot += us
                    if 'facet_cheb_kernel' in ev.key:
                        k10 += us
                    if 'k8_theta_qp_kernel' in ev.key:
                        k8 += us
                rec.update(gpu_kernel_ms=tot / 1e3, k10_ms=k10 / 1e3, k8_ms=k8 / 1e3)
            print(json.dumps(rec), flush=True)
            fh.write(json.dumps(rec) + '\n')
            fh.flush()
    fh.close()


if __name__ == '__main__':
    main()
