"""Relaxation tree of a mixed-integer program (K11) on one GPU: nodes per second, pivots per node per depth and the
inherited share, against HiGHS on one host core (one node LP per call) and, at nb = 16, the 2^nb screen
(``screen='enumerate'``: one engine per assignment).

    python scripts/mitree_bench.py [--out profiles/r07_mitree_bench.txt] [--enum-subset 256]

Programs: tests/mitree_programs.py's ``random_program(16, 5)`` and the nb = 40 program of tests/test_gpu_mitree.py
(sum(y) <= 2, couplings x <= 10 y).  The tree is timed with a host clock around the whole call (it synchronises once per
depth), after a warm-up run; HiGHS on every node of the same tree; the 2^nb screen on the first ``--enum-subset``
assignments, extrapolated to all 2^16 and labelled so."""
import argparse
import itertools
import os
import subprocess
import sys
import time

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from mitree_programs import random_program, relaxation_margin  # noqa: E402
from test_gpu_mitree import _sum_program  # noqa: E402
from ppopt_b200.mp_solvers import mitree  # noqa: E402
from ppopt_b200.mp_solvers import mpmiqp_enumeration as enum  # noqa: E402


def tree_run(prog, inherit, reps=5):
    mitree.feasible_combinations(prog, inherit=inherit)   # warm-up
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        res = mitree.feasible_combinations(prog, inherit=inherit)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None or dt < best else best
    return res, best


def highs_nodes(prog, res, limit):
    """HiGHS on the nodes of the tree, one LP per call (the first `limit` nodes in tree order)"""
    nb = len(prog.binary_indices)
    level, done, t0 = [()], 0, time.perf_counter()
    for d in range(nb + 1):
        nxt = []
        for y in level:
            if done >= limit:
                return done, time.perf_counter() - t0
            ok = relaxation_margin(prog, y) <= 0.0
            done += 1
            if ok and d < nb:
                nxt += [y + (0,), y + (1,)]
        level = nxt
    return done, time.perf_counter() - t0


def enumerate_subset(prog, k):
    t0 = time.perf_counter()
    for y in itertools.islice(itertools.product((0, 1), repeat=len(prog.binary_indices)), k):
        if not enum.binary_rows_hold(prog, y):
            continue
        try:
            sub = prog.generate_substituted_problem(list(y))
        except Exception:
            continue
        enum.leaf_is_feasible(sub)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='also write the report to this file')
    ap.add_argument('--enum-subset', type=int, default=256)
    ap.add_argument('--highs-nodes', type=int, default=4000)
    a = ap.parse_args()
    lines = []

    def out(s=''):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    out(f'# K11 relaxation tree bench  ({smi}; torch {torch.__version__})')
    progs = {'nb16 random_program(16, 5)': random_program(16, 5), 'nb40 sum(y) <= 2': _sum_program(40, 2, 1, 2, False)}
    for name, prog in progs.items():
        out(f'\n## {name}: {prog.A.shape[0]} rows, {prog.A.shape[1]} variables, {prog.F.shape[1]} parameters')
        for inherit in (True, False):
            res, dt = tree_run(prog, inherit)
            st = res.stats
            nodes = sum(st['nodes'])
            out(f'tree inherit={int(inherit)}: {len(res.leaves)} leaves, {nodes} nodes, {sum(st["lps"])} LPs, '
                f'{sum(st["inherited"])} inherited ({100.0 * sum(st["inherited"]) / max(1, nodes):.1f} %), '
                f'{dt * 1e3:.2f} ms (best of 5), {nodes / dt:.0f} nodes/s')
            if inherit:
                out('depth  nodes  feasible  LPs  inherited  pivots/LP')
                for d in range(len(st['nodes'])):
                    out(f'{d:5d} {st["nodes"][d]:6d} {st["feasible"][d]:9d} {st["lps"][d]:4d} {st["inherited"][d]:10d} '
                        f'{st["pivots"][d] / max(1, st["lps"][d]):10.2f}')
        done, ht = highs_nodes(prog, res, a.highs_nodes)
        out(f'HiGHS (scipy linprog, one host core, one node per call): {done} nodes in {ht:.2f} s = {done / ht:.0f} nodes/s'
            + ('' if done >= nodes else f' (first {done} of {nodes} nodes)'))
        if len(prog.binary_indices) <= 20:
            k = min(a.enum_subset, 2 ** len(prog.binary_indices))
            et = enumerate_subset(prog, k)
            out(f"screen='enumerate' (one engine per assignment): first {k} assignments in {et:.2f} s; EXTRAPOLATED to all "
                f"{2 ** len(prog.binary_indices)}: {et * 2 ** len(prog.binary_indices) / k:.1f} s")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
