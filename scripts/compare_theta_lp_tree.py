"""Bit identity of two builds of libppgpu.so on the fixed-theta LP (K9), the relaxation tree's node LPs (K11) and the
fixed-theta QP (K8).

    python scripts/compare_theta_lp_tree.py LIB_A LIB_B [--out report.txt]

Each library runs in a subprocess of its own (``ppopt_b200._lib.LIB_PATH`` is set before ``load()``) that dumps every output
array of every case into an .npz; the report says, case by case, whether the arrays of the two libraries are equal
(``numpy.array_equal(..., equal_nan=True)``).  The exit status is 1 when any array differs.

Cases, all seeded:
  K9  ThetaLPSolver.solve_batch (status, x, dual, active mask, iters = pivots and Phase 1 pivots) on the mpLPs of
      tests/test_gpu_solve_theta_lp.py: the LP goldens, seeded_eq, bench_mplp and the two envelope shapes, at points of
      Theta and at points of a box twice the width of Theta's sampling box (mostly outside Theta); and the hand-made
      infeasible and unbounded LPs over a sweep of theta.
  K11 RelaxationTree.eval at every depth (nodes, status, point, iters) on random_program(nb, seed) and the nb = 40 program
      of tests/test_gpu_mitree.py, with point inheritance off and on.
  K8  ThetaSolver.solve_batch (the outputs of K9, iters = steps) on every QP golden whose reduced Hessian is positive
      definite, at the same kinds of points.
"""
import argparse
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
SEP = '|'


def thetas(solver, k, seed):
    """up to k points of Theta (rejection in its sampling box), then k // 4 points of a box twice as wide"""
    from ppopt_b200.solve_theta import theta_box
    inside = solver.sample_thetas(8 * k, seed)[:k]
    lo, hi = theta_box(solver.A_t, solver.b_t)
    w = hi - lo
    outside = numpy.random.default_rng(seed + 1).uniform(lo - w / 2, hi + w / 2, size=(k // 4, len(lo)))
    return numpy.vstack([inside, outside])


def batch(solver, th):
    out = solver.solve_batch(th)
    return {'theta': th} | {f: out[f].cpu().numpy() for f in ('status', 'x', 'dual', 'active', 'iters')}


def k9_cases():
    from test_gpu_solve_theta_lp import ENVELOPE, _tiny, envelope_mplp, lp_solver
    from test_theta_lp_dict import LP_GOLDEN, program
    progs = [(name, program(name), 20000) for name in LP_GOLDEN + ['seeded_eq', 'bench_mplp']]
    progs += [(f'envelope_{mi}_{n}_{t}', envelope_mplp(mi, n, t), 4000) for mi, n, t in ENVELOPE]
    for name, g, k in progs:
        solver = lp_solver(g)
        yield name, batch(solver, thetas(solver, k, seed=11))
        solver.close()
    sweep = numpy.linspace(-12.0, 12.0, 241).reshape(-1, 1)
    tiny = {'tiny_infeasible': _tiny([[1, 0], [-1, 0], [0, 1], [0, -1]], [0, -1, 1, 1], [1, 0, 0, 0], [1, 1]),
            'tiny_unbounded': _tiny([[1, 0], [0, 1]], [1, 1], [0, 0], [-1, -1], H=[[1.0], [0.0]])}
    for name, g in tiny.items():
        solver = lp_solver(g)
        yield name, batch(solver, sweep)
        solver.close()


def k11_cases():
    import torch
    from mitree_programs import random_program
    from ppopt_b200.mp_solvers.mitree import RelaxationTree
    from test_gpu_mitree import _sum_program
    progs = [(f'random_program({nb}, {s})', lambda nb=nb, s=s: random_program(nb, s)) for nb, s in ((6, 0), (8, 3), (12, 4), (16, 5))]
    progs.append(('sum_program(40, 2, 1, 2)', lambda: _sum_program(40, 2, 1, 2, False)))
    for name, make in progs:
        for inherit in (False, True):
            tree = RelaxationTree(make(), inherit=inherit)
            out = {}
            nodes = torch.zeros(1, dtype=torch.int64, device=tree.tdev)
            pp = po = None
            for d in range(tree.nb + 1):
                st, pt, it = tree.eval(nodes, d, points=True, parent_point=pp, parent_of=po)
                out |= {f'd{d}_nodes': nodes.cpu().numpy(), f'd{d}_status': st.cpu().numpy(), f'd{d}_point': pt.cpu().numpy(),
                        f'd{d}_iters': it.cpu().numpy()}
                if d < tree.nb:
                    nodes, po = tree.children(nodes, st, d)
                    pp = pt
            tree.close()
            yield f'{name} inherit={int(inherit)}', out


def k8_cases():
    from ppopt_b200.mplp_program import load_presolved
    from ppopt_b200.solve_theta import ThetaSolver
    for f in sorted(os.listdir(GOLDEN)):
        if not f.endswith('.npz') or str(numpy.load(os.path.join(GOLDEN, f))['kind']) != 'qp':
            continue
        try:
            solver = ThetaSolver(load_presolved(os.path.join(GOLDEN, f)))
        except NotImplementedError:
            continue
        yield f[:-4], batch(solver, thetas(solver, 20000, seed=21))
        solver.close()


def dump(lib_path, out_path):
    from ppopt_b200 import _lib
    _lib.LIB_PATH = os.path.abspath(lib_path)
    _lib.load()
    arrays = {}
    for kernel, cases in (('K9', k9_cases), ('K11', k11_cases), ('K8', k8_cases)):
        for name, res in cases():
            arrays |= {SEP.join((kernel, name, k)): v for k, v in res.items()}
    with open('/proc/self/maps') as f:
        loaded = sorted({ln.split()[-1] for ln in f if 'libppgpu' in ln})
    assert loaded == [_lib.LIB_PATH], (loaded, _lib.LIB_PATH)
    numpy.savez(out_path, **arrays)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('libs', nargs='*', help='the two libppgpu.so to compare')
    ap.add_argument('--out', default=None, help='also write the report to this file')
    ap.add_argument('--dump', nargs=2, metavar=('LIB', 'NPZ'), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.dump:
        dump(*a.dump)
        return 0
    assert len(a.libs) == 2, 'give two libraries'
    lines = []

    def out(s=''):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip()
    out(f'# K9 / K11 / K8 outputs of two libppgpu.so builds ({smi})')
    res = []
    with tempfile.TemporaryDirectory() as tmp:
        for i, lib in enumerate(a.libs):
            with open(lib, 'rb') as f:
                out(f'library {"AB"[i]}: {os.path.relpath(os.path.abspath(lib), ROOT)} (md5 {hashlib.md5(f.read()).hexdigest()})')
            path = os.path.join(tmp, f'{i}.npz')
            subprocess.run([sys.executable, os.path.abspath(__file__), '--dump', lib, path], check=True)
            res.append(numpy.load(path))
        assert sorted(res[0].files) == sorted(res[1].files), 'the two dumps hold different cases'
        cases = {}
        for key in res[0].files:
            kernel, name, field = key.split(SEP)
            cases.setdefault((kernel, name), []).append(field)
        n_bad = 0
        out('\ncase: arrays, elements, statuses (A) -> verdict')
        for (kernel, name), fields in cases.items():
            got = [{f: r[SEP.join((kernel, name, f))] for f in fields} for r in res]
            bad = [f for f in fields if not numpy.array_equal(got[0][f], got[1][f], equal_nan=got[0][f].dtype.kind == 'f')]
            n_bad += len(bad)
            size = sum(v.size for v in got[0].values())
            st = numpy.concatenate([v.ravel() for f, v in got[0].items() if f.endswith('status')])
            counts = dict(zip(*[v.tolist() for v in numpy.unique(st, return_counts=True)]))
            out(f'{kernel} {name}: {len(fields)} arrays, {size} elements, status {counts} -> '
                + ('equal' if not bad else 'DIFFER: ' + ', '.join(bad)))
    out(f'\n{sum(len(f) for f in cases.values())} arrays in {len(cases)} cases; '
        + ('all equal' if n_bad == 0 else f'{n_bad} differ'))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')
    return 1 if n_bad else 0


if __name__ == '__main__':
    sys.exit(main())
