#!/usr/bin/env python
"""bench.py - candidate active sets / second of the combinatorial mpQP enumeration (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            this repo's CUDA engine (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  the UNMODIFIED reference on the host cores
    python bench.py ... --dump-outputs DIR                   also writes the outputs of the last timed step (dump_outputs)

Workload (config.workload): BASELINE.json configs[4], the synthetic dense mpQP with 100 constraints / 30 variables /
6 parameters = generate_mpqp(30, 6, 40, seed=0) after the reference's presolve (tests/golden/synthetic_30_6_40_s0.npz),
combinatorial levels 1..L (default L = 5: 74,536,536 candidate active sets; L = 4: 3,940,375; L = 3: 163,810).
A "step" is one full pass of the level loop over that program.

  value   device-resident throughput: program constants already in HBM, every kernel of the path runs (K1 rank, K2w / K2a /
          K2 feasibility, K3/K4 optimality screen, K5 region emission, K6 next-level generation), region buffers stay
          in HBM.  CUDA events on the launch stream, max over ranks, L2 flushed between steps.
  e2e     the same pass through the public call solve_mpqp(program, mpqp_algorithm.combinatorial) with HOST numpy
          program data: upload, all kernels, download of the region matrices, CriticalRegion objects built.
  roofline  the kernel family with the largest share of the step (round 2: the vertex walk K2w): useful fp64 flops counted
          in-kernel / its summed launch durations (CUDA events recorded around each launch inside libppgpu), against the
          fp64 FMA peak measured on this device by a register-resident DFMA loop (MEASURED_PEAKS.json has no fp64 entry).
          The path is fp64 / shared-memory-latency bound, not HBM bound: 8W+2 algorithmic bytes per candidate per pass.
  parity  N > 1: the sharded run's digest (decision bits of every candidate of every level + the region list) must
          equal the digest of a single-GPU run of the same program made by rank 0 in the same process; the bench FAILS
          otherwise.
  reference arm / cpu_baseline  the UNMODIFIED reference (baseline/_ref, imported under the LP shim of oracle/ref_shim:
          cvxopt/GLPK are not in this image, HiGHS answers solve_lp) doing the stock per-candidate work of its parallel
          combinatorial solver - mpqp_parrallel_combinatorial.full_process (feasibility LP, optimality LP, region
          build, child generation against the pruning list) mapped over a pathos-style pool of ALL host cores, and the
          same on one core (serial solver's loop body) - on a bounded random sample of the SAME workload: candidates
          drawn from levels 1..L in proportion to the true level sizes (levels 1-3: the golden level lists; levels 4-5:
          the 40,000 candidates sampled from the engine's own level arrays, tests/golden/sampled/).  kind = "reference";
          falls back to the numpy/HiGHS port (kind = "port") only if the reference cannot be imported.
  full_solves  (metric ii) complete solves, wall-clock through solve_mpqp, of programs both sides can finish.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    'synthetic_30_6_40_s0': 'synthetic dense mpQP 100 constraints / 30 vars / 6 params (generate_mpqp(30,6,40,seed=0))',
    'mpc_n10': 'explicit MPC double integrator, horizon N=10',
    'ctrl_alloc_n5': 'control allocation, 4 rotors, 5 stacked steps',
}
METRIC = 'candidate active sets/sec'


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# --------------------------------------------------------------------------------------------- CPU arm
FULL_SOLVES = ['factory_mpqp', 'rand_6_3_12_s1', 'ctrl_alloc_n2']   # small enough for the reference inside a bench run


def _lists(masks, n_eq):
    m = numpy.ascontiguousarray(masks).view(numpy.uint64)
    m = m.reshape(m.shape[0], -1)
    bits = numpy.unpackbits(m.view(numpy.uint8).reshape(m.shape[0], -1), axis=1, bitorder='little')
    eq = list(range(n_eq))
    return [eq + (numpy.nonzero(r)[0] + n_eq).tolist() for r in bits]


class Workload:
    """candidate pools of levels 1..L of a golden program, with the true level sizes"""

    def __init__(self, name, L):
        g = numpy.load(os.path.join(ROOT, 'tests', 'golden', name + '.npz'))
        sp = os.path.join(ROOT, 'tests', 'golden', 'sampled', name + '.npz')
        s = numpy.load(sp) if os.path.exists(sp) else None
        self.name, self.L = name, L
        self.pools, self.sizes, self.murder = [], [], []
        for lv in range(L):
            if lv < int(g['n_levels']):
                c, st = g[f'level{lv}_candidates'], g[f'level{lv}_status']
                self.pools.append(c)
                self.sizes.append(len(c))
                self.murder.extend(tuple(x) for x in c[(st & 2) == 0].tolist())
            elif s is not None and lv in s['levels'].tolist():
                c, st = s[f'level{lv}_candidates'], s[f'level{lv}_status']
                # every region the engine found was added to the sample on purpose: leave them out of the timing pool
                # (true frequency 6e-5; the reference spends ~100 LPs on each)
                self.pools.append(c[(st & 8) == 0])
                self.sizes.append(int(s[f'level{lv}_size']))
            else:
                raise SystemExit(f'no candidate pool for level {lv + 1} of {name}')
        self.total = sum(self.sizes)

    def draw(self, n, rng):
        """n (candidate, level) pairs: level ~ true level sizes, candidate uniform in the level's pool"""
        lv = rng.choice(len(self.sizes), size=n, p=numpy.array(self.sizes, dtype=float) / self.total)
        return [(self.pools[l][rng.integers(len(self.pools[l]))].tolist(), int(l)) for l in lv]


def _load_reference():
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    try:
        import ref_harness
        if not ref_harness.available():
            return None
        return ref_harness.load()
    except Exception as e:   # noqa: BLE001
        print(f'[bench] reference not importable ({e}); falling back to the port', file=sys.stderr)
        return None


def _reference_program(name):
    import problems
    from ppopt.mplp_program import MPLP_Program
    from ppopt.mpqp_program import MPQP_Program
    d = problems.CONFIGS[name]()
    kw = {'post_process': d['post_process']} if 'post_process' in d else {}
    if d['kind'] == 'qp':
        return MPQP_Program(d['A'], d['b'], d['c'], d['H'], d['Q'], d['A_t'], d['b_t'], d['F'],
                            equality_indices=list(d['equality_indices']), **kw)
    return MPLP_Program(d['A'], d['b'], d['c'], d['H'], d['A_t'], d['b_t'], d['F'],
                        equality_indices=list(d['equality_indices']), **kw)


class ReferenceRunner:
    """the stock per-candidate work of the reference's combinatorial solvers on a sample of the workload"""

    def __init__(self, wl, cores):
        from pathos.multiprocessing import ProcessingPool as Pool   # the shim over multiprocess.Pool (oracle/ref_shim)
        from ppopt.mp_solvers.mpqp_parrallel_combinatorial import full_process
        from ppopt.mp_solvers.solver_utils import CombinationTester
        self.wl, self.cores = wl, cores
        self.program = _reference_program(wl.name)
        self.murder = CombinationTester()
        self.murder.add_combos(set(wl.murder))
        self.full_process = full_process
        self.pool = Pool(cores) if cores > 1 else None
        program, murder, L = self.program, self.murder, wl.L
        # exactly the closure of mpqp_parrallel_combinatorial.solve (:110): the pool pickles program + pruning list
        self.f = lambda x: full_process(program, x[0], murder, x[1] + 1 < L)

    def run(self, sample):
        t0 = time.perf_counter()
        outs = self.pool.map(self.f, sample) if self.pool is not None else [self.f(x) for x in sample]
        dt = time.perf_counter() - t0
        return dt, sum(1 for o in outs if not o[1]), sum(1 for o in outs if o[0] is not None)

    def rate(self, seconds, rng):
        probe = self.wl.draw(max(8, 4 * self.cores), rng)
        dt, _, _ = self.run(probe)
        n = int(max(2 * len(probe), len(probe) / max(dt, 1e-6) * seconds))
        dt, feas, regs = self.run(self.wl.draw(n, rng))
        return n / dt, n, dt, feas, regs

    def close(self):
        if self.pool is not None:
            self.pool.clear()


def reference_full_solves(names):
    """(metric ii) the reference's own solve_mpqp, serial and all-core parallel, on programs it can finish"""
    from ppopt.mp_solvers.solve_mpqp import mpqp_algorithm, solve_mpqp
    out = []
    for name in names:
        prog = _reference_program(name)
        row = {'program': name}
        for key, algo in (('serial_s', mpqp_algorithm.combinatorial), ('parallel_s', mpqp_algorithm.combinatorial_parallel)):
            t0 = time.perf_counter()
            sol = solve_mpqp(prog, algo)
            row[key] = time.perf_counter() - t0
            row['regions_' + key[:-2]] = len(sol.critical_regions)
        out.append(row)
    return out


def cpu_baseline(args, seconds, serial_seconds):
    """dict for the cpu_baseline key (and the reference arm): the unmodified reference when it is importable, else the port"""
    cores = host_cores()
    wl = Workload(args.workload, args.levels)
    rng = numpy.random.default_rng(0)
    if _load_reference() is not None:
        par = ReferenceRunner(wl, cores)
        rate, n, dt, feas, regs = par.rate(seconds, rng)
        ser = ReferenceRunner(wl, 1)
        srate, sn, sdt, _, _ = ser.rate(serial_seconds, rng)
        mix = ', '.join(f'L{i + 1} {100.0 * s / wl.total:.3g}%' for i, s in enumerate(wl.sizes))
        return par, wl, {
            'value': rate, 'unit': 'candidates/s', 'cores': cores, 'kind': 'reference',
            'sample': f'{n} candidates in {dt:.1f}s on {cores} processes: mpqp_parrallel_combinatorial.full_process of the '
                      f'unmodified reference (HiGHS behind the cvxopt shim) over a pathos-style pool, candidates drawn from '
                      f'levels 1..{wl.L} of the same program in proportion to the true level sizes ({mix}); '
                      f'{feas} feasible, {regs} regions in the sample',
            'serial': {'value': srate, 'unit': 'candidates/s', 'cores': 1,
                       'sample': f'{sn} candidates in {sdt:.1f}s, same draw, one process (the serial solver\'s loop body)'}}
    # fallback: the numpy/HiGHS port
    import ppopt_oracle as oracle
    P = oracle.Program.from_npz(os.path.join(ROOT, 'tests', 'golden', args.workload + '.npz'))
    sample = [c for c, _ in wl.draw(max(64, int(200 * cores * seconds / 15)), rng)]
    t0 = time.perf_counter()
    oracle.evaluate_many(P, sample, cores)
    dt = time.perf_counter() - t0
    return None, wl, {'value': len(sample) / dt, 'unit': 'candidates/s', 'cores': cores, 'kind': 'port',
                      'sample': f'{len(sample)} candidates of levels 1..{wl.L} (true level mix) in {dt:.1f}s on {cores} '
                                f'processes, oracle/ppopt_oracle.py (reference not importable)'}


def run_reference(args, rank):
    if rank != 0:
        return
    n_steps = args.steps + args.warmup
    per_step = max(2.0, min(15.0, 150.0 / max(1, n_steps)))
    runner, wl, base = cpu_baseline(args, per_step, min(10.0, per_step))
    rng = numpy.random.default_rng(1)
    tot_n, tot_t = 0, 0.0
    if runner is not None:
        n_per = max(8, int(base['value'] * per_step))
        for i in range(n_steps):
            dt, _, _ = runner.run(wl.draw(n_per, rng))
            if i >= args.warmup:
                tot_n += n_per
                tot_t += dt
        runner.close()
    value = tot_n / tot_t if tot_t > 0 else base['value']
    full = []
    if runner is not None and not args.no_full_solves:
        try:
            full = reference_full_solves(FULL_SOLVES)
        except Exception as e:   # noqa: BLE001
            full = [{'error': str(e)}]
    base = dict(base, value=value)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'candidates/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot_t / max(1, args.steps),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': WORKLOADS[args.workload] + f', combinatorial levels 1..{args.levels}', 'levels': args.levels,
                   'candidates_per_step': wl.total,
                   'sampled': f'each step = {tot_n // max(1, args.steps)} candidates drawn from levels 1..{args.levels} in '
                              f'proportion to the true level sizes (a bounded sample: the full pass is {wl.total} candidates)',
                   'l2': 'n/a (CPU arm)'},
        'cpu_baseline': base,
        'e2e': {'value': value, 'unit': 'candidates/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'full_solves': full,
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- GPU arm
class ClockSampler(threading.Thread):
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                                      '-i', str(self.gpu)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(s[1]) for s in self.samples if len(s) > 2 and s[1].replace('.', '', 1).isdigit()]
        mx = [float(s[2]) for s in self.samples if len(s) > 2 and s[2].replace('.', '', 1).isdigit()]
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for s in self.samples:
            for nm, v in zip(names, s[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(numpy.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(self.samples)}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, dev_sol, e2e_sol):
    """Writes what the last timed step of each GPU path returned, as float64 .npy files, so that two builds can be compared
    output for output: level_stats (level, candidates, feasible, optimal, regions) of the device-resident pass, and the
    critical regions of the end-to-end solve.  A and b are stacked per region; the rows of C, d, E, f and the active sets
    are concatenated over the regions, region_rows gives each region's (active set length, rows of E).  Above DUMP_BYTES
    a fixed seeded sample of the regions is written; region_index lists which ones."""
    os.makedirs(out_dir, exist_ok=True)
    f64 = lambda x: numpy.asarray(x, dtype=numpy.float64)
    stats = f64([[s['level'], s['candidates'], s['feasible'], s['optimal'], s['regions']] for s in dev_sol.level_stats])
    regions = e2e_sol.critical_regions
    size = [8 * (numpy.size(r.A) + numpy.size(r.b) + numpy.size(r.C) + numpy.size(r.d) + numpy.size(r.E) + numpy.size(r.f)
                 + len(r.active_set) + 3) for r in regions]
    keep = list(range(len(regions)))
    room = DUMP_BYTES - stats.nbytes - (16 << 10)   # the .npy headers
    if sum(size) > room:
        keep = []
        for i in numpy.random.default_rng(0).permutation(len(regions)).tolist():
            if size[i] <= room:
                keep.append(i)
                room -= size[i]
        keep.sort()
    sel = [regions[i] for i in keep]
    t = e2e_sol.program.num_t()
    n = e2e_sol.program.num_x()
    out = {
        'level_stats': stats.reshape(-1, 5),
        'region_index': f64(keep),
        'region_rows': f64([[len(r.active_set), numpy.shape(r.E)[0]] for r in sel]).reshape(-1, 2),
        'region_active_set': f64([i for r in sel for i in r.active_set]),
        'region_A': f64([r.A for r in sel]).reshape(-1, n, t),
        'region_b': f64([r.b for r in sel]).reshape(-1, n),
    }
    for fld, shape in (('C', (-1, t)), ('d', (-1,)), ('E', (-1, t)), ('f', (-1,))):
        rows = [f64(getattr(r, fld)).reshape(shape) for r in sel]
        out['region_' + fld] = numpy.concatenate(rows) if rows else numpy.zeros((0,) + shape[1:])
    for name, a in out.items():
        numpy.save(os.path.join(out_dir, name + '.npy'), a)


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from ppopt_b200 import engine, mpqp_algorithm, solve_mpqp
    from ppopt_b200.mplp_program import load_presolved
    path = os.path.join(ROOT, 'tests', 'golden', args.workload + '.npz')
    prog = load_presolved(path)
    L = args.levels
    dev = torch.device('cuda', local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn):
        """one step: L2 flush, barrier, CUDA events around fn on the current stream, max over ranks"""
        flush.zero_()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    eng = engine.Engine(engine.program_arrays(prog), device=local_rank)
    dev_step = lambda: engine.solve(prog, max_levels=L, engine=eng, materialize=False)
    e2e_step = lambda: solve_mpqp_capped(prog, L)

    def solve_mpqp_capped(p, levels):
        # the public entry point is solve_mpqp(program, mpqp_algorithm.combinatorial); the depth cap (the reference has
        # none, bench.py applies the same cap to both arms) is passed through the engine behind it
        if levels >= eng.max_depth:
            return solve_mpqp(p, mpqp_algorithm.combinatorial)
        return engine.solve(p, max_levels=levels)

    for _ in range(args.warmup):
        timed(dev_step)
    # Python runtime hygiene for the timed loops: everything alive after the warm-up (torch's and numpy's module objects: a
    # couple of million containers) goes to the collector's permanent generation, so that a generation-2 collection inside
    # a timed step traverses that step's own objects only (measured on the B200 box: such a collection costs ~0.5 s in this
    # process and hit one end-to-end step in three).  All work of a step stays inside the timed region.
    import gc
    gc.collect()
    gc.freeze()
    eng.counters(reset=True)
    eng.profile(True)
    eng.profile_read(reset=True)
    launches0 = eng.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, units = [], 0
    for _ in range(args.steps):
        ms, sol = timed(dev_step)
        ms_dev.append(ms)
        units = sol.total_candidates
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join(timeout=2)
    prof = eng.profile_read(reset=True)
    eng.profile(False)
    if os.environ.get('PPGPU_BENCH_VERBOSE'):
        print(f'[rank {rank}] ms/step dev {sum(ms_dev) / len(ms_dev):.1f} kernels ' + str({k: round(v['ms'] / len(ms_dev), 1) for k, v in prof.items() if v['launches']}), file=sys.stderr, flush=True)
    counters = eng.counters()
    launches = eng.launch_count() - launches0
    levels_stats = sol.level_stats
    # ---- end to end through the public API with host buffers
    ms_e2e, h2d, d2h, n_regions = [], 0, 0, 0
    for i in range(max(1, min(args.warmup, 2)) + args.steps):
        ms, s2 = timed(e2e_step)
        if i >= max(1, min(args.warmup, 2)):
            ms_e2e.append(ms)
            h2d, d2h, n_regions = s2.h2d_bytes, s2.d2h_bytes, len(s2.critical_regions)
    if os.environ.get('PPGPU_BENCH_VERBOSE'):
        print(f'[rank {rank}] e2e ms per step ' + str([round(x, 1) for x in ms_e2e]), file=sys.stderr, flush=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sol, s2)
    # ---- parity of the sharded run: same digest as a single-GPU run of the same program (rank 0, same process)
    parity = None
    d_all = engine.solve(prog, max_levels=L, engine=eng, digest=True).digest
    if world > 1:
        d_one = engine.solve(prog, max_levels=L, engine=eng, digest=True, distributed=False).digest if rank == 0 else None
        agree = torch.tensor([1 if (rank != 0 or d_one == d_all) else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        parity = {'digest': d_all, 'single_gpu_digest': d_one, 'equal': bool(agree.item())}
        if not parity['equal']:
            raise SystemExit(f'[bench] PARITY FAILURE: the {world}-GPU run decides differently from the 1-GPU run '
                             f'({d_all} vs {d_one})')
    else:
        parity = {'digest': d_all}
    # ---- (metric ii) complete solves through the public call, programs the reference can finish too
    full = []
    if rank == 0 and not args.no_full_solves:
        from ppopt_b200.mplp_program import load_presolved as _lp
        for name in FULL_SOLVES + ['mpc_n7']:
            p2 = _lp(os.path.join(ROOT, 'tests', 'golden', name + '.npz'))
            g2 = numpy.load(os.path.join(ROOT, 'tests', 'golden', name + '.npz'))
            best = None
            for _ in range(3):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                s3 = engine.solve(p2, distributed=False)
                torch.cuda.synchronize(dev)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            full.append({'program': name, 'seconds': best, 'regions': len(s3.critical_regions),
                         'candidates': s3.total_candidates,
                         'regions_equal_reference': [list(r.active_set) for r in s3.critical_regions] ==
                         [g2[f'r{i}_active_set'].tolist() for i in range(int(g2['n_regions']))],
                         'reference_serial_s_build_container': float(g2['reference_solve_seconds']) if 'reference_solve_seconds' in g2 else float(numpy.sum(g2['replay_seconds']))})
    fp64_peak = engine.measure_fp64_peak()
    total_launches = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(total_launches)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    value = units * len(ms_dev) / (sum(ms_dev) * 1e-3)
    e2e_value = units * len(ms_e2e) / (sum(ms_e2e) * 1e-3)
    # dominant kernel family of the timed steps and its in-kernel count of useful fp64 FMAs
    fams = {'k2w_walk': ('k2w_walk_kernel (feasibility certificates shared between the candidates of a prefix by a primal-simplex '
                         'walk over vertices, slack dictionary in shared memory)', counters['k2w_work'], counters['k2w_certified']),
            'k2a_relax': ('k2p_relax_kernel (feasibility certificates, prefix-projected Gram in shared memory)', counters['k2a_work'], counters['k2a_tried']),
            'k2_feas_lp': ('k2_feas_kernel (feasibility simplex)', counters['k2_work'], counters['k2_lps']),
            'k34_kkt_cheb': ('k34_kernel (KKT + Chebyshev screen)', counters['k4_work'], counters['k4_lps'])}
    dom = max(fams, key=lambda f: prof[f]['ms'])
    k2 = prof[dom]
    dom_name, dom_work, dom_units = fams[dom]
    k2_flops = 2.0 * dom_work
    k2_tflops = k2_flops / max(k2['ms'] * 1e-3, 1e-12) / 1e12
    hbm_bytes = (8.0 * eng.W + 2.0) * dom_units  # mask in, status byte in + out
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    traffic, smem = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', f'r02_{dom}_traffic.json')))
        traffic = tj.get('dram_bytes_per_launch')
        if dom == 'k2w_walk':
            # what actually bounds the walk: every entry of the slack dictionary is read and written once per pivot in SHARED
            # memory (16 B per counted FMA); peak = 128 B / clock / SM at the SM clock sampled during the timed region
            clk = (sampler.summary().get('sm_mhz') or 1965.0) * 1e6
            sm_peak = eng.sm_count * 128.0 * clk / 1e12
            sm_ach = 16.0 * dom_work / max(k2['ms'] * 1e-3, 1e-12) / 1e12
            smem = {'bound': 'shared memory', 'achieved': sm_ach, 'peak': sm_peak, 'unit': 'TB/s', 'frac': sm_ach / sm_peak,
                    'ncu_wavefronts_pct_of_peak': tj.get('smem_wavefronts_pct_of_peak'),
                    'note': 'algorithmic shared-memory bytes (dictionary read + write per pivot) over the kernel time; the ncu figure '
                            'counts every shared-memory wavefront of the level-5 launch (profiles/r02_k2w_ncu.txt)'}
    except Exception:
        pass
    line = {
        'metric': METRIC, 'value': value, 'unit': 'candidates/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': sum(ms_dev) / len(ms_dev), 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': WORKLOADS[args.workload] + f', combinatorial levels 1..{L}', 'levels': L,
                   'candidates_per_step': units, 'regions_per_step': n_regions, 'parallelism': f'level-sharded x{world}',
                   'l2': 'flushed between steps (256 MiB write)',
                   'python_gc': 'gc.freeze() after the warm-up (the interpreter baseline heap is not re-traversed inside timed steps)',
                   'per_level': [[s['candidates'], s['feasible'], s['optimal']] for s in levels_stats]},
        'e2e': {'value': e2e_value, 'unit': 'candidates/s', 'ms_per_step': sum(ms_e2e) / len(ms_e2e),
                'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h), 'call': 'solve_mpqp(program, combinatorial)'},
        'gpu_launches': int(total_launches.item()),
        'roofline': {'kernel': dom_name, 'bound': 'fp64', 'achieved': k2_tflops, 'peak': fp64_peak, 'unit': 'TFLOP/s',
                     'frac': k2_tflops / fp64_peak if fp64_peak else None, 'traffic': traffic,
                     'traffic_source': 'dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this '
                                       f'kernel (profiles/r02_{dom}_traffic.json, which names the launch); ncu cannot run inside '
                                       'the timed run',
                     'peak_source': 'measured on this device: register-resident DFMA loop (ppgpu_measure_fp64_peak); '
                                    'MEASURED_PEAKS.json carries no fp64 figure',
                     'launches': k2['launches'], 'avg_launch_ms': k2['ms'] / max(1, k2['launches']),
                     'flops_per_launch': k2_flops / max(1, k2['launches']), 'units': dom_units,
                     'share_of_step': k2['ms'] / max(1e-9, sum(v['ms'] for v in prof.values())),
                     'flop_model': 'useful fp64 FMAs counted in-kernel: K2w pivots x basic rows x columns of the slack dictionary '
                                   '(rank-1 update); K2a relaxation steps x R0 x 3; K2/K4 pivots x live rows x columns',
                     'k2w': {'certified': counters['k2w_certified'], 'pivots': counters['k2w_pivots'], 'gave_up': counters['k2w_giveup']},
                     'inherited': {'certified': counters['inherited'], 'lookups': counters['inherit_lookups'],
                                   'note': 'candidates certified by the witness vertex of one of their parents (no LP work)'},
                     'shared_memory': smem,
                     'k2a': {'tried': counters['k2a_tried'], 'certified': counters['k2a_certified'], 'steps': counters['k2a_steps']},
                     'k2': {'lps': counters['k2_lps'], 'pivots': counters['k2_pivots']},
                     'hbm': {'achieved': hbm_bytes / max(k2['ms'] * 1e-3, 1e-12) / 1e9, 'peak': peaks.get('hbm_gbs'),
                             'unit': 'GB/s', 'note': 'algorithmic bytes are 8W+2 B per candidate: not HBM bound'}},
        'kernels_ms_per_step': {k: v['ms'] / len(ms_dev) for k, v in prof.items() if v['launches']},
        'clocks': sampler.summary(),
        'fp64_peak_tflops': fp64_peak,
        'parity': parity,
        'full_solves': full,
        'flagged': {k: (v if isinstance(v, int) else len(v)) for k, v in sol.flagged.items()},
    }
    if world == 1 and not args.no_cpu_baseline:
        runner, _wl, base = cpu_baseline(args, args.cpu_seconds, min(8.0, args.cpu_seconds))
        if runner is not None:
            runner.close()
        line['cpu_baseline'] = base
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--levels', type=int, default=5)
    ap.add_argument('--workload', default='synthetic_30_6_40_s0', choices=list(WORKLOADS))
    ap.add_argument('--cpu-seconds', type=float, default=15.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-full-solves', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='GPU arm: write what the last timed step returned as DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
