#!/usr/bin/env python
"""Benchmark of the GLAMR global-optimisation hot path (BASELINE.json metric: global-opt iterations/sec over
frames x persons), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--extras all|none|a,b,..] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one optimiser iteration of GlobalReconOptimizer.optimize_main (trajectory codec + camera + full SMPL
LBS for every frame-person + projection + residuals + analytic backward [+ one all-reduce of the packed gradient when
N > 1] + Adam).  Headline workload (config.workload): the glamr_dynamic stage on N persons x 300 frames, one person
per GPU (weak scaling; N = 1 is BASELINE.json configs[1]).  Rank 0 prints ONE JSON line.  Keyed extra results on the
same line (`extras`): the north-star video (glamr_static_multi, 4 persons x 300 frames, frame-persons sharded over the
N GPUs = strong scaling), configs[3] (8 x 500 glamr_static_multi), configs[2] (prior networks, 64 x 120) and configs[4]
(32 independent 300-frame sequences through run_dataset, replicas over the N GPUs).

--impl reference times the reference algorithm's CPU path on this box's host cores: the oracle port under oracle/
(torch-CPU restatement pinned to the executed reference by tests/golden), because /root/reference is not on the
GPU box.  It is the only place besides tests/ and smoke() that executes oracle/ code.
"""
import argparse
import copy
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

FRAMES = 300
CFG_ID = 'glamr_dynamic'
BYTES_CONST = 19_595_160          # SURVEY.md §8(d): SMPL constants, fp32 dense
BYTES_PER_FP = 1_460              # SURVEY.md §8(d): per frame-person reads + gradient writes + Adam traffic
FLOPS_PER_FP = 15.85e6            # SURVEY.md §8(d): dense full-LBS forward (algorithmic)
FLOPS_PER_FP_EXECUTED = 9.8e6     # K-sparse skinning (4 weights per vertex): what the kernel really issues
T_START = time.perf_counter()
# soft wall-clock budget of one `python bench.py` (our arm): the keyed extras (north star, C4, C3, C5) are skipped, with a note, once 60 % of it
# is spent, so that the headline line is always printed within minutes even on a host that is busy with other jobs
BENCH_BUDGET_S = float(os.environ.get('GLAMR_BENCH_BUDGET_S', 480.0))
REF_BUDGET_S = float(os.environ.get('GLAMR_REF_BUDGET_S', 150.0))   # wall-clock bound (s) of the CPU reference arm (--impl reference)
# dram__bytes_read.sum + dram__bytes_write.sum of one LBS launch, keyed by frame-persons per launch (ncu capture, profiles/)
NCU_BLEND_DRAM_BYTES = {300: 37911808 + 2394624}               # lbs_blend_tc_kernel alone
NCU_LBS_DRAM_BYTES = {300: 37911808 + 2394624 + 26944768}     # blend (read + write) + tensor-core skinning (read), profiles/lbs_tc_kernels_r02_final.md
# switches that change what the library executes: the bench refuses to run with any of them set
FORBIDDEN_ENV = ['GLAMR_B200_SO', 'GLAMR_LBS_DEBUG', 'GLAMR_TC_DEBUG', 'GLAMR_PDL', 'GLAMR_LBS_STAGES', 'GLAMR_TC_NTILE']
ECHO_ENV = FORBIDDEN_ENV + ['GLAMR_ITER_PATH', 'GLAMR_LBS_PATH', 'GLAMR_PRIOR_GRAPH', 'GLAMR_NET_WIMG', 'GLAMR_NET_SKINNY', 'GLAMR_ALLREDUCE', 'OMP_NUM_THREADS', 'NCCL_ALGO', 'NCCL_PROTO']
ALL_EXTRAS = ['north_star', 'c4', 'c3', 'c5']


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--frames', type=int, default=FRAMES)
    ap.add_argument('--persons', type=int, default=0, help='default: one per GPU')
    ap.add_argument('--extras', default='all', help="'all', 'none' or a comma list of " + ','.join(ALL_EXTRAS))
    ap.add_argument('--cpu-sample-iters', type=int, default=20)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed (optimisation variables and per-frame outputs) as DIR/<name>.npy')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    return a


def refuse_experiment_switches():
    bad = {k: os.environ[k] for k in FORBIDDEN_ENV if os.environ.get(k)}
    if bad:
        print(json.dumps({'error': 'refusing to benchmark with experiment switches set', 'env': bad}))
        sys.exit(2)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100', '-i', str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], f[4:8]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def make_problem(cfg_id, persons, frames, seed=0, gaps=False):
    from glamr_b200.config import Config
    from glamr_b200.synthetic import make_in_dict, make_smpl_assets
    assets = make_smpl_assets(0)
    in_dict = make_in_dict(assets, persons, frames, seed=seed, gaps=gaps, seq_name='bench')
    cfg = Config(cfg_id, out_dir='/tmp/glamr_b200_bench')
    return assets, in_dict, cfg


# ---------------------------------------------------------------------------------------------------- CPU arm (oracle port)
def host_threads():
    return max(1, len(os.sched_getaffinity(0)))


class CpuLegTimeout(Exception):
    pass


class wall_clock_limit:
    """Hard wall-clock bound for a CPU leg of the bench (the oracle port is thousands of small torch CPU ops per iteration, so a
    SIGALRM handler gets to run between two of them).  On hosts that are shared with other jobs a many-thread torch CPU
    iteration has been seen to take from 4 s to minutes; without a bound one such iteration decides how long bench.py runs."""

    pool = None          # seconds all CPU legs of this process may still spend together (None: no shared budget)

    def __init__(self, seconds):
        self.seconds = max(1, int(seconds))

    def _fire(self, signum, frame):
        raise CpuLegTimeout(f'CPU leg exceeded {self.seconds} s')

    def __enter__(self):
        import signal
        import threading
        cls = wall_clock_limit
        if cls.pool is not None:
            if cls.pool < 2.0:
                raise CpuLegTimeout('the CPU-time budget of this bench run is spent')
            self.seconds = max(1, min(self.seconds, int(cls.pool)))
        self.t0 = time.perf_counter()
        self.active = threading.current_thread() is threading.main_thread()
        if self.active:
            self.old = signal.signal(signal.SIGALRM, self._fire)
            signal.alarm(self.seconds)
        return self

    def __exit__(self, *exc):
        if self.active:
            import signal
            signal.alarm(0)
            signal.signal(signal.SIGALRM, self.old)
        if wall_clock_limit.pool is not None:
            wall_clock_limit.pool -= time.perf_counter() - self.t0
        return False


class CpuPort:
    """the oracle port (torch CPU) set up on one workload; `time_iterations` runs optimize_main of one stage and returns the
    per-iteration seconds.  Timing protocol (SURVEY.md §8d): thread-count sweep, warm-up discarded, >= 20 timed iterations,
    median AND best reported with the full per-iteration list."""

    def __init__(self, assets, in_dict, cfg, stage=None):
        import torch
        from glamr_b200.synthetic import LatentInjector
        from glamr_b200.synthetic_nets import make_prior_states
        from oracle.global_opt import OracleGlobalRecon
        from oracle.nets import MotionTrajJoint
        from oracle.smpl import OracleSMPL
        self.torch = torch
        cfg = copy.deepcopy(cfg)
        torch.set_num_threads(host_threads())      # torchrun exports OMP_NUM_THREADS=1, which would time a single-threaded reference
        st_m, st_t = make_prior_states(1234)
        self.model = OracleGlobalRecon(cfg, assets, mt_model=LatentInjector(MotionTrajJoint(st_m, st_t, OracleSMPL(assets)), 0))
        self.data = self.model.init_data(copy.deepcopy(in_dict))
        stages = list(cfg.opt_stage_specs.items())
        self.stage, self.specs = stages[0] if stage is None else [s for s in stages if s[0] == stage][0]

    def time_iterations(self, n, threads=None):
        if threads is not None:
            self.torch.set_num_threads(threads)
        times = []
        self._times = times                      # readable by a caller whose wall-clock limit interrupts the loop
        sp = self.specs
        self.model.optimize_main(self.data, sp['opt_variables'], sp['opt_lr'], n, sp['loss_cfg'], {'stage': self.stage},
                                 on_iter=lambda it, last, dt: times.append(dt))
        return times

    def sweep_threads(self, warm=1, probe=3, budget_s=40.0):
        """median seconds per iteration for each candidate thread count, smallest count first.  Bounded three ways (boxes exist
        where many-thread torch CPU runs are 25-250x slower than 8 threads, and hosts shared with other jobs where they take
        minutes): the all-threads candidate only runs on hosts with <= 64 threads (128 threads measured 4.5 - 12 s per iteration
        against 45 - 100 ms at 16 - 32, profiles/README_r02.md); a candidate is abandoned as soon as one of its iterations takes
        > 3x the best median so far; the sweep stops when a candidate is slower than the one before it (the scaling has turned
        over), when `budget_s` is spent, or when a candidate hits its own wall-clock limit.  -> (best_threads, {threads: median})"""
        cands = sorted({t for t in (8, 16, 32) if t <= host_threads()} | ({host_threads()} if host_threads() <= 64 else set()))
        res, t_start, prev = {}, time.perf_counter(), None
        for t in cands:
            left = budget_s - (time.perf_counter() - t_start)
            if res and left <= 0:
                break
            ts = []
            try:
                with wall_clock_limit(max(10.0, left) if res else 120.0):
                    for i in range(warm + probe):
                        (dt,) = self.time_iterations(1, threads=t)
                        ts.append(dt)
                        if res and dt > 3.0 * min(res.values()):
                            break
            except CpuLegTimeout:
                if not ts and not res:
                    raise
                if not ts:
                    break
            res[t] = float(np.median(ts[warm:] or ts))
            if prev is not None and res[t] > 1.25 * prev:
                break
            prev = res[t]
        best = min(res, key=res.get)
        return best, res


def cpu_baseline_block(assets, in_dict, cfg, units, iters, stage=None, sweep=True, threads=None, budget_s=60.0):
    """the CPU port on one workload, bounded by wall-clock: thread sweep (<= 40 s), then min(iters, what fits `budget_s`) timed
    iterations but never fewer than 5; every part runs under a hard wall-clock limit and the block degrades to what it has
    measured (or to a 'skipped' note) instead of stalling the bench on a host that is busy with other jobs"""
    t_block = time.perf_counter()
    try:
        with wall_clock_limit(120):
            port = CpuPort(assets, in_dict, cfg, stage)
            port.time_iterations(1, threads=threads or min(8, host_threads()))       # first-call warm-up (allocator, thread pool)
        if sweep:
            threads, sweep_res = port.sweep_threads()
            per = sweep_res[threads]
        else:
            threads, sweep_res = threads or min(8, host_threads()), {}
            with wall_clock_limit(90):
                (per,) = port.time_iterations(1, threads=threads)
    except CpuLegTimeout as e:
        return {'skipped': f'{e} during set-up / thread sweep (host busy); see --impl reference', 'kind': 'port', 'seconds_spent': time.perf_counter() - t_block}
    n = int(max(5, min(iters, budget_s / max(per, 1e-6))))
    ts, cut = [], False
    try:
        with wall_clock_limit(max(3.0 * budget_s, 8.0 * per * 5)):
            port.torch.set_num_threads(threads)
            sp = port.specs
            port.model.optimize_main(port.data, sp['opt_variables'], sp['opt_lr'], n, sp['loss_cfg'], {'stage': port.stage},
                                     on_iter=lambda it, last, dt: ts.append(dt))
    except CpuLegTimeout:
        cut = True
    if not ts:
        ts = [per]
    med, best = float(np.median(ts)), float(np.min(ts))
    return {'value': units / med, 'value_best': units / best, 'unit': 'frame*person*iter/s', 'cores': threads, 'host_threads_available': host_threads(),
            'kind': 'port', 'ms_per_iter_median': med * 1e3, 'ms_per_iter_best': best * 1e3,
            'thread_sweep_ms_per_iter': {str(k): round(v * 1e3, 2) for k, v in sweep_res.items()},
            'ms_per_iter_list': [round(t * 1e3, 1) for t in ts],
            'sample': f'{len(ts)} timed iterations (median; best in value_best) of the oracle port (torch CPU, {threads} threads' +
                      (' = fastest of the sweep' if sweep else '') + f') on the same workload ({port.stage}), after warm-up; bounded to ~{budget_s:.0f} s' +
                      (' (cut by the wall-clock limit)' if cut else '')}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    persons = args.persons or args.gpus
    assets, in_dict, cfg = make_problem(CFG_ID, persons, args.frames)
    K, W = max(args.steps, 1), max(args.warmup, 1)
    # Each step is a bounded sample of the workload so that K + W steps end within REF_BUDGET_S: a probe on the full workload
    # gives the per-iteration time; if K of them do not fit, a step processes the first `sample` persons only (the reference
    # loops over persons, its cost per frame-person is the same) and the metric counts those units; if one person is still
    # too slow, fewer timed steps run (stated in `sample`).
    sample = persons
    with wall_clock_limit(180):
        port = CpuPort(assets, in_dict, cfg)
        port.time_iterations(1, threads=min(8, host_threads()))
    threads, sweep_res = port.sweep_threads(warm=1, probe=3)
    probe = sweep_res[threads]
    if probe * (K + W) > REF_BUDGET_S and persons > 1:
        sample = max(1, min(persons, int(persons * REF_BUDGET_S / (probe * (K + W)))))
        assets, in_dict, cfg = make_problem(CFG_ID, sample, args.frames)
        port = CpuPort(assets, in_dict, cfg)
    k_run = K
    if probe * sample / persons * (K + W) > REF_BUDGET_S:
        k_run = max(20, int(REF_BUDGET_S / (probe * sample / persons)) - W)
    cut = False
    try:
        with wall_clock_limit(2.5 * REF_BUDGET_S):
            ts = port.time_iterations(W + k_run, threads=threads)[W:]
    except CpuLegTimeout:                        # host busy with other jobs: report what was timed
        ts, cut = list(port._times[W:]) or [probe * sample / persons], True
        k_run = len(ts)
    med, best = float(np.median(ts)), float(np.min(ts))
    units = sample * args.frames
    val = units / med
    out = {
        'impl': 'reference', 'metric': 'global_opt_frame_person_iterations_per_sec', 'value': val, 'unit': 'frame*person*iter/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': med * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'iters_per_sec': 1.0 / med, 'value_best': units / best,
        'config': {'workload': f'{CFG_ID}:init_opt, {persons} person(s) x {args.frames} frames, full-LBS every iteration', 'persons': persons,
                   'frames': args.frames},
        'cpu_baseline': {'value': val, 'value_best': units / best, 'unit': 'frame*person*iter/s', 'cores': threads, 'host_threads_available': host_threads(),
                         'kind': 'port', 'thread_sweep_ms_per_iter': {str(k): round(v * 1e3, 2) for k, v in sweep_res.items()},
                         'ms_per_iter_list': [round(t * 1e3, 1) for t in ts],
                         'sample': f'{k_run} timed iterations (median; best in value_best) after {W} warm-up of the oracle port (torch CPU, {threads} threads = '
                                   f'fastest of the sweep), each over {sample} of the {persons} person(s) x {args.frames} frames' + (' (cut by the wall-clock limit)' if cut else '')},
        'e2e': {'value': val, 'unit': 'frame*person*iter/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------------- GPU arm
def nbytes(x):
    import torch
    if isinstance(x, np.ndarray):
        return x.nbytes
    if isinstance(x, torch.Tensor):
        return x.numel() * x.element_size()
    if isinstance(x, dict):
        return sum(nbytes(v) for v in x.values())
    return 0


def _dbg(*a):
    if os.environ.get('BENCH_DEBUG'):
        print(f'[bench rank {os.environ.get("RANK", 0)}] {time.time() % 1000:.1f}', *a, file=sys.stderr, flush=True)


class Ctx:
    """per-process state shared by the headline run and the extras"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from glamr_b200.motion_traj import MotionTrajJointModel
        from glamr_b200.smpl import SMPL
        from glamr_b200.synthetic import make_smpl_assets
        from glamr_b200.synthetic_nets import make_prior_states
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get('WORLD_SIZE', 1))
        self.rank = int(os.environ.get('RANK', 0))
        self.local = int(os.environ.get('LOCAL_RANK', 0))
        torch.cuda.set_device(self.local)
        self.dev = torch.device('cuda', self.local)
        if self.world > 1:
            dist.init_process_group('nccl', device_id=self.dev)
        self.assets = make_smpl_assets(0)
        self.smpl = SMPL(self.assets, device=self.dev)
        self.prior = MotionTrajJointModel(None, self.dev, None, smpl=self.smpl, states=make_prior_states(1234))
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)

    def model(self, cfg, graph=True, sharded=True):
        from glamr_b200.recon import GlobalReconOptimizer
        from glamr_b200.synthetic import LatentInjector
        c = copy.deepcopy(cfg)
        c.grecon_model_specs['use_cuda_graph'] = graph
        return GlobalReconOptimizer(c, self.dev, None, smpl=self.smpl, mt_model=LatentInjector(self.prior, 0),
                                    dist=(self.rank, self.world) if (self.world > 1 and sharded) else None)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


class StageLoop:
    """one stage of one model set up for timing: `step()` runs ONE optimiser iteration (a replayed CUDA graph of backward
    [+ all-reduce] + Adam when capture works)"""

    def __init__(self, ctx, model, data, stage, specs, hist_rows, warmup):
        from glamr_b200 import lib as L
        torch = ctx.torch
        self.ctx, self.model = ctx, model
        model._cur_vars, model._cur_stage, model._loss_cfg = specs['opt_variables'], stage, specs['loss_cfg']
        model._set_stage(data, specs['opt_variables'], specs['loss_cfg'], stage, reset_adam=True, begin=True)
        self.hist = torch.zeros((hist_rows, L.NUM_TERMS + 1), device=ctx.dev)
        lib, lr = model._lib, float(specs['opt_lr'])

        self.native = bool(getattr(model, '_peer_ok', False))      # gradient all-reduce over NVLink peer memory inside the Adam kernel
        if ctx.world == 1 or self.native:
            # the library's own iteration (one GPU: Adam fused into the tail of the backward pass; peer path: the all-reduce fused
            # into the Adam kernel), launched eagerly here and captured below into ONE graph per step
            def iteration():
                L.check(lib.glamr_opt_iterate(model._opt, L.ptr(model._theta), L.ptr(model._reduce), lr, L.ptr(self.hist), L.NUM_TERMS + 1,
                                              1, 0, L.stream_ptr()), 'iterate')
        else:
            def iteration():
                model._backward(for_apply=True)            # backward pass + NCCL all-reduce of [grad | term sums]
                L.check(lib.glamr_opt_apply(model._opt, L.ptr(model._theta), L.ptr(model._reduce), lr, L.ptr(self.hist), L.NUM_TERMS + 1,
                                            L.stream_ptr()), 'apply')
        self.iteration = iteration
        self.graph = None
        for _ in range(warmup):
            iteration()
        try:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                iteration()
        except Exception:
            self.graph = None
            torch.cuda.synchronize()
        self.step = self.graph.replay if self.graph is not None else iteration
        for _ in range(3):
            self.step()

    def time(self, K):
        """-> (ms per L2-flushed iteration, ms per back-to-back iteration), each the max over ranks"""
        ctx, torch = self.ctx, self.ctx.torch
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        ctx.barrier()
        for a, b in evs:
            ctx.flush.fill_(1)                   # evict L2 (126 MB) between timed iterations
            a.record()
            self.step()
            b.record()
        ctx.barrier()
        cold = sum(a.elapsed_time(b) for a, b in evs)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            self.step()
        e1.record()
        ctx.barrier()
        warm = e0.elapsed_time(e1)
        cold, warm = ctx.max_over_ranks(cold, warm)
        return cold / K, warm / K

    def lbs_ms(self, n=50):
        """the LBS kernel alone, timed by the library's event pair on the launching stream, L2 flushed before each iteration"""
        from glamr_b200 import lib as L
        lib, model = self.model._lib, self.model
        L.check(lib.glamr_opt_kernel_timing(model._opt, 1), 'timing')
        out, crit, side = [], [], []
        for _ in range(n):
            self.ctx.flush.fill_(1)
            self.iteration()
            ms, c, b = ctypes.c_float(), ctypes.c_float(), ctypes.c_float()
            L.check(lib.glamr_opt_last_lbs_ms(model._opt, ctypes.byref(ms)), 'lbs_ms')
            L.check(lib.glamr_opt_last_lbs_parts_ms(model._opt, ctypes.byref(c), ctypes.byref(b)), 'lbs_parts_ms')
            out.append(ms.value), crit.append(c.value), side.append(b.value)
        L.check(lib.glamr_opt_kernel_timing(model._opt, 0), 'timing')
        self.lbs_parts = {'critical_path_ms': float(np.mean(crit)), 'side_stream_blend_ms': float(np.mean(side))}
        return float(np.mean(out))

    def blend_ms(self, reps=20):
        """the tensor-core blend (feature kernel + GEMM) alone, warm L2; None on the SIMT path"""
        from glamr_b200 import lib as L
        ms = ctypes.c_float()
        rc = self.model._lib.glamr_opt_time_blend(self.model._opt, reps, ctypes.byref(ms))
        return float(ms.value) if rc == 0 else None

    def release(self):
        self.graph, self.step = None, None


PER_PERSON_OUTPUTS = ['smpl_orient_world', 'root_trans_world', 'smpl_orient_world_base', 'root_trans_world_base', 'kp_2d_pred',
                      'smpl_orient_cam_in_world', 'root_trans_cam_in_world', 'joints_world', 'traj_local']
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(model, data, out_dir, rank):
    """Write what the last timed step computed, as optimize_main hands it back to its caller: the optimisation variables
    (theta, every variable of the stage packed) and the per-frame outputs of that step's closure, persons concatenated along
    axis 0.  All float32.  Above DUMP_LIMIT_BYTES each array keeps a fixed seeded sample of its rows, so that two builds run
    with the same arguments write the same elements.  Collective when frame-persons are sharded over ranks; rank 0 writes."""
    model._scatter_outputs(data)
    if rank != 0:
        return None
    import torch
    persons = list(data['person_data'].values())
    arrays = {'theta': model._theta, 'cam_pose': data['cam_pose'], 'cam_pose_inv': data['cam_pose_inv']}
    for k in PER_PERSON_OUTPUTS:
        arrays[k] = torch.cat([d[k] for d in persons])
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    sampled = total > DUMP_LIMIT_BYTES
    if sampled:
        rng = np.random.default_rng(0)
        for k, a in arrays.items():
            n = max(1, a.shape[0] * DUMP_LIMIT_BYTES // total)
            arrays[k] = a[np.sort(rng.choice(a.shape[0], n, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)
    return {'dir': out_dir, 'arrays': sorted(arrays), 'bytes': sum(a.nbytes for a in arrays.values()), 'sampled_rows': sampled}


def measure_fp32_peak(ctx):
    """TFLOP/s of a register-resident FFMA loop on this GPU right now (best of 5 launches of ~1 ms)"""
    from glamr_b200 import lib as L
    torch = ctx.torch
    lib = L.load()
    sms = lib.glamr_device_sm_count()
    scratch = torch.empty(sms * 8 * 256, device=ctx.dev)
    flops = ctypes.c_double()
    best = 0.0
    for i in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(lib.glamr_fp32_probe(4096, L.ptr(scratch), scratch.numel(), ctypes.byref(flops), L.stream_ptr()), 'fp32_probe')
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def e2e_optimize(ctx, cfg, in_dict, niters=None):
    """GlobalReconOptimizer.optimize(host numpy) -> host numpy, second call timed (the first pays one-time CUDA/graph setup)"""
    torch = ctx.torch
    model = ctx.model(cfg)
    if niters is not None:
        for st in model.cfg.opt_stage_specs.values():
            st['opt_niters'] = niters
    model.optimize(copy.deepcopy(in_dict))
    ctx.barrier()
    t0 = time.perf_counter()
    out = model.optimize(copy.deepcopy(in_dict))
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    (secs,) = ctx.max_over_ranks(secs)
    n_stages = len(model.cfg.opt_stage_specs)
    total_iters = sum(st['opt_niters'] for st in model.cfg.opt_stage_specs.values())
    info = {'seconds': secs, 'iterations': total_iters, 'phase_seconds': {k: round(v, 5) for k, v in model.phase_seconds.items()},
            'loop_ms_per_iter': {s: round(ms, 5) for s, _, ms in model.iter_ms[-n_stages:]}}
    h2d = nbytes(in_dict['est'])
    d2h = nbytes({k: v for k, v in out.items() if k != 'gt'})
    del model
    return info, h2d, d2h


def multi_gpu_parity(ctx, cfg, in_dict, iters=20):
    """the sharded job against a single-GPU run of the same problem: max |difference| of every optimisation variable and of
    the per-frame outputs after `iters` iterations of the first stage (rank 0 runs the unsharded copy)"""
    stage, specs = next(iter(cfg.opt_stage_specs.items()))
    ms = ctx.model(cfg)
    ds = ms.init_data(copy.deepcopy(in_dict))
    ms.optimize_main(ds, specs['opt_variables'], specs['opt_lr'], iters, specs['loss_cfg'], {'stage': stage})
    res = None
    if ctx.rank == 0:
        m1 = ctx.model(cfg, sharded=False)
        d1 = m1.init_data(copy.deepcopy(in_dict))
        m1.optimize_main(d1, specs['opt_variables'], specs['opt_lr'], iters, specs['loss_cfg'], {'stage': stage})
        diff = {'theta': float((m1._theta - ms._theta).abs().max()), 'cam_pose': float((d1['cam_pose'] - ds['cam_pose']).abs().max())}
        where = {}
        for k in ['smpl_orient_world', 'root_trans_world', 'kp_2d_pred', 'joints_world', 'smpl_orient_cam_in_world', 'root_trans_cam_in_world']:
            worst = (-1.0, None)
            for pid, (a, b) in enumerate(zip(d1['person_data'].values(), ds['person_data'].values())):
                e = (a[k] - b[k]).abs()
                m = float(e.max())
                if m > worst[0]:
                    pos = [int(i) for i in np.unravel_index(int(e.argmax()), tuple(e.shape))]
                    worst = (m, {'person': pid, 'index': pos, 'single': float(a[k][tuple(pos)]), 'sharded': float(b[k][tuple(pos)])})
            diff[k] = worst[0]
            where[k] = worst[1]
        # a projected keypoint blows up when its joint passes the camera plane (|u| ~ 1e7 px for a synthetic track): compare those relatively
        kp_rel = 0.0
        for a, b in zip(d1['person_data'].values(), ds['person_data'].values()):
            kp_rel = max(kp_rel, float(((a['kp_2d_pred'] - b['kp_2d_pred']).abs() / a['kp_2d_pred'].abs().clamp_min(1000.0)).max()))
        diff['kp_2d_pred_rel_to_max(|u|,1000px)'] = kp_rel
        res = {'max_abs': max(diff['theta'], diff['cam_pose'], diff['smpl_orient_world'], diff['root_trans_world']), 'per_tensor': diff,
               'iterations': iters, 'bound': 1e-5, 'where': where,
               'what': f'{ctx.world}-GPU sharded run vs single-GPU run of the same problem, rank 0; kp_2d_pred in pixels (its worst entry is a projection through the camera plane, see where / the relative figure)'}
        res['ok'] = bool(res['max_abs'] <= res['bound'])
        del m1
    ctx.barrier()
    del ms
    return res


def staged_workload(ctx, cfg_id, persons, frames, K, with_e2e=True, cpu_iters=0, cpu_threads=None):
    """a multi-stage config on one video, frame-persons sharded over the ranks: per-stage iteration times + end to end"""
    assets, in_dict, cfg = make_problem(cfg_id, persons, frames)
    units = persons * frames
    model = ctx.model(cfg)
    data = model.init_data(copy.deepcopy(in_dict))
    res = {'workload': f'{cfg_id}, {persons} persons x {frames} frames, full-LBS every iteration', 'frame_persons': units,
           'parallelism': f'frame-persons sharded over {ctx.world} GPU(s) (fixed video: strong scaling)' if ctx.world > 1 else 'single GPU', 'stages': {}}
    last = list(cfg.opt_stage_specs)[-1]
    for stage, specs in cfg.opt_stage_specs.items():
        loop = StageLoop(ctx, model, data, stage, specs, 4 * K + 64, warmup=5)
        cold, warm = loop.time(K)
        res['stages'][stage] = {'ms_per_iter': cold, 'ms_per_iter_l2_warm': warm, 'value': units / (cold * 1e-3), 'iters_per_sec': 1e3 / cold,
                                'yaml_iterations': specs['opt_niters'], 'cuda_graph': bool(loop.graph is not None)}
        if stage == last:
            res['lbs_kernel_ms'] = loop.lbs_ms(20)
            res['lbs_frame_persons_per_launch'] = model._n_range[1] - model._n_range[0]
        loop.release()
    del model
    res['value'] = res['stages'][last]['value']
    res['unit'] = 'frame*person*iter/s'
    res['ms_per_step'] = res['stages'][last]['ms_per_iter']
    if with_e2e:
        info, h2d, d2h = e2e_optimize(ctx, cfg, in_dict)
        res['e2e'] = {'value': units * info['iterations'] / info['seconds'], 'unit': 'frame*person*iter/s', **info,
                      'h2d_bytes': h2d, 'd2h_bytes': d2h, 'what': 'optimize(in_dict numpy) -> numpy dict incl. init_data, all YAML iterations of both stages'}
    if cpu_iters and ctx.rank == 0 and ctx.world == 1:
        # this leg may use at most a third of the run's CPU budget: the headline workload's leg comes last
        pool0 = wall_clock_limit.pool
        if pool0 is not None:
            wall_clock_limit.pool = pool0 / 3.0
        res['cpu_baseline'] = cpu_baseline_block(assets, in_dict, cfg, units, cpu_iters, stage=last, sweep=False, threads=cpu_threads, budget_s=30.0)
        if pool0 is not None:
            wall_clock_limit.pool = pool0 - (pool0 / 3.0 - wall_clock_limit.pool)
    return res


def c3_prior(ctx):
    """BASELINE.json configs[2]: infiller + trajectory predictor, 64 sequences x 120 frames (frames 40-69 masked), ms per batch"""
    torch = ctx.torch
    g = torch.Generator().manual_seed(0)
    B, T = 64, 120
    pose = (torch.randn(B, T, 69, generator=g) * 0.3).to(ctx.dev)
    mask = torch.ones(B, T, device=ctx.dev)
    mask[:, 40:70] = 0
    batch = {'in_body_pose': pose * mask[..., None], 'frame_mask': mask, 'in_motion_latent': torch.randn(4, 128, generator=g).to(ctx.dev),
             'in_traj_latent': torch.randn(1, 128, generator=g).to(ctx.dev)}
    for _ in range(3):
        ctx.prior.inference(batch)
    ts = []
    for _ in range(10):
        ctx.flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.prior.inference(batch)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = float(np.median(ts))
    return {'workload': 'motion_infiller + traj_pred inference, 64 x 120 frames, frames 40-69 masked (replicated per rank, rank 0 reported)',
            'ms_per_batch': ms, 'sequences_per_sec': B / (ms * 1e-3), 'frames_per_sec': B * T / (ms * 1e-3), 'algorithmic_gflop': 94.0,
            'tflops_algorithmic': 94.0 / ms, 'weights': 'seeded stand-ins (no checkpoints offline)'}


def c5_sweep(ctx, n_seq=32, frames=300):
    """BASELINE.json configs[4]: 32 independent 300-frame sequences with occlusion gaps, full infill -> trajectory ->
    glamr_3dpw optimisation (200 + 500 iterations) through run_dataset; sequences are replicas over the ranks"""
    import shutil
    from glamr_b200.global_recon import run_dataset as RD
    from glamr_b200.recon import GlobalReconOptimizer
    out_dir = f'/tmp/glamr_b200_bench_c5_rank{ctx.rank}'
    shutil.rmtree(out_dir, ignore_errors=True)
    a = RD.parse(['--cfg', 'glamr_3dpw', '--out_dir', out_dir, '--synthetic', str(n_seq), '--frames', str(frames), '--gaps', '--quiet'])
    models = []

    def make_model(cfg, local):
        m = GlobalReconOptimizer(cfg, ctx.dev, None, smpl=ctx.smpl, mt_model=ctx.prior)
        models.append(m)
        return m
    # the HybrIK-shaped inputs of this rank's sequences are generated BEFORE the timed region (data generation is not the path)
    from glamr_b200.synthetic import make_in_dict as synth
    names = RD.shard(RD.list_sequences(a), ctx.rank, ctx.world)
    inputs = {n: synth(ctx.assets, 1, frames, seed=int(n.rsplit('_', 1)[1]), gaps=True, seq_name=n) for n in names}
    ctx.barrier()
    t0 = time.perf_counter()
    done = RD.run(a, make_model=make_model, make_in_dict=lambda n: copy.deepcopy(inputs[n]))
    ctx.torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    (secs,) = ctx.max_over_ranks(secs)
    iters = sum(st['opt_niters'] for st in models[0].cfg.opt_stage_specs.values())
    shutil.rmtree(out_dir, ignore_errors=True)
    return {'workload': f'{n_seq} independent sequences x {frames} frames (3DPW-like gaps), glamr_3dpw, infill -> trajectory -> {iters} iterations each, '
                        f'pickle written per sequence; replicas over {ctx.world} GPU(s)',
            'seconds': secs, 'sequences_per_sec': n_seq / secs, 'value': n_seq * frames * iters / secs, 'unit': 'frame*person*iter/s',
            'sequences_this_rank': len(done), 'ms_per_sequence_this_rank': float(np.mean([d[3] for d in done]) * 1e3) if done else None}


def run_ours(args):
    refuse_experiment_switches()
    # all CPU legs of this run (main cpu_baseline + the north-star one) share one wall-clock budget: the GPU numbers must not wait for a busy host
    wall_clock_limit.pool = float(os.environ.get('GLAMR_CPU_BUDGET_S', 180.0))
    ctx = Ctx()
    torch, world, rank = ctx.torch, ctx.world, ctx.rank
    persons = args.persons or world
    assets, in_dict, cfg = make_problem(CFG_ID, persons, args.frames)
    stage, specs = next(iter(cfg.opt_stage_specs.items()))
    K, W = args.steps, max(args.warmup, 3)
    _dbg('problem made')

    # ---------------- device-resident timing: K iterations, L2 flushed between iterations, CUDA events per iteration
    model = ctx.model(cfg)
    data = model.init_data(copy.deepcopy(in_dict))
    loop = StageLoop(ctx, model, data, stage, specs, W + 3 * K + 256, warmup=W)
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()
    cold_ms, warm_ms = loop.time(K)
    clocks = sampler.stop() if rank == 0 else None
    _dbg('timed loops done')
    # before lbs_ms below, which runs further iterations of the same model
    dumped = dump_outputs(model, data, args.dump_outputs, rank) if args.dump_outputs else None
    lbs_ms = loop.lbs_ms(min(K, 50))
    blend_ms = loop.blend_ms()
    lbs_parts = dict(getattr(loop, 'lbs_parts', {}))
    n_local = model._n_range[1] - model._n_range[0]
    peer = bool(getattr(model, '_peer_ok', False))
    graph_on = bool(loop.graph is not None)
    launches_per_iter = model.launches_per_iteration()
    loop.release()
    del model, loop
    fp32_peak = measure_fp32_peak(ctx)
    _dbg('lbs / fp32 peak done')

    # ---------------- end to end through the public API with host buffers
    e2e_info, h2d, d2h = e2e_optimize(ctx, cfg, in_dict, niters=K)
    _dbg('e2e done')
    parity = multi_gpu_parity(ctx, cfg, in_dict) if world > 1 else None

    # ---------------- extras
    want = ALL_EXTRAS if args.extras == 'all' else ([] if args.extras == 'none' else args.extras.split(','))
    extras = {}
    Kx = min(K, 100)
    def in_budget(name):
        """same decision on every rank (the extras contain collectives)"""
        (el,) = ctx.max_over_ranks(time.perf_counter() - T_START)
        if el > 0.6 * BENCH_BUDGET_S:
            extras[name] = {'skipped': f'{el:.0f} s of the {BENCH_BUDGET_S:.0f} s bench budget were spent before this extra (busy host); run `python bench.py --extras {name}`'}
            return False
        return True
    if 'north_star' in want and in_budget('north_star'):
        extras['north_star'] = staged_workload(ctx, 'glamr_static_multi', 4, 300, Kx, cpu_iters=0 if args.no_cpu_baseline else 8)
        _dbg('north_star done')
    if 'c4' in want and in_budget('c4'):
        extras['c4'] = staged_workload(ctx, 'glamr_static_multi', 8, 500, min(Kx, 50), with_e2e=False)
        _dbg('c4 done')
    if 'c3' in want and in_budget('c3'):
        r = c3_prior(ctx)
        if rank == 0:
            extras['c3'] = r
        _dbg('c3 done')
    if 'c5' in want and in_budget('c5'):
        extras['c5'] = c5_sweep(ctx)
        _dbg('c5 done')

    bad = False
    if rank == 0:
        units = persons * args.frames
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        hbm_peak = peaks.get('hbm_gbs', 6650.0)
        alg_bytes = BYTES_CONST + n_local * BYTES_PER_FP
        achieved = alg_bytes / (lbs_ms * 1e-3) / 1e9
        fp32_tf = FLOPS_PER_FP * n_local / (lbs_ms * 1e-3) / 1e12
        fp32_exec = FLOPS_PER_FP_EXECUTED * n_local / (lbs_ms * 1e-3) / 1e12
        hbm_roofline = {'bound': 'hbm', 'kernel': 'LBS of the iteration: lbs_blend_tc_kernel (+ feature kernel) + lbs_skin_tc_kernel', 'achieved': achieved, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': achieved / hbm_peak,
                         'traffic': NCU_LBS_DRAM_BYTES.get(n_local), 'traffic_source': 'profiles/ (ncu --set full, dram__bytes_read + write, per launch)' if n_local in NCU_LBS_DRAM_BYTES else None,
                         'peak_source': 'MEASURED_PEAKS.json hbm_gbs' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s',
                         'algorithmic_bytes': alg_bytes, 'kernel_ms': lbs_ms, 'kernel_share_of_step': lbs_ms / cold_ms,
                         'kernel_parts': {**lbs_parts,
                                          'note': 'kernel_ms = skinning (on the critical path) + blend timed in situ on its side stream, where it overlaps the other kernels of the evaluation, '
                                                  'so kernel_share_of_step counts overlapped time; both with L2 flushed. traffic (ncu, cold) is 3.3x the algorithmic bytes: the 3xTF32 hi/lo '
                                                  'constant image is 2 x 18.6 MB and v_posed makes one 25 MB round trip through L2/HBM between the two kernels; back-to-back iterations keep both in the 126 MB L2'},
                         'tensor': None if blend_ms is None else {
                             'kernel': 'blend_features_kernel + lbs_blend_tc_kernel launched alone (warm L2)', 'kernel_ms': blend_ms,
                             'achieved_tflops_tf32': 3 * 2 * 224 * 20736 * (-(-n_local // 128) * 128) / (blend_ms * 1e-3) / 1e12,
                             'peak_tflops_tf32': peaks.get('bf16_tflops', 2250.0) / 2,
                             'frac': 3 * 2 * 224 * 20736 * (-(-n_local // 128) * 128) / (blend_ms * 1e-3) / 1e12 / (peaks.get('bf16_tflops', 2250.0) / 2),
                             'note': '3xTF32: three kind::tf32 MMAs per product; peak = half of the measured dense bf16 throughput (MEASURED_PEAKS.json); '
                                     'ncu: sm__pipe_tensor_cycles_active 56.6 % of peak, 167 MB L2->SM per launch (profiles/lbs_tc_kernels_r02_final.md)'},
                         'fp32': {'achieved_tflops': fp32_tf, 'executed_tflops': fp32_exec, 'peak_tflops': fp32_peak, 'frac': fp32_tf / fp32_peak, 'frac_executed': fp32_exec / fp32_peak,
                                  'peak_source': 'glamr_fp32_probe: register-resident FFMA loop timed in this run (best of 5)',
                                  'note': 'algorithmic LBS flops (15.85 MFLOP per frame-person, dense skinning) over the LBS time (blend GEMM timed in situ on its side stream + skinning kernel) against the measured FP32 FFMA peak; '
                                          'both LBS kernels run on the tensor cores now (3xTF32: the top-level roofline is the blend; the skinning is a K = 24 GEMM whose time is its TMEM epilogue and operand loads), so this FP32-FMA fraction is a comparison figure against the round-1 SIMT kernel, not a bound; the HBM fraction is small by construction (constants stay L2-resident)'}}
        tensor = hbm_roofline.pop('tensor')
        if tensor is not None:
            # the dominant kernel of the iteration is the tensor-core blend GEMM: quote the roofline against the tensor pipe.  Algorithmic flops =
            # the blend contraction of lbs.py:240,256-267 (207 pose features + 10 betas per vertex coordinate; the template is an add):
            # 2 x 217 x 20670 per frame-person -- the share of SURVEY 8(d)'s 15.85 MFLOP that this kernel computes.  The kernel ISSUES 3x that
            # (3xTF32) on padded tiles: issued_* below.
            alg_flops = 2.0 * 217 * 20670 * n_local
            tf32_peak = tensor['peak_tflops_tf32']
            ach = alg_flops / (tensor['kernel_ms'] * 1e-3) / 1e12
            roofline = {'bound': 'tensor', 'kernel': 'lbs_blend_tc_kernel (+ blend_features_kernel): the longest kernel of the iteration, launched alone (warm L2)',
                        'achieved': ach, 'peak': tf32_peak, 'unit': 'TFLOP/s', 'frac': ach / tf32_peak,
                        'traffic': NCU_BLEND_DRAM_BYTES.get(n_local), 'traffic_source': 'profiles/lbs_tc_kernels_r02_final.md (ncu --set full, dram read + write of the blend kernel, cold)' if n_local in NCU_BLEND_DRAM_BYTES else None,
                        'peak_source': ('MEASURED_PEAKS.json bf16_tflops / 2' if 'bf16_tflops' in peaks else 'fallback: nominal 2250 / 2') + ' = dense TF32',
                        'algorithmic_flops': alg_flops, 'kernel_ms': tensor['kernel_ms'],
                        'issued_tflops_tf32': tensor['achieved_tflops_tf32'], 'issued_frac': tensor['frac'],
                        'note': 'frac = algorithmic blend flops / time / dense TF32 peak; issued_frac counts the three kind::tf32 MMAs per product (3xTF32) on 128 x 256 tiles '
                                '(ncu: tensor pipe active 48 % of the cycles at 300 frames, 0.71 of peak issue at 1200 frames, profiles/chain_analysis_r02.md)',
                        'hbm': hbm_roofline, 'fp32': hbm_roofline.pop('fp32'), 'kernel_parts': hbm_roofline.pop('kernel_parts')}
        else:
            roofline = hbm_roofline
        res = {
            'metric': 'global_opt_frame_person_iterations_per_sec', 'value': units / (cold_ms * 1e-3), 'unit': 'frame*person*iter/s',
            'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': cold_ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'iters_per_sec': 1e3 / cold_ms,
            'value_l2_warm': units / (warm_ms * 1e-3), 'ms_per_step_l2_warm': warm_ms,
            'config': {'workload': f'{CFG_ID}:init_opt, {persons} person(s) x {args.frames} frames, full-LBS every iteration',
                       'persons': persons, 'frames': args.frames,
                       'parallelism': (f'frame-persons sharded over {world} GPU(s), ' + ('gradient reduction over NVLink peer memory fused into the Adam kernel' if peer else '1 NCCL allreduce/iter')) if world > 1 else 'single GPU',
                       'l2': 'flushed between timed iterations (256 MiB fill); value_l2_warm = back-to-back replays',
                       'cuda_graph': graph_on, 'prior': 'CUDA infiller+traj-pred with seeded stand-in weights (no checkpoints offline), latents injected',
                       'env': {k: os.environ.get(k) for k in ECHO_ENV if os.environ.get(k) is not None}},
            'clocks': clocks,
            'gpu_launches': launches_per_iter * K,
            'gpu_launches_per_step': launches_per_iter,
            'e2e': {'value': units * K / e2e_info['seconds'], 'unit': 'frame*person*iter/s', 'h2d_bytes_per_step': h2d / K, 'd2h_bytes_per_step': d2h / K,
                    'what': f'GlobalReconOptimizer.optimize(in_dict numpy)->numpy dict incl. init_data, {K} iterations', **e2e_info},
            'roofline': roofline,
            'extras': extras,
        }
        if dumped is not None:
            res['outputs_dump'] = dumped
        if parity is not None:
            res['parity'] = parity
            bad = not parity['ok']
        if world == 1 and not args.no_cpu_baseline:
            left = BENCH_BUDGET_S - (time.perf_counter() - T_START)
            wall_clock_limit.pool = max(25.0, min(wall_clock_limit.pool if wall_clock_limit.pool is not None else 180.0, left))
            res['cpu_baseline'] = cpu_baseline_block(assets, in_dict, cfg, units, args.cpu_sample_iters)
        elif world > 1:
            res['cpu_baseline'] = {'skipped': 'N > 1: the reference arm (--impl reference) times the CPU path; rank 0 does not stall the other GPUs'}
        print(json.dumps(res))
    if world > 1:
        # captured graphs hold NCCL work: leave without the interpreter's shutdown path (a destroy with live captures can block)
        torch.cuda.synchronize()
        ctx.dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(1 if bad else 0)
    if bad:
        sys.exit(1)


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
