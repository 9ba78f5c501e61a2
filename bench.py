#!/usr/bin/env python
"""Benchmark of the nmrfit objective-evaluation hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload metric|c1|c2|c3|c4]
                    [--dump-outputs DIR]

Headline workload (`metric`): the shape BASELINE.json's metric string is quoted on - 6 peaks on a 4,096-point
window (the configs[0] spectrum) - with one swarm generation of 65,536 particles per GPU as the batch.  A *step* is
one swarm generation on the device: velocity/position update (device Philox), objective of every particle, personal
bests, swarm best (+ one best-record exchange when the particles are sharded over N > 1 GPUs; weak scaling: each rank
holds 65,536 particles of one 65,536*N-particle swarm).

One JSON line on stdout (rank 0):
  value      objective evaluations per second over all GPUs, everything resident in HBM (CUDA events, max over ranks);
  e2e        the same metric through the public host-buffer call (`equations.objective_batch`): particle positions
             copied H2D and objective values copied D2H inside the timed region, every step;
  roofline   the evaluation kernel against the FP64 pipe: EXECUTED FP64 instructions (ncu count per peak-point of the
             same kernel and workload, profiles/objective_ncu.json, times the peak-points of a launch) over the kernel's
             CUDA-event time, divided by the DFMA issue rate measured in this run - a hardware fraction <= 1.  The
             ratio of SURVEY.md 8(d)'s canonical cost model to what the kernel executes is `algorithmic_speedup`;
  secondary  the other BASELINE configs (C2, C3, C4) measured in the same run with fewer steps;
  cpu_baseline  the UNMODIFIED reference objective (baseline/_ref) on the host cores, bounded sample.

`--impl reference` times the CPU arm alone on the same config: `nmrfit.equations.objective` of the unmodified
reference package called once per particle over a multiprocessing pool with every host core - what
`nmrfit.fit(..., processes=N)` does through pyswarm.  Each step is a bounded sample of the generation.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json "metric": "Voigt objective evals/s (6 peaks, 4k pts)"
    'metric': dict(P=6, N=4096, S=65536, seed=1000,
                   title='BASELINE metric shape: 6 peaks, 4,096-point window (the configs[0] spectrum), one swarm generation '
                         'of 65,536 particles per GPU, FP64 objective'),
    'c1': dict(P=6, N=4096, S=100, seed=1000,
               title='BASELINE configs[0] C1: 6 peaks, 4,096 points, swarmsize 100 (launch-latency bound per-step path)'),
    'c2': dict(P=12, N=32768, S=4096, seed=2000,
               title='BASELINE configs[1] C2: single fit, 12 peaks, 32,768-point window, swarmsize 4,096 per GPU, FP64 objective'),
    # BASELINE configs[2]: 1,024 independent spectra, one swarm of 204 (the reference default) each; the
    # spectra are split over the ranks (strong scaling, no data-path collective)
    'c3': dict(P=6, N=16384, S=204, seed=3000, B=1024,
               title='BASELINE configs[2] C3: 1,024 independent spectra (6 peaks, 16,384 points), one swarm of 204 '
                     'particles each, FP64 objective'),
    # BASELINE configs[3]: 65,536 particles on one 24-peak 64k-point spectrum over 8 GPUs -> 8,192 per GPU
    'c4': dict(P=24, N=65536, S=8192, seed=4000,
               title='BASELINE configs[3] C4: one 24-peak 65,536-point spectrum, 8,192 particles per GPU (65,536 over 8 GPUs), '
                     'FP64 objective'),
}
METRIC = 'voigt_objective_evals_per_s'
PSO = dict(omega=-0.2134, phip=-0.3344, phig=2.3259)


def flop_per_eval(n_points, n_peaks):
    """SURVEY.md section 8(d) canonical cost model: 50 FP64 flop per peak-point + 20 per (particle, point)."""
    return n_points * (50 * n_peaks + 20)


def make_inputs(name):
    from nmrfit_b200 import synth, utils
    wl = WORKLOADS[name]
    data, true = synth.multiplet(wl['N'], wl['P'], seed=wl['seed'])
    weights = utils.compute_weights(data.w, data.peaks)
    lo, up = data.generate_solution_bounds()
    return data, weights, np.array(lo), np.array(up), true


def workload_config(name, gpus, exchange='p2p'):
    wl = WORKLOADS[name]
    if 'B' in wl:
        return {'workload': wl['title'], 'n_peaks': wl['P'], 'n_points': wl['N'], 'particles_per_swarm': wl['S'],
                'spectra_total': wl['B'], 'spectra_per_gpu': wl['B'] // gpus,
                'parallelism': 'spectra sharded over %d GPU(s), no data-path collective' % gpus,
                'l2': 'working set (spectra + swarm constants) exceeds L2; also flushed between timed steps'}
    return {'workload': wl['title'], 'n_peaks': wl['P'], 'n_points': wl['N'], 'particles_per_gpu': wl['S'],
            'swarm_total': wl['S'] * gpus,
            'parallelism': 'particles sharded over %d GPU(s), one best-record %s per generation'
                           % (gpus, 'exchange over peer memory inside the finish kernel (NVLink stores)' if exchange == 'p2p'
                              else 'NCCL all-gather'),
            'l2': 'flushed between timed steps (256 MiB fill outside the per-step event brackets)'}


# ---------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference objective over all host cores (oracle port only when baseline/_ref is absent)
# ---------------------------------------------------------------------------------------------
_pool_args = None
_pool_fn = None


def _cpu_objective():
    """(callable objective(x, w, u, v, weights, fit_im), kind).  kind 'reference' = nmrfit.equations.objective of the
    unmodified reference package; 'port' = oracle/nmrfit_oracle.py (bit-identical on the golden vectors)."""
    from oracle import ref_loader                      # CPU baseline leg: the one place bench.py touches oracle/
    try:
        ref = ref_loader.load_reference()
        return ref.equations.objective, 'reference'
    except ImportError:
        from oracle import nmrfit_oracle as orc
        return orc.objective, 'port'


def _pool_init(fn, w, u, v, weights):
    global _pool_args, _pool_fn
    _pool_fn, _pool_args = fn, (w, u, v, weights)


def _pool_eval(x):
    return _pool_fn(x, *_pool_args, False)


def cpu_arm(name, n_particles, repeats, cores=None):
    """evals/s of the reference numpy objective, one call per particle, Pool.map over `cores` processes."""
    import multiprocessing as mp
    from nmrfit_b200 import synth
    fn, kind = _cpu_objective()
    data, weights, lo, up, _ = make_inputs(name)
    xs = synth.particles(lo, up, n_particles, seed=7)
    cores = cores or os.cpu_count() or 1
    ctx = mp.get_context('fork')
    times = []
    with ctx.Pool(cores, initializer=_pool_init, initargs=(fn, data.w, data.u, data.v, weights)) as pool:
        pool.map(_pool_eval, list(xs[:cores]))                     # warm the workers
        for _ in range(repeats):
            t0 = time.perf_counter()
            pool.map(_pool_eval, list(xs))
            times.append(time.perf_counter() - t0)
    return n_particles / np.array(times), cores, kind


def cpu_fit_c1():
    """configs[0] on one host core, as BASELINE.md section 3 specifies: the reference's own nmrfit.fit / FitUtility with
    the restated pyswarm loop bound as `pyswarm` (oracle/pso_oracle.py; pyswarm itself is not installable here)."""
    from oracle import ref_loader, nmrfit_oracle as orc, pso_oracle
    import contextlib
    import io
    data, weights, lo, up, _ = make_inputs('c1')
    np.random.seed(0)
    try:
        ref = ref_loader.load_reference()
        rd = ref_loader.reference_data(ref, data)
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            fit = ref.fit(rd, list(lo), list(up), summary=False, options={'swarmsize': 100, 'maxiter': 100})
        dt = time.perf_counter() - t0
        kind, err = 'reference nmrfit.fit + restated pyswarm.pso', float(fit.error)
    except ImportError:
        t0 = time.perf_counter()
        x, err, info = pso_oracle.pso(orc.objective, lo, up, args=(data.w, data.u, data.v, weights, False),
                                      swarmsize=100, maxiter=100, quiet=True, **PSO)
        dt = time.perf_counter() - t0
        kind = 'oracle port + restated pyswarm.pso'
    return {'c1_fit_seconds_one_core': dt, 'c1_fits_per_s_one_core': 1.0 / dt, 'c1_fit_kind': kind, 'c1_fit_error': err}


def reference_sample(name, cores):
    """Particles per step of the CPU arm: about one second of wall time per step (0.8 ms per evaluation per core at
    6 peaks x 4,096 points, scaling with n_points * n_peaks)."""
    wl = WORKLOADS[name]
    return int(min(wl['S'], max(cores, 1000 * cores * 24576.0 / (wl['N'] * wl['P']))))


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    sample = reference_sample(args.workload, cores)
    rates, cores, kind = cpu_arm(args.workload, sample, args.warmup + args.steps)
    rates = rates[args.warmup:]
    value = float(sample * len(rates) / np.sum(sample / rates))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'evals/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': float(1e3 * np.mean(sample / rates)),
        'higher_is_better': True, 'scaling': 'strong' if 'B' in wl else 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic', 'config': workload_config(args.workload, args.gpus),
        'cpu_baseline': {'value': value, 'unit': 'evals/s', 'cores': cores, 'kind': kind,
                         'sample': '%d particles per step (of %d), %s once per particle over a %d-process pool'
                                   % (sample, wl['S'], 'nmrfit.equations.objective of the unmodified reference (baseline/_ref)'
                                      if kind == 'reference' else 'numpy oracle port of the reference objective', cores)},
        'e2e': {'value': value, 'unit': 'evals/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'peak_points_per_s': value * wl['N'] * wl['P'],
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------
# clocks: NVML polled from a thread every ~2 ms (the timed region is tens of milliseconds), nvidia-smi as fallback
# ---------------------------------------------------------------------------------------------
def _nvml_index(local):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES', '')
    try:
        ids = [int(t) for t in vis.split(',') if t.strip() != '']
        return ids[local] if ids else local
    except (ValueError, IndexError):
        return local


class ClockSampler:
    def __init__(self, local):
        self.rows, self.local, self.stop_flag, self.thread, self.source = [], local, False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(_nvml_index(self.local))
            self.nv = pynvml
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.source = 'nvml'
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
        except Exception:
            self.source = 'nvidia-smi'
            try:
                self.proc = subprocess.Popen(
                    ['nvidia-smi', '-i', str(_nvml_index(self.local)),
                     '--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
                     'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
                     'clocks_event_reasons.sw_power_cap', '--format=csv,noheader,nounits', '-lms', '20'],
                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except OSError:
                self.source = None
                return
            self.thread = threading.Thread(target=self._poll_smi, daemon=True)
        self.thread.start()

    def _poll_nvml(self):
        nv = self.nv
        names = (('hw_slowdown', nv.nvmlClocksEventReasonHwSlowdown), ('hw_thermal_slowdown', nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ('sw_thermal_slowdown', nv.nvmlClocksEventReasonSwThermalSlowdown), ('sw_power_cap', nv.nvmlClocksEventReasonSwPowerCap))
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                power = nv.nvmlDeviceGetPowerUsage(self.h) / 1e3
                self.rows.append((time.perf_counter(), sm, self.smax, power, [n for n, bit in names if mask & bit]))
            except Exception:
                pass
            time.sleep(0.002)

    def _poll_smi(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(',')]
            try:
                reasons = [n for n, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), parts[3:7])
                           if val.lower().startswith('active')]
                self.rows.append((time.perf_counter(), float(parts[0]), float(parts[1]), float(parts[2]), reasons))
            except (ValueError, IndexError):
                continue

    def stop(self, t0, t1):
        self.stop_flag = True
        if self.source is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no clock source (NVML and nvidia-smi unavailable)']}
        if self.source == 'nvidia-smi':
            self.proc.terminate()
        else:
            self.thread.join(timeout=1.0)
        inside = [r for r in list(self.rows) if t0 <= r[0] <= t1]
        near = inside or [r for r in list(self.rows) if t0 - 0.1 <= r[0] <= t1 + 0.1]
        reasons = sorted({n for r in near for n in r[4]})
        out = {'sm_mhz': float(np.median([r[1] for r in near])) if near else None,
               'sm_max_mhz': near[0][2] if near else None,
               'power_w_max': max(r[3] for r in near) if near else None,
               'samples_in_timed_region': len(inside), 'source': self.source, 'reasons': reasons}
        if not inside:
            out['note'] = 'no sample fell inside the timed region; the values are from within 100 ms of it'
        return out


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
class SwarmRun:
    """One BASELINE workload set up on this rank's GPU: spectra resident, swarm initialised, `step()` = one generation."""

    def __init__(self, name, world, rank, local, exchange='p2p', tune='', particles=None):
        import torch
        import torch.distributed as dist
        from nmrfit_b200 import _cabi, swarm, synth, utils
        self.torch, self.dist = torch, dist
        wl = WORKLOADS[name]
        self.name, self.world, self.rank, self.local = name, world, rank, local
        self.P, self.N, self.S = wl['P'], wl['N'], int(particles or wl['S'])
        self.D = 4 + 3 * self.P
        self.batched = 'B' in wl
        self.B = wl['B'] // world if self.batched else 1
        self.stream = torch.cuda.current_stream().cuda_stream
        self.ctx = ctx = _cabi.Context(self.B, self.N, self.P, device=local)
        if tune:
            th, r, tb, sp = (int(t) for t in tune.split(','))
            ctx.set_tuning(th, r, tb, sp)
        if self.batched:
            W, U, V, WT, los, ups = [], [], [], [], [], []
            for bb in range(self.B):
                d, _ = synth.multiplet(self.N, self.P, seed=wl['seed'] + rank * self.B + bb)
                W.append(d.w); U.append(d.u); V.append(d.v); WT.append(utils.compute_weights(d.w, d.peaks))
                l, u_ = d.generate_solution_bounds()
                los.append(l); ups.append(u_)
            ctx.set_spectra(np.array(W), np.array(U), np.array(V), np.array(WT))
            self.lo, self.up = np.array(los), np.array(ups)
            self.data, self.weights = None, None
        else:
            self.data, self.weights, self.lo, self.up, _ = make_inputs(name)
            ctx.set_spectrum(0, self.data.w, self.data.u, self.data.v, self.weights)
        off = 0 if self.batched else rank * self.S
        opts = swarm._make_opts(self.S, 10 ** 9, PSO['omega'], PSO['phip'], PSO['phig'], 0.0, 0.0, False, 1234, offset=off,
                                spectrum_offset=rank * self.B if self.batched else 0)
        opts.minstep = -1.0      # never stop early: every timed step does the full generation's work
        opts.minfunc = -1.0
        self.sharded = world > 1 and not self.batched
        self.p2p = self.sharded and exchange == 'p2p'
        self.exchange_note = None
        if self.p2p:
            # map every rank's exchange window (CUDA IPC).  Every rank must end up on the same path: if the mapping
            # fails anywhere (IPC not permitted on the box) all ranks take the NCCL all-gather instead, and say so
            ok, err = 1, ''
            try:
                handle, _ = ctx.peer_export(world, rank)
                handles = [None] * world
                dist.all_gather_object(handles, handle)
                ctx.peer_open(ipc_handles=handles)
            except Exception as e:                          # noqa: BLE001 - reported, not swallowed
                ok, err = 0, str(e)
                if 'handles' not in locals():
                    dist.all_gather_object([None] * world, None)
            flag = torch.tensor([ok], device='cuda')
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                self.p2p = False
                self.exchange_note = 'peer-memory exchange unavailable (%s): NCCL all-gather used' % (err or 'failed on another rank')
            dist.barrier()
        ctx.pso_begin(self.lo, self.up, opts, stream=self.stream)
        self.rec = None
        if self.sharded and not self.p2p:
            ptr, nrec = ctx.pso_record()
            self.rec = torch.as_tensor(swarm._DeviceArray(ptr, nrec), device='cuda:%d' % local)
        self._gather = swarm.gather_records
        self.commit()
        self.generations = 0

    def commit(self):
        if self.p2p:
            self.ctx.pso_commit_peers(stream=self.stream)
        elif self.sharded:
            self.ctx.pso_commit(self._gather(self.rec), self.world, stream=self.stream)
        else:
            self.ctx.pso_commit(stream=self.stream)

    def step(self):
        if self.p2p:
            self.ctx.pso_step_peers(stream=self.stream)     # particle-sharded, records exchanged over peer memory
        elif self.sharded:
            self.ctx.pso_advance(stream=self.stream)        # particle-sharded: advance, all-gather the best records, commit
            self.commit()
        else:
            self.ctx.pso_step(stream=self.stream)           # the swarm lives in this context: one call, three launches
        self.generations += 1

    def sync_all(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, steps, warmup, flush, sampler=None):
        """W untimed + K timed generations; per-step CUDA events on the launching stream, L2 flushed between steps.
        Returns a dict: total_ms (max over ranks), step_ms, kernel split, launches, wall-clock bracket."""
        from nmrfit_b200 import _cabi
        torch, dist = self.torch, self.dist
        for _ in range(warmup):
            self.step()
        self.sync_all()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.ctx.profile(True)
        launches0 = _cabi.launch_count()
        self.sync_all()
        t0 = time.perf_counter()
        for a, b in ev:
            flush.fill_(1)
            a.record()
            self.step()
            b.record()
        self.sync_all()
        t1 = time.perf_counter()
        launches = _cabi.launch_count() - launches0
        prep_ms, eval_ms, kernel_launches = self.ctx.profile_read_split()
        self.ctx.profile(False)
        step_ms = np.array([a.elapsed_time(b) for a, b in ev])
        total = torch.tensor([float(step_ms.sum())], dtype=torch.float64, device='cuda')
        if self.world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        return dict(total_ms=float(total.item()), step_ms=step_ms, prep_ms=prep_ms, eval_ms=eval_ms,
                    kernel_launches=kernel_launches, launches=int(launches), t0=t0, t1=t1)

    def check_state(self, expect_generations):
        """Every generation ran, nothing stopped, the best is finite - and, when the particles are sharded, the swarm
        best (position, value, generation count) is bit-identical on all ranks."""
        torch, dist = self.torch, self.dist
        x, f, it, stop = self.ctx.pso_best()
        assert np.all(it == expect_generations) and np.all(np.isfinite(f)) and np.all(stop == 0), (it, f, stop)
        same = None
        if self.sharded:
            blob = torch.tensor(np.concatenate([x.ravel(), f, it.astype(float)]), device='cuda')
            parts = [torch.empty_like(blob) for _ in range(self.world)]
            dist.all_gather(parts, blob)
            same = all(torch.equal(p, parts[0]) for p in parts)
            assert same, 'swarm best differs between ranks'
        return same

    def evals_per_step(self):
        return self.S * self.B * self.world

    def close(self):
        if self.world > 1:
            self.dist.barrier()                             # nobody unmaps a window a peer may still store into
        self.ctx.close()


def load_ncu(name):
    path = os.path.join(ROOT, 'profiles', 'objective_ncu.json')
    if not os.path.exists(path):
        return None
    return json.load(open(path)).get(name)


def roofline(name, run, res, burst, sustained, sm_mhz=None):
    """The evaluation kernel against the FP64 pipe.  `achieved` counts what the hardware EXECUTED: FP64 instructions
    per peak-point from the ncu capture of this kernel on this workload x the peak-points of a launch / the kernel's
    CUDA-event time, two flop per instruction slot (the DFMA convention of the measured peak) - so achieved / peak is
    the fraction of the FP64 pipe's issue slots the kernel filled."""
    from nmrfit_b200 import _cabi
    P, N = run.P, run.N
    n = max(res['kernel_launches'], 1)
    eval_ms, prep_ms = res['eval_ms'] / n, res['prep_ms'] / n
    pp = float(run.S) * run.B * N * P                      # peak-points per launch on this GPU
    ncu = load_ncu(name)
    uniform = run.ctx.get_algorithm() == _cabi.ALGO_UNIFORM
    out = {'bound': 'fp64', 'unit': 'TFLOP/s', 'peak': sustained, 'peak_burst': burst,
           'peak_source': 'DFMA probe (nmrfit_fp64_peak) measured in this run, back-to-back average (burst %.2f); '
                          'MEASURED_PEAKS.json has no FP64 entry' % burst,
           'kernel': ('objective_stream_kernel' if run.ctx.get_variant(run.S)[0] == 1 else 'objective_uniform_kernel')
                     if uniform else 'objective_kernel',
           'kernel_ms_per_launch': eval_ms, 'prepare_ms_per_launch': prep_ms,
           'kernel_share_of_step': res['eval_ms'] / float(res['step_ms'].sum()),
           'prepare_share_of_step': res['prep_ms'] / float(res['step_ms'].sum()),
           'peak_points_per_launch': pp,
           'canonical_flop_per_eval': flop_per_eval(N, P)}
    canonical = run.S * run.B * flop_per_eval(N, P) / (eval_ms * 1e-3) / 1e12
    if ncu and ncu.get('fp64_arith_inst_per_peak_point'):
        inst = ncu['fp64_arith_inst_per_peak_point'] * pp
        out['achieved'] = 2.0 * inst / (eval_ms * 1e-3) / 1e12
        out['frac'] = out['achieved'] / sustained
        flop = ncu.get('fp64_flop_per_peak_point')
        if flop:
            out['achieved_flop_counting_dmul_dadd_as_one'] = flop * pp / (eval_ms * 1e-3) / 1e12
        out['fp64_inst_per_peak_point'] = ncu['fp64_arith_inst_per_peak_point']
        out['algorithmic_speedup'] = canonical / out['achieved']
        # What actually bounds the kernel: the warp schedulers' issue ports.  An FP64 warp instruction holds its
        # sub-partition's port for two cycles (64 FP64 lanes per SM) and nothing else issues in its shadow
        # (tools/probes/issue_probe.cu, profiles/r02b_issue_probe.log: 8 DFMA + M integer ops cost 16 + ~1.25 M cycles),
        # so the port time of a launch is 2 x FP64 instructions + every other instruction.
        if ncu.get('warp_inst_per_peak_point') and sm_mhz:
            total_w = ncu['warp_inst_per_peak_point'] * pp / 32.0
            fp64_w = inst / 32.0
            ports = 148 * 4 * sm_mhz * 1e6 * (eval_ms * 1e-3)                 # issue cycles available, all sub-partitions
            out['issue_port'] = {'frac': (total_w + fp64_w) / ports, 'fp64_share_of_instructions': fp64_w / total_w,
                                 'fp64_frac_ceiling_at_this_mix': 2 * fp64_w / (total_w + fp64_w), 'sm_mhz': sm_mhz,
                                 'note': 'port cycles used / available = (all warp instructions + FP64 ones once more) / '
                                         '(592 sub-partitions x SM clock x kernel time); the ceiling is what roofline.frac '
                                         'could reach at this instruction mix with the ports 100 % busy'}
        out['traffic'] = ncu.get('dram_bytes_per_launch')
        out['ncu'] = ncu
        out['note'] = ('achieved = FP64 instructions the kernel EXECUTES (ncu: smsp__sass_thread_inst_executed_op_{dfma,dmul,'
                       'dadd}, per peak-point, from profiles/objective_ncu.json for this kernel and workload) x 2 flop / the '
                       'CUDA-event time of the kernel in this run; frac = share of the FP64 pipe\'s issue slots filled.  '
                       'algorithmic_speedup = SURVEY 8(d)\'s canonical cost (one exponential + one reciprocal per '
                       'peak-point) / executed: the recurrences and the far-field polynomial, not the hardware.')
    else:
        out['achieved'] = None
        out['frac'] = None
        out['traffic'] = None
        out['note'] = 'no ncu instruction count for this workload under profiles/objective_ncu.json: hardware fraction not stated'
    out['canonical_model_tflops'] = canonical
    algo_bytes = run.B * (4 * N * 8 + run.S * run.D * 8 + run.S * 8)
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    hbm_peak = json.load(open(peaks_path)).get('hbm_gbs') if os.path.exists(peaks_path) else 6650.0
    out['hbm'] = {'algorithmic_bytes_per_launch': algo_bytes, 'achieved_gbs': algo_bytes / (eval_ms * 1e-3) / 1e9,
                  'peak_gbs': hbm_peak, 'peak_source': 'MEASURED_PEAKS.json' if os.path.exists(peaks_path) else 'fallback'}
    return out


def measure_e2e(run, steps, warmup):
    """The metric through the public host-buffer API: positions H2D and objective values D2H inside the timed region."""
    import torch
    import torch.distributed as dist
    from nmrfit_b200 import equations, synth
    B, S, D = run.B, run.S, run.D
    if run.batched:
        # the B spectra stay resident in the context (a fit uploads them once); every step copies the
        # generation's positions [B][S][D] host -> device and the objective values [B][S] back
        xs = torch.empty((B, S, D), dtype=torch.float64).pin_memory().numpy()
        for bb in range(B):
            xs[bb] = synth.particles(run.lo[bb], run.up[bb], S, seed=7 + run.rank * B + bb)
        call = lambda: run.ctx.objective_host(xs)
        api = ('nmrfit_b200._cabi.Context.objective_host(xs[B][S][D]) with host arrays; the %d spectra are resident in '
               'the context (uploaded once per fit); the positions sit in page-locked host memory and cross PCIe once per '
               'step, read in place by the prepare kernel' % B)
        h2d, d2h = B * S * D * 8, B * S * 8
    else:
        xs = torch.empty((S, D), dtype=torch.float64).pin_memory().numpy()
        xs[:] = synth.particles(run.lo, run.up, S, seed=7 + run.rank)
        d, wts = run.data, run.weights
        call = lambda: equations.objective_batch(xs, d.w, d.u, d.v, wts)
        api = ('nmrfit_b200.equations.objective_batch(xs, w, u, v, weights) with host arrays; every call hands over '
               'the spectrum too (the reference\'s calling convention) - the library compares it with its host '
               'copy and re-sends it only when it changed, so the per-step H2D traffic is the positions.  The positions '
               'sit in page-locked host memory; the library\'s prepare kernel reads them from there itself (every element '
               'crosses PCIe once per step, inside the timed region) and the values are copied back')
        h2d, d2h = S * D * 8, S * 8
    for _ in range(max(3, warmup)):
        call()
    run.sync_all()
    e0 = time.perf_counter()
    for _ in range(steps):
        fx = call()
    torch.cuda.synchronize()
    e_ms = torch.tensor([(time.perf_counter() - e0) * 1e3], dtype=torch.float64, device='cuda')
    if run.world > 1:
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
    assert fx.size == S * B and np.all(np.isfinite(fx))
    return {'value': run.evals_per_step() * steps / (float(e_ms.item()) * 1e-3), 'unit': 'evals/s',
            'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h), 'api': api}, fx


DUMP_BYTES = 64 << 20


def swarm_outputs(run):
    """What the last timed generation left for a caller: the swarm best (``pso_best``) and the swarm state
    (``pso_state``: positions, velocities, personal bests and the objective values of the generation), float64, one row
    per particle (row = spectrum * particles + particle).  When the whole exceeds DUMP_BYTES, the per-particle arrays
    keep a fixed, seeded sample of rows, listed in ``sample_index``."""
    x, f, it, stop = run.ctx.pso_best()
    out = {'best_x': x, 'best_f': f, 'best_generations': it, 'best_stop': stop}
    rows = run.B * run.S
    per = {'swarm_' + k: a.reshape(rows, -1) if a.ndim == 3 else a.reshape(rows) for k, a in run.ctx.pso_state().items()}
    fixed = 8 * (sum(a.size for a in out.values()) + rows)            # + the end-to-end objective values
    row_bytes = 8 * sum(a.size // rows for a in per.values())
    budget = DUMP_BYTES - (64 << 10)                                    # room for the .npy headers
    if fixed + rows * row_bytes > budget:
        keep = (budget - fixed) // (row_bytes + 8)
        idx = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        per = {k: a[idx] for k, a in per.items()}
        out['sample_index'] = idx
    out.update(per)
    return {k: np.asarray(a, dtype=np.float64) for k, a in out.items()}


def secondary(name, world, rank, local, exchange, flush, steps, burst, sustained, particles=None, want_e2e=True):
    """One more BASELINE config measured like the headline (fewer steps): value, e2e, hardware fraction."""
    run = SwarmRun(name, world, rank, local, exchange, particles=particles)
    res = run.timed(steps, 3, flush)
    same = run.check_state(3 + steps)
    out = {'workload': WORKLOADS[name]['title'], 'config': workload_config(name, world, exchange),
           'value': run.evals_per_step() * steps / (res['total_ms'] * 1e-3), 'unit': 'evals/s',
           'ms_per_step': res['total_ms'] / steps, 'steps': steps, 'scaling': 'strong' if run.batched else 'weak',
           'peak_points_per_s': run.evals_per_step() * steps / (res['total_ms'] * 1e-3) * run.N * run.P}
    if particles:
        out['config']['particles_per_gpu'] = run.S
        out['config']['swarm_total'] = run.S * world
    if same is not None:
        out['sharded_identical_on_all_ranks'] = bool(same)
    rf = roofline(name, run, res, burst, sustained)
    out['roofline'] = {k: rf.get(k) for k in ('frac', 'achieved', 'peak', 'kernel_ms_per_launch', 'prepare_ms_per_launch',
                                              'kernel_share_of_step', 'algorithmic_speedup', 'fp64_inst_per_peak_point',
                                              'traffic', 'hbm')}
    if want_e2e:
        out['e2e'], _ = measure_e2e(run, max(3, steps // 2), 3)
    run.close()
    return out


def identity_flags(world, rank, local):
    """Multi-GPU correctness where the driver can see it: a small swarm (6 peaks, 4,096 points, 256 particles per rank,
    16 generations, pyswarm's stop tests live) run sharded over all ranks with either exchange, then the SAME swarm
    unsharded on every rank's own GPU.  Flags: identical on all ranks; bit-identical to the one-GPU run."""
    import torch
    import torch.distributed as dist
    from nmrfit_b200 import swarm
    data, weights, lo, up, _ = make_inputs('c1')
    kw = dict(swarmsize=256 * world, maxiter=16, seed=77, **PSO)
    out = {'swarmsize': 256 * world, 'generations': 16}
    x1, f1, info1 = swarm.pso_single(data.w, data.u, data.v, weights, lo, up, rng='device', quiet=True, device=local,
                                     fused='off', **kw)
    all_same, all_bits = True, True
    for exchange in ('nccl', 'p2p'):
        x, f, info = swarm.pso_sharded(data.w, data.u, data.v, weights, lo, up, device=local, exchange=exchange, **kw)
        blob = torch.tensor(np.concatenate([x, [f, info['generations'], info['stop']]]), device='cuda')
        parts = [torch.empty_like(blob) for _ in range(world)]
        dist.all_gather(parts, blob)
        same = all(torch.equal(p, parts[0]) for p in parts)
        bits = bool(np.array_equal(x, x1) and f == f1 and info['generations'] == info1['generations'] and
                    info['stop'] == info1['stop'])
        flag = torch.tensor([int(bits)], device='cuda')
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)         # true only if it holds on every rank
        out[exchange] = {'identical_on_all_ranks': bool(same), 'bit_identical_to_one_gpu': bool(flag.item())}
        all_same, all_bits = all_same and same, all_bits and bool(flag.item())
    out['sharded_identical_on_all_ranks'] = bool(all_same)
    out['bit_identical_to_one_gpu'] = bool(all_bits)
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from nmrfit_b200 import _cabi

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d (launch N>1 with torch.distributed.run)' % (args.gpus, world))
    wl = WORKLOADS[args.workload]

    # CPU baseline first (rank 0, N == 1): fork-based pool must not inherit a CUDA context
    cpu = None
    if world == 1 and not args.no_cpu_baseline and not args.quick:
        n_cores = os.cpu_count() or 1
        sample = reference_sample(args.workload, n_cores)
        rates, n_cores, kind = cpu_arm(args.workload, sample, 3)
        one, _, _ = cpu_arm(args.workload, max(8, sample // n_cores // 2), 2, cores=1)
        cpu = {'value': float(np.median(rates)), 'unit': 'evals/s', 'cores': n_cores, 'kind': kind,
               'sample': '%d of %d particles, %s once per particle, %d-process pool, median of 3'
                         % (sample, wl['S'], 'nmrfit.equations.objective of the unmodified reference (baseline/_ref)'
                            if kind == 'reference' else 'numpy oracle port of the reference objective', n_cores),
               'one_core_value': float(np.median(one))}
        cpu.update(cpu_fit_c1())

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    run = SwarmRun(args.workload, world, rank, local, args.exchange, args.tune)
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.05)
    res = run.timed(args.steps, args.warmup, flush)
    clocks = sampler.stop(res['t0'], res['t1'])
    same_main = run.check_state(args.warmup + args.steps)
    total_ms = res['total_ms']
    value = run.evals_per_step() * args.steps / (total_ms * 1e-3)
    outputs = swarm_outputs(run) if args.dump_outputs and rank == 0 else None

    e2e, e2e_f = measure_e2e(run, args.steps, args.warmup)
    if outputs is not None:
        outputs['e2e_objective'] = np.asarray(e2e_f, dtype=np.float64)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    burst, sustained = _cabi.fp64_peak(local, iters=4096, repeats=20)
    rf = roofline(args.workload, run, res, burst, sustained, clocks.get('sm_mhz'))
    tune = run.ctx.get_tuning(run.S)
    run.close()

    second, flags, extras = {}, None, None
    if not args.quick:
        ksteps = max(5, min(args.steps, 20))
        for name in ('c2', 'c3', 'c4', 'metric'):
            if name == args.workload:
                continue
            parts = None
            if name == 'c4' and world > 1:
                parts = 65536 // world                      # BASELINE configs[3]: 65,536 particles over the GPUs of the box
            second[name] = secondary(name, world, rank, local, args.exchange, flush, ksteps, burst, sustained, particles=parts,
                                     want_e2e=(world == 1))
        if world > 1:
            flags = identity_flags(world, rank, local)
            assert flags['sharded_identical_on_all_ranks'] and flags['bit_identical_to_one_gpu'], flags
        else:
            extras = extra_measurements(local)

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': 'evals/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': total_ms / args.steps, 'higher_is_better': True,
            'scaling': 'strong' if run.batched else 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': dict(workload_config(args.workload, world, 'p2p' if run.p2p or not run.sharded else 'nccl'), kernel=tune),
            'peak_points_per_s': value * run.N * run.P,
            'roofline': rf,
            'e2e': e2e,
            'gpu_launches': res['launches'],
            'clocks': clocks,
        }
        if run.exchange_note:
            line['config']['exchange_note'] = run.exchange_note
        if same_main is not None:
            line['sharded_identical_on_all_ranks'] = bool(same_main)
        if flags:
            line['sharded_identical_on_all_ranks'] = bool(line.get('sharded_identical_on_all_ranks', True) and
                                                          flags['sharded_identical_on_all_ranks'])
            line['bit_identical_to_one_gpu'] = flags['bit_identical_to_one_gpu']
            line['multi_gpu_identity'] = flags
        if cpu:
            line['cpu_baseline'] = cpu
        if second:
            line['secondary'] = second
        if extras:
            line.update(extras)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def extra_measurements(device):
    """One GPU only: configs[0] at its own swarm size (objective launch latency), fits/s of configs[0] through the public
    API, and the opt-in FP32 mode on the C2 shape."""
    import contextlib
    import io
    import torch
    import nmrfit_b200
    from nmrfit_b200 import _cabi, synth
    out = {}
    wl = WORKLOADS['c1']
    P, N, seed = wl['P'], wl['N'], wl['seed']
    data, weights, lo, up, true = make_inputs('c1')
    with _cabi.Context(1, N, P, device=device) as ctx:
        ctx.set_spectrum(0, data.w, data.u, data.v, weights)
        S = 100
        xs = torch.from_numpy(synth.particles(lo, up, S, seed=7)).cuda()
        f = torch.empty(S, dtype=torch.float64, device='cuda')
        for _ in range(5):
            ctx.objective_device(xs, S, f)
        ctx.profile(True)
        for _ in range(200):
            ctx.objective_device(xs, S, f)
        ms, n = ctx.profile_read()
        ctx.profile(False)
    out['configs0_objective_100_particles'] = {
        'evals_per_s': S / (ms / n * 1e-3), 'kernel_us': 1e3 * ms / n, 'peak_points_per_s': S * N * P / (ms / n * 1e-3),
        'note': 'prepare + evaluation kernels alone, inputs resident: launch-latency bound at this size'}
    # opt-in FP32 mode (north_star: <= 1e-5 relative) on the C2 shape, and its error against the FP64 kernel
    w2 = WORKLOADS['c2']
    d2, wt2, lo2, up2, _ = make_inputs('c2')
    xs = torch.from_numpy(synth.particles(lo2, up2, w2['S'], seed=7)).cuda()
    res = {}
    for name, prec in (('fp64', _cabi.FP64), ('fp32', _cabi.FP32)):
        with _cabi.Context(1, w2['N'], w2['P'], device=device, precision=prec) as ctx:
            ctx.set_spectrum(0, d2.w, d2.u, d2.v, wt2)
            f = torch.empty(w2['S'], dtype=torch.float64, device='cuda')
            for _ in range(5):
                ctx.objective_device(xs, w2['S'], f)
            ctx.profile(True)
            for _ in range(50):
                ctx.objective_device(xs, w2['S'], f)
            ms, n = ctx.profile_read()
            res[name] = (f.cpu().numpy(), ms / n)
    rel = np.abs(res['fp32'][0] / res['fp64'][0] - 1)
    out['fp32_mode'] = {'workload': 'configs[1] shape, 4,096 particles, objective kernels alone',
                        'evals_per_s': w2['S'] / (res['fp32'][1] * 1e-3), 'kernel_ms': res['fp32'][1],
                        'fp64_kernel_ms': res['fp64'][1], 'speedup_vs_fp64': res['fp64'][1] / res['fp32'][1],
                        'max_rel_err_vs_fp64': float(rel.max()), 'median_rel_err_vs_fp64': float(np.median(rel)),
                        'tolerance': 1e-5,
                        'note': 'meets the 1e-5 contract; the data side of the residual must stay FP64 (near the optimum the '
                                'residual is noise at 1e-4 of the signal), which bounds the gain - see DESIGN.md'}
    # fits/s, configs[0]: one fit at a time through nmrfit_b200.fit, then 256 fits advanced together
    opts = {'swarmsize': 100, 'maxiter': 100}
    sink = io.StringIO()
    fits = {}
    for rng, fused in (('host', 'auto'), ('device', 'auto'), ('device', 'off')):
        times = []
        for rep in range(4):
            np.random.seed(rep)
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(sink):
                fit = nmrfit_b200.fit(data, lo, up, summary=False, options=dict(opts, rng=rng, seed=rep, fused=fused))
            times.append(time.perf_counter() - t0)
        tag = 'rng_%s' % rng + ('' if fused == 'auto' else '_per_step_kernels')
        fits['single_fit_ms_' + tag] = 1e3 * float(np.median(times[1:]))
        fits['single_fit_generations_' + tag] = int(fit.fit_info['generations'])
    # the reference's defaults (swarmsize 204, maxiter 2000, stops on minfunc/minstep) on the same spectrum
    for fused in ('auto', 'off'):
        times = []
        for rep in range(3):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(sink):
                fit = nmrfit_b200.fit(data, lo, up, summary=False, options=dict(rng='device', seed=rep, fused=fused))
            times.append(time.perf_counter() - t0)
        tag = 'default_fit' + ('' if fused == 'auto' else '_per_step_kernels')
        fits[tag + '_ms'] = 1e3 * float(np.median(times[1:]))
        fits[tag + '_generations'] = int(fit.fit_info['generations'])
    B = 256
    datas, los, ups = [], [], []
    for b in range(B):
        d, _ = synth.multiplet(N, P, seed=seed + 1 + b)
        l, u = d.generate_solution_bounds()
        datas.append(d); los.append(l); ups.append(u)
    times = []
    for rep in range(3):
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(sink):
            nmrfit_b200.fit_batch(datas, los, ups, summary=False, options=dict(opts, rng='device', seed=rep))
        times.append(time.perf_counter() - t0)
    fits['batched_fits'] = B
    fits['batched_fits_per_s'] = B / float(np.median(times[1:]))
    fits['single_fits_per_s'] = 1e3 / fits['single_fit_ms_rng_device']
    fits['note'] = ('configs[0]: 6 peaks, 4,096 points, swarmsize 100, maxiter 100, wall clock through the public API '
                    'incl. weights, uploads and result readback; rng=host replays numpy\'s legacy stream (parity mode); single fits run '
                    'the fused swarm kernel (one cooperative launch per chunk of generations), *_per_step_kernels = 3 launches '
                    'per generation; default_fit = swarmsize 204, maxiter 2000, pyswarm stop rules')
    out['fits'] = fits
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='metric', choices=sorted(WORKLOADS))
    ap.add_argument('--exchange', default='p2p', choices=['nccl', 'p2p'],
                    help='particle sharding (N > 1): the best records exchanged over peer memory inside the finish kernel '
                         '(CUDA IPC windows, NVLink stores: three launches per generation, no collective call; default), '
                         'or one NCCL all-gather + a commit kernel per generation')
    ap.add_argument('--tune', default='', help='threads,points_per_thread,exp_table_bits,particles_per_cta')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--quick', action='store_true', help='main measurement only (no CPU baseline, no secondary configs / fits)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (float64, at most '
                         '64 MiB; rank 0\'s particles when sharded): swarm best, swarm state, and the objective values '
                         'of the last end-to-end call.  The inputs are seeded, so two builds can be compared file by file')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200')
    if args.warmup < 3:
        args.warmup = 3
    return run_reference(args) if args.impl == 'reference' else run_b200(args)


if __name__ == '__main__':
    sys.exit(main())
