#!/usr/bin/env python
"""bench.py -- agent-days/sec of the per-day agent loop (BASELINE.json), measured on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload hus|varsinais|scenario:<name>|synth50m]
                    [--replicas R | --total-seeds T] [--days D] [--impl reference] [--dump-outputs DIR]

Default workload `hus`: a "step" is one complete HUS run (1,685,983 agents x 180 days, the reference's default
interventions; BASELINE configs[1]) of an ensemble of R seeds per GPU advanced by the same launches (configs[3]), every
step with fresh seeds.  `value` times only the device-resident multi-day run (CUDA events on the engine's stream, inputs
already in HBM); `e2e` times the same step through the public API (`Context.reset` + `upload_inputs` + `run` +
`moments`) with host buffers, host->device and device->host copies included.  For N > 1 (one rank per GPU, launched by
torchrun) the ensemble is partitioned over the GPUs -- independent units, no data-path collective -- and the only
exchange is the final ncclAllReduce of the daily curves, issued by the engine itself (rb_reduce_moments); barrier and
max-over-ranks go through the same communicator.  No torch anywhere in this file.

    --replicas R       R seeds PER GPU (weak scaling, the default: 256)
    --total-seeds T    T seeds in total, T / N per GPU (configs[3] as written: strong scaling)
    --workload varsinais | scenario:hammer-and-dance | scenario:mitigation | ...   the other ensemble configurations
    --workload synth50m  configs[4]: ONE synthetic 5e7-agent population, population-sharded over the N GPUs

    --dump-outputs DIR what the timed path returned in its last timed step, as DIR/<name>.npy in float64: for the ensemble
                       workloads moments_sum and moments_sumsq ([days, row], sums over all replicas of all ranks of each
                       stats column and of its square) and n_replicas (0-d, the number of replicas summed); for synth50m
                       series ([1, days, row], rank 0's int32 stats rows).  Every step's seeds follow from the arguments,
                       so two builds run with the same arguments can be compared array for array.  Not available with
                       --impl reference: that arm keeps only the timings of its runs, not their series.

The default run also reports, beside the headline: the 256-total-seed strong-scaling point (N > 1), the synthetic
50 M-agent population on the same N GPUs, the single-seed run, per-kernel device times in the production launch
geometry and in isolation, and the reference's Cython engine on this box's host cores (N = 1).

`--impl reference` times the UNMODIFIED reference engine (oracle/_ref, built from /root/reference by
oracle/build_ref.sh) on this box's host cores: one seed per core, same workload and metric.
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
# stdout carries the ONE JSON line: whatever NCCL has to say (its version banner, NCCL_DEBUG=INFO output) goes to stderr
os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')

N_HUS = 1685983
N_SYNTH = 50_000_000


# ---------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------
def workload_spec(name):
    """-> dict(area, scenario, label, config) for the ensemble workloads."""
    if name == 'hus':
        return dict(area='HUS', scenario=None, label='HUS 1,685,983 agents, default interventions (BASELINE configs[1] / [3])')
    if name == 'varsinais':
        return dict(area='Varsinais-Suomi', scenario=None, label='Varsinais-Suomi 479,861 agents, default interventions (BASELINE configs[0])')
    if name.startswith('scenario:'):
        sc = name.split(':', 1)[1]
        return dict(area='HUS', scenario=sc, label='HUS 1,685,983 agents, scenario %s (BASELINE configs[2])' % sc)
    raise SystemExit('unknown workload %r' % name)


def metric_name(workload):
    return 'agent-days/sec (HUS 1.7M)' if workload == 'hus' else 'agent-days/sec (%s)' % workload


def make_context(spec, n_replicas, device, days, seed):
    from reina_b200 import inputs, model
    v = inputs.default_variables()
    args = inputs.build_context_args(v, area=spec['area'])
    args['random_seed'] = seed
    ctx = model.Context(n_replicas=n_replicas, device=device, max_days=days + 1, **args)
    for iv in inputs.active_interventions(v, spec['scenario']):
        ctx.add_intervention(iv)
    return ctx


def make_synth_context(n_agents, device, days, shard):
    """BASELINE configs[4]: HUS age histogram scaled to n_agents, capacity and imports scaled alike."""
    from reina_b200 import inputs, model
    f = n_agents / float(N_HUS)
    v = inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = int(round(2600 * f)), int(round(300 * f))
    ivs = []
    for iv in v['interventions']:
        iv = list(iv)
        if iv[0] in ('import-infections', 'import-infections-weekly'):
            iv[2] = int(round(iv[2] * f))
        ivs.append(iv)
    v['interventions'] = ivs
    args = inputs.build_context_args(v, age_count_override=inputs.synthetic_age_counts(n_agents))
    args['random_seed'] = 0
    ctx = model.Context(n_replicas=1, device=device, max_days=days + 1, shard=shard, **args)
    for iv in inputs.active_interventions(v):
        ctx.add_intervention(iv)
    return ctx


# ---------------------------------------------------------------------------------------------------
# measurement helpers
# ---------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def kernel_source_stamp():
    """sha1 over the CUDA sources: an ncu traffic capture is only valid for the kernels it was taken from."""
    import hashlib
    h = hashlib.sha1()
    d = os.path.join(ROOT, 'reina_b200', 'csrc')
    for name in sorted(os.listdir(d)):
        with open(os.path.join(d, name), 'rb') as f:
            h.update(name.encode() + b'\0' + f.read())
    return h.hexdigest()


def load_traffic(kernel, n_replicas, days):
    """Mean DRAM bytes (read + write) per launch of `kernel` from the committed ncu pass (profiles/r02_dram_traffic_R<R>.json,
    written by tools/ncu_traffic.py with the source stamp of the kernels it measured).  None -- never a stale number -- if
    the sources have changed since, or the capture was taken at another replica count / run length."""
    p = os.path.join(ROOT, 'profiles', 'r02_dram_traffic_R%d.json' % n_replicas)
    if not os.path.exists(p):
        return None, 'no capture for R=%d' % n_replicas
    with open(p) as f:
        t = json.load(f)
    if t.get('source_stamp') != kernel_source_stamp():
        return None, 'capture is stale (kernel sources changed since)'
    if t.get('days') != days or kernel not in t.get('kernels', {}):
        return None, 'capture does not cover this run'
    return float(t['kernels'][kernel]['mean_traffic_bytes']), t.get('command')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.device), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                 '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(smax) if smax else None,
                    samples=len(sm), reasons=sorted(reasons))


def algorithmic_bytes(s1, n_agents, n_replicas, G):
    """SURVEY.md section 8d: bytes_day = 4 N + 12 I_d + 8 E_d, summed over days and replicas.
    s1: [D, row_len] sums over replicas of the stats rows (I_d = infected that day, E_d = contacts sampled that day)."""
    from reina_b200 import _abi
    nA = len(_abi.ATTRS)
    i_inf = _abi.ATTRS.index('infected')
    I = s1[:, i_inf * G:(i_inf + 1) * G].sum(axis=1)                     # state at start of day d, all replicas
    E = s1[:, nA * G + _abi.SCALARS.index('exposed_per_day')]            # contacts of day d-1, all replicas
    D = s1.shape[0]
    sweep = 4.0 * n_agents * n_replicas * D + 12.0 * I.sum()
    expose = 8.0 * E.sum()
    return dict(sweep=sweep, expose=expose, total=sweep + expose, sum_infected=float(I.sum()), sum_contacts=float(E.sum()),
                mean_infected=float(I.mean() / n_replicas),
                mean_contacts=float(E[1:].mean() / n_replicas) if D > 1 else 0.0,
                daily_infected=(I / n_replicas).tolist(), daily_contacts=(E / n_replicas).tolist())


# ---------------------------------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------------------------------
def cpu_baseline(spec, n_agents, days, seeds, processes):
    """The reference's own Cython engine (oracle/_ref) -- or, if it is not built, the C oracle port -- timed on
    this box's host cores: agent-days/s over the summed iterate() time of a bounded sample."""
    from oracle import ref_harness
    if ref_harness.available():
        ref_harness.load_model()          # in THIS process too: the driver's loaded-library record then shows oracle/_ref
        t0 = time.perf_counter()
        _, t_iter, wall = ref_harness.run_ensemble(seeds, days=days, processes=processes, area=spec['area'], scenario=spec['scenario'])
        # rate of each core = agent-days of its run / time spent inside iterate() (setup excluded); cores add up
        value = float((n_agents * days / t_iter).sum()) if processes > 1 else n_agents * days * len(seeds) / float(t_iter.sum())
        return dict(value=value, unit='agent-days/s', cores=processes, kind='reference',
                    sample='%d seed(s) x %s %d days, unmodified cythonsim engine (oracle/_ref), %s'
                           % (len(seeds), spec['area'], days, 'sum of iterate() time' if processes == 1 else 'sum over cores of agent-days / iterate() time'),
                    seconds=time.perf_counter() - t0)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import helpers
    t0 = time.perf_counter()
    ctx = helpers.make_context(helpers.oracle_library(), area=spec['area'], scenario=spec['scenario'], seed=int(seeds[0]), max_days=days + 1)
    ctx.run(days)
    t = time.perf_counter() - t0
    return dict(value=n_agents * days / t, unit='agent-days/s', cores=1, kind='port',
                sample='1 seed x %s %d days, C oracle port (oracle/_ref not built)' % (spec['area'], days), seconds=t)


def run_reference(a, rank, world):
    if rank != 0:
        return
    name = 'hus' if a.workload == 'synth50m' else a.workload      # the reference has no sharded mode: its HUS run stands in
    spec = workload_spec(name)
    from reina_b200 import inputs
    n_agents = int(sum(inputs.build_context_args(inputs.default_variables(), area=spec['area'])['population_params']['age_structure'].values()))
    procs = min(os.cpu_count() or 1, 32)
    vals = []
    for step in range(a.warmup + a.steps):
        if step < a.warmup and step > 0:
            continue        # one warm-up pass is enough to page the extension in; each pass costs ~15 s
        seeds = np.arange(procs) + 100000 + 1000 * step
        b = cpu_baseline(spec, n_agents, a.days, seeds, procs)
        if step >= a.warmup:
            vals.append(b)
    value = float(np.mean([b['value'] for b in vals]))
    ms = 1e3 * n_agents * a.days * procs / value
    out = dict(metric=metric_name(name), value=value, unit='agent-days/s', impl='reference',
               n_gpus=a.gpus, steps=a.steps, warmup=a.warmup, ms_per_step=ms, higher_is_better=True,
               scaling='weak', vs_baseline=None, dtype='int32/f32 state, f64 uniforms', data='synthetic',
               config=dict(workload='%s x %d days, %d seeds per step (one per host core)' % (spec['label'], a.days, procs)),
               cpu_baseline=dict(value=value, unit='agent-days/s', cores=procs, kind=vals[0]['kind'], sample=vals[0]['sample']),
               e2e=dict(value=value, unit='agent-days/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU arms
# ---------------------------------------------------------------------------------------------------
def timed_ensemble(ctx, comm, days, steps, warmup, seed_of, sampler=None):
    """W untimed + K timed steps of the ensemble on `ctx`.  Returns device ms / wall s per step (max over ranks), the last
    step's replica-summed stats rows, per-step copy volumes and the launch count."""
    eng = ctx._engine

    def one_step(step):
        t0 = time.perf_counter()
        ctx.reset(seed_of(step))                   # fresh ensemble; device state re-initialised in place
        ctx.upload_inputs()                        # contact tables of every mobility epoch, from host memory
        ctx.run(days)                              # schedule H2D + the simulated days + sync
        dev_ms = eng.last_step_ms()                # CUDA events around the multi-day run only
        s1, s2, n = ctx.moments(0, days, reduce=True)      # the step's result: k_moments + ONE ncclAllReduce + D2H
        return dev_ms, time.perf_counter() - t0, dict(moments_sum=s1, moments_sumsq=s2, n_replicas=n)

    for step in range(warmup):
        one_step(step)
    if sampler:
        sampler.start()
    launches0, (h0, d0) = eng.launch_count(), eng.copied_bytes()
    comm.barrier()
    dev_ms_total, wall_total = 0.0, 0.0
    for step in range(warmup, warmup + steps):
        dev_ms, wall, outputs = one_step(step)
        dev_ms_total += dev_ms
        wall_total += wall
    comm.barrier()
    clocks = sampler.stop() if sampler else None
    launches, (h1, d1) = eng.launch_count() - launches0, eng.copied_bytes()
    dev_ms_total, wall_total = (float(x) for x in comm.allreduce(np.array([dev_ms_total, wall_total]), 'max'))
    s1, _ = eng.read_moments(0, days)              # this rank's curves of the last step: the algorithmic bytes are computed from them
    return dict(ms_per_step=dev_ms_total / steps, wall_per_step=wall_total / steps, s1=s1, h2d=(h1 - h0) / steps, d2h=(d1 - d0) / steps,
                launches=launches, clocks=clocks, outputs=outputs)


def dump_outputs(directory, outputs):
    """Write the last timed step's results as DIR/<name>.npy in float64, so that two builds can be compared value for value
    (the seeds of every step are fixed by the arguments)."""
    os.makedirs(directory, exist_ok=True)
    for name, x in outputs.items():
        np.save(os.path.join(directory, name + '.npy'), np.asarray(x, dtype=np.float64))


def bench_synth(a, rank, world, local, n_agents, days, steps, warmup):
    """configs[4]: one synthetic population sharded over the ranks.  -> (dict for the JSON line, the last step's results)."""
    from reina_b200 import comm as rcomm, sharded
    spec = sharded.shard_spec() if world > 1 else None
    ctx = make_synth_context(n_agents, local, days, spec)
    comm = rcomm.EngineComm(ctx._engine) if world > 1 else rcomm.LocalComm()
    ms, walls = [], []
    for step in range(warmup + steps):
        comm.barrier()
        t0 = time.perf_counter()
        ctx.reset(1000 + step)                     # the same seed on every rank
        ctx.run(days)
        rows = ctx.series(0, days)                 # the run's result on every rank
        wall = time.perf_counter() - t0
        t = comm.allreduce(np.array([ctx._engine.last_step_ms(), wall]), 'max')
        if step >= warmup:
            ms.append(float(t[0])); walls.append(float(t[1]))
    G = len(ctx.age_group_labels)
    chk = float(rows[0, -1, 3 * G:4 * G].sum())
    lo, hi = float(-comm.allreduce(np.array([-chk]), 'max')[0]), float(comm.allreduce(np.array([chk]), 'max')[0])
    eng = ctx._engine
    out = dict(value=n_agents * days / (np.mean(ms) / 1e3), unit='agent-days/s', agents=n_agents, days=days, n_gpus=world,
               ms_per_run=float(np.mean(ms)), e2e_value=n_agents * days / float(np.mean(walls)), scaling='strong',
               all_infected_last_day=chk, ranks_agree=bool(lo == hi),
               exchange={0: 'none', 1: 'ncclAllGather', 2: 'NVLink peer memory'}[int(eng.lib.f['shard_exchange'](eng.h))],
               message_bytes_per_rank_per_day=int(eng.lib.f['shard_message_bytes'](eng.h)))
    ctx.close()
    return out, dict(series=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='hus')
    ap.add_argument('--replicas', type=int, default=256, help='ensemble members (seeds) per GPU (weak scaling)')
    ap.add_argument('--total-seeds', type=int, default=0, help='seeds in total, split evenly over the GPUs (configs[3] as written: strong scaling)')
    ap.add_argument('--days', type=int, default=180)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='headline only: no strong-scaling point, synthetic population, single seed')
    ap.add_argument('--dump-daily', default=None, help='write the per-day I_d, E_d (ensemble means) the algorithmic bytes are computed from')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write what the timed path returned in its last step as DIR/<name>.npy (float64): the ensemble moments '
                         '(moments_sum, moments_sumsq, n_replicas), or the daily rows (series) of --workload synth50m')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs is not available with --impl reference')

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))

    if a.impl == 'reference':
        run_reference(a, rank, world)
        return

    from reina_b200 import comm as rcomm
    D = a.days
    peak_gbs, peak_src = load_peaks()

    if a.workload == 'synth50m':
        r, outputs = bench_synth(a, rank, world, local, N_SYNTH, D, a.steps, a.warmup)
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, outputs)
        if rank == 0:
            bytes_run = None
            out = dict(metric='agent-days/sec (synthetic 50M, population-sharded)', value=r['value'], unit='agent-days/s', n_gpus=world,
                       steps=a.steps, warmup=a.warmup, ms_per_step=r['ms_per_run'], higher_is_better=True, scaling='strong',
                       vs_baseline=None, dtype='int32/f32 state, f64 uniforms', data='synthetic',
                       config=dict(workload='synthetic 50,000,000 agents x %d days (HUS age histogram x 29.66, capacity and imports scaled; '
                                            'BASELINE configs[4]), ONE population sharded over %d GPU(s)' % (D, world),
                                   l2='2.6 GB of agent state >> L2'),
                       e2e=dict(value=r['e2e_value'], unit='agent-days/s'), synth50m=r)
            print(json.dumps(out), flush=True)
        return

    spec = workload_spec(a.workload)
    strong = a.total_seeds > 0
    if strong and a.total_seeds % world:
        raise SystemExit('--total-seeds must be a multiple of the number of GPUs')
    R = a.total_seeds // world if strong else a.replicas
    ctx = make_context(spec, R, local, D, seed=1)
    eng = ctx._engine
    comm = rcomm.connect(eng, rank, world)        # NCCL through the engine's own C-ABI; LocalComm for one process
    N = ctx.n_agents
    G = len(ctx.age_group_labels)
    seed_of = lambda step: 1_000_000 * (rank + 1) + 1000 * step     # fresh seeds every step, distinct per rank

    res = timed_ensemble(ctx, comm, D, a.steps, a.warmup, seed_of, ClockSampler(local) if rank == 0 else None)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, res['outputs'])
    agent_days_step = float(N) * D * R * world
    ms_per_step = res['ms_per_step']
    value = agent_days_step / (ms_per_step / 1e3)
    e2e_value = agent_days_step / res['wall_per_step']
    alg = algorithmic_bytes(res['s1'], N, R, G)

    if a.dump_daily and rank == 0:
        with open(a.dump_daily, 'w') as f:
            json.dump(dict(note='%s, ensemble means over %d seeds of the last timed step: I_d = infected at the start of day d, '
                                'E_d = contacts sampled on day d-1 (stats row d); bytes_d = 4 N + 12 I_d + 8 E_d (SURVEY.md 8d)' % (spec['area'], R),
                           agents=N, days=D, I_d=alg['daily_infected'], E_d=alg['daily_contacts']), f)

    # ---------------- per-kernel device times: production geometry and isolated (two extra runs) ----------------
    knames = ['k_pre', 'k_sweep', 'k_expose', 'k_resolve', 'k_post']

    def prepare():
        ctx.reset(seed_of(a.warmup + a.steps - 1))
        while len(ctx._plan) < D:
            ctx._plan_next_day()
        eng.set_schedule(0, ctx._plan[:D])

    prepare()
    t_ms, t_cnt, t_wall = eng.step_timed(D)           # rb_step's groups / streams / grids, events around every launch
    prepare()
    iso = eng.step_profiled(D)                        # one kernel at a time, full-wave grids
    share = t_ms / max(float(t_ms.sum()), 1e-9)
    dom = int(np.argmax(t_ms))
    kname = knames[dom]
    # SURVEY 8(d) per-unit figures x the units one launch processes: sweep 4 B/agent + 12 B/infected agent, expose 8 B/contact
    nominal = {'k_sweep': alg['sweep'], 'k_expose': alg['expose']}.get(kname, 0.0)
    # what this design's kernels have to move at least: sweep = 16 B per active-list entry (8 read + 8 written); expose = 2 B of
    # work item + 4 B of susceptibility word per contact
    design = {'k_sweep': 16.0 * alg['sum_infected'], 'k_expose': 6.0 * alg['sum_contacts']}.get(kname, 0.0)
    n_launch = max(int(t_cnt[dom]), 1)
    avg_ms = float(t_ms[dom]) / n_launch
    achieved = nominal / n_launch / (avg_ms / 1e3) / 1e9 if avg_ms > 0 else 0.0
    iso_ms = float(iso[dom]) / D
    traffic, traffic_src = load_traffic(kname, R, D)
    whole = alg['total'] / (ms_per_step / 1e3) / 1e9

    out = dict(
        metric=metric_name(a.workload), value=value, unit='agent-days/s', n_gpus=world, steps=a.steps,
        warmup=a.warmup, ms_per_step=ms_per_step, higher_is_better=True, scaling='strong' if strong else 'weak', vs_baseline=None,
        dtype='int32/f32 state, f64 uniforms', data='synthetic',
        config=dict(
            workload='%s x %d days, ensemble of %d seeds per GPU advanced by the same launches%s'
                     % (spec['label'], D, R, ' (%d seeds in total, configs[3] as written)' % a.total_seeds if strong else ' (configs[3] share per GPU)'),
            replicas_per_gpu=R, total_seeds=R * world, days=D, agents=N, parallelism='ensemble x%d' % world,
            l2='inputs larger than L2 (%.1f GB of agent state per GPU)' % (R * N * 52.3 / 1e9) if R > 2 else
               'single 6.7 MB packed-state array is L2-resident by nature of the workload (180 dependent days)',
        ),
        e2e=dict(value=e2e_value, unit='agent-days/s', h2d_bytes_per_step=int(res['h2d']), d2h_bytes_per_step=int(res['d2h']),
                 ms_per_step=1e3 * res['wall_per_step'], ms_over_device=1e3 * res['wall_per_step'] - ms_per_step),
        gpu_launches=int(res['launches']),
        clocks=res['clocks'],
        roofline=dict(bound='hbm', kernel=kname, achieved=achieved, peak=peak_gbs, unit='GB/s', frac=achieved / peak_gbs,
                      traffic=traffic, traffic_source=traffic_src, peak_source=peak_src,
                      algorithmic_bytes_per_launch=nominal / n_launch, avg_launch_ms=avg_ms, launches=n_launch,
                      geometry='production: %d replica group(s) on concurrent streams, events around every launch on its own stream; '
                               'launches of different groups overlap, so a launch shares the GPU' % max(1, n_launch // D),
                      share_of_step=float(share[dom]),
                      frac_dram=(traffic / (avg_ms / 1e3) / 1e9 / peak_gbs) if traffic else None,
                      design_bytes_per_launch=design / n_launch, frac_design=design / n_launch / (avg_ms / 1e3) / 1e9 / peak_gbs if avg_ms > 0 else None,
                      isolated=dict(avg_launch_ms=iso_ms, note='the same kernel over all %d replicas in ONE full-wave launch with the GPU to itself' % R,
                                    frac=(nominal / D / (iso_ms / 1e3) / 1e9 / peak_gbs) if iso_ms > 0 else None,
                                    # measured DRAM bytes of a day (the production launches of all groups together) over the isolated launch time
                                    frac_dram=(traffic * n_launch / D / (iso_ms / 1e3) / 1e9 / peak_gbs) if traffic and iso_ms > 0 else None),
                      note='algorithmic bytes follow SURVEY.md 8(d), defined against the minimal hot state independently of the layout '
                           '(sweep 4 B/agent + 12 B/infected, contacts 8 B/contact); the list-based sweep never touches the 4 B/agent of the '
                           'idle population, hence frac_design (this design\'s own minimum) and frac_dram (measured DRAM bytes) beside it'),
        roofline_whole_run=dict(achieved=whole, peak=peak_gbs, unit='GB/s', frac=whole / peak_gbs,
                                bytes_per_agent_day=alg['total'] / (float(N) * D * R),
                                mean_infected=alg['mean_infected'], mean_contacts_per_day=alg['mean_contacts']),
        kernel_ms_per_day=dict(production={k: float(v) / D for k, v in zip(knames, t_ms)}, production_wall_ms_per_day=t_wall / D,
                               isolated={k: float(v) / D for k, v in zip(knames, iso)}),
    )
    ctx.close()

    extras = not a.no_extras and a.workload == 'hus' and not strong
    # ---------------- configs[3] as written: 256 seeds in total, 256 / N per GPU (strong scaling) ----------------
    if extras and world > 1 and 256 % world == 0:
        c2 = make_context(spec, 256 // world, local, D, seed=1)
        comm2 = rcomm.connect(c2._engine, rank, world, key='strong')
        r2 = timed_ensemble(c2, comm2, D, max(2, a.steps // 2), 2, seed_of)
        out['strong_scaling_256_seeds'] = dict(
            value=float(N) * D * 256 / (r2['ms_per_step'] / 1e3), unit='agent-days/s', total_seeds=256, replicas_per_gpu=256 // world,
            ms_per_step=r2['ms_per_step'], e2e_value=float(N) * D * 256 / r2['wall_per_step'], scaling='strong')
        c2.close()
    # ---------------- configs[4]: the synthetic 50 M population on the same GPUs ----------------
    if extras:
        out['synth50m'], _ = bench_synth(a, rank, world, local, N_SYNTH, D, 2, 1)
    # ---------------- single-seed run of the same configuration (latency-bound, reported beside) ----------------
    if extras and rank == 0 and R != 1:
        c1 = make_context(spec, 1, local, D, seed=1)
        for s in range(2):
            c1.reset(50 + s); c1.run(D)
        ms = []
        for s in range(3):
            c1.reset(60 + s); c1.run(D); ms.append(c1._engine.last_step_ms())
        out['single_seed'] = dict(value=N * D / (np.mean(ms) / 1e3), unit='agent-days/s',
                                  ms_per_run=float(np.mean(ms)), us_per_day=1e3 * float(np.mean(ms)) / D)
        c1.close()

    if rank == 0 and not a.no_cpu_baseline and world == 1:
        b = cpu_baseline(spec, N, D, np.array([0]), 1)
        out['cpu_baseline'] = {k: b[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
    elif rank == 0:
        out['cpu_baseline'] = None

    if rank == 0:
        print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
