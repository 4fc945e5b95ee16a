#!/usr/bin/env python
"""Cost of Context.transmission_stats() at the bench geometry: full HUS (1,685,983 agents), 256 replicas, after a 180-day
run with the default interventions.

    python tools/transmission_bench.py [--replicas 256] [--days 180] [--calls 30] [--settings] [--out FILE]

Prints one JSON line: ms per call (host clock around the call, which ends in a stream synchronise), the byte model of
k_transmission over that time as a share of the measured HBM bandwidth, and the ratio to the time of the 180-day run
itself (last_step_ms).  The card's name and power limit are read in the same process.  --settings: a second line, the
same for Context.transmission_settings() (k_transmission_settings) on the same state.

Byte model per replica (what the pass has to move at least): the susceptibility bitmap (N / 8 bytes), and per infected
agent its 4-byte packed word and its 32-byte agent record, plus one gathered 32-byte record of the infector for every
agent that has one.  The call also runs k_flush_lists (reads the active lists) and copies the tables to the host; both
are inside the measured time and outside the byte model.

Byte model of k_transmission_settings per replica: the bitmap (N / 8), 36 bytes per infected agent as above, and per
child the 32-byte sector of its infector's packed word (the infector's state: closed or not).  The contact tables it
searches (a few hundred kB per epoch) stay in L2 and are left out.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6456.2     # HBM bandwidth measured on a B200 (the peak of bench.py's roofline, profiles/r02_bench_R256_n1.json)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def byte_model(stats, n_agents):
    infected = stats['cohort_infected'].sum(axis=1)          # per replica
    children = stats['cohort_offspring'].sum(axis=1)         # = agents with an infector
    per_rep = n_agents / 8.0 + (4.0 + 32.0) * infected + 32.0 * children
    return float(per_rep.sum()), float(infected.mean()), float(children.mean())


def settings_byte_model(settings, n_agents):
    bdp = settings['by_day_place']
    infected = bdp.sum(axis=(1, 2))
    children = bdp[:, :, :-1].sum(axis=(1, 2))                # every place column but the roots'
    per_rep = n_agents / 8.0 + (4.0 + 32.0) * infected + 32.0 * children
    return float(per_rep.sum()), float(infected.mean()), float(children.mean())


def timed(fn, calls):
    first = fn()                                              # warm-up: module load, table allocation
    times = []
    for _ in range(calls):
        t0 = time.perf_counter()
        x = fn()
        times.append(1e3 * (time.perf_counter() - t0))
    assert all(np.array_equal(x[k], first[k]) for k in first), 'repeated calls differ'
    return first, times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--replicas', type=int, default=256)
    ap.add_argument('--days', type=int, default=180)
    ap.add_argument('--calls', type=int, default=30)
    ap.add_argument('--settings', action='store_true', help='also time Context.transmission_settings()')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    from reina_b200 import inputs, model
    v = inputs.default_variables()
    args = inputs.build_context_args(v, area='HUS')
    args['random_seed'] = 1
    ctx = model.Context(n_replicas=a.replicas, max_days=a.days + 1, **args)
    for iv in inputs.active_interventions(v, None):
        ctx.add_intervention(iv)
    ctx.run(a.days)
    step_ms = ctx._engine.last_step_ms()
    def line(call, times, model):
        ms = float(np.median(times))
        total, mean_inf, mean_child = model
        return json.dumps(dict(
            what='Context.%s() after a %d-day HUS run, %d replicas' % (call, a.days, a.replicas), card=card(),
            calls=a.calls, ms_per_call_median=ms, ms_per_call_min=float(min(times)), ms_per_call_max=float(max(times)),
            run_ms=step_ms, share_of_run=ms / step_ms if step_ms > 0 else None, model_bytes=total,
            model_gbs=total / (ms / 1e3) / 1e9, hbm_gbs=HBM_GBS, share_of_hbm=total / (ms / 1e3) / 1e9 / HBM_GBS,
            mean_infected_per_replica=mean_inf, mean_children_per_replica=mean_child, agents=ctx.n_agents))

    stats, times = timed(ctx.transmission_stats, a.calls)
    lines = [line('transmission_stats', times, byte_model(stats, ctx.n_agents))]
    if a.settings:
        settings, times = timed(ctx.transmission_settings, a.calls)
        lines.append(line('transmission_settings', times, settings_byte_model(settings, ctx.n_agents)))
    print('\n'.join(lines), flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
