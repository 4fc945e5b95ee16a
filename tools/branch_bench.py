#!/usr/bin/env python
"""Cost of Context.branch() and of a particle filter at the bench geometry: full HUS (1,685,983 agents), 256 replicas,
default interventions.

    python tools/branch_bench.py [--replicas 256] [--day 60] [--calls 20] [--out FILE]

Line 1: Context.branch() after `--day` days with half of the slots copied (odd slot j from even slot j - 1), as the
median of repeated calls (host clock around the call, which ends in a stream synchronise), with its byte model.
Line 2: a 180-day run under ensemble.particle_filter with weekly in_ward / in_icu observations of a synthetic truth (one
replica of the same inputs with a seed outside the ensemble's), against a plain 180-day run of the same ensemble; and
the branch time as a share of the filter's run.  The card's name and power limit are read in the same process.

Byte model per copied replica (what the copy has to move at least, read once and written once): the sections of one
replica in the rb_save_state blob -- 4 N (packed words) + 32 N (agent records) + N / 4 (the two bitmaps) + the counters
+ both test queues + the stats rows + the seed history -- taken from the blob size.  The flush of every replica's active
lists before the copy and the list rebuild of the copies after it are inside the measured time and outside the model.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from transmission_bench import HBM_GBS, card  # noqa: E402


def make(model, inputs, replicas, seed, max_days):
    v = inputs.default_variables()
    args = inputs.build_context_args(v, area='HUS')
    args['random_seed'] = seed
    ctx = model.Context(n_replicas=replicas, max_days=max_days, **args)
    for iv in inputs.active_interventions(v, None):
        ctx.add_intervention(iv)
    return ctx


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--replicas', type=int, default=256)
    ap.add_argument('--day', type=int, default=60)
    ap.add_argument('--days', type=int, default=180)
    ap.add_argument('--calls', type=int, default=20)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    from reina_b200 import ensemble, inputs, model
    R = a.replicas
    gpu = card()

    # ---- Context.branch
    ctx = make(model, inputs, R, 1, a.days + 1)
    ctx.run(a.day)
    src = np.arange(R)
    src[1::2] = np.arange(0, R - 1, 2)
    n_copy = int((src != np.arange(R)).sum())
    seeds = ctx.replica_seeds()
    ctx.branch(src, seeds)                                   # warm-up: module load, argument buffer
    times = []
    for _ in range(a.calls):
        t0 = time.perf_counter()
        ctx.branch(src, seeds)
        times.append(1e3 * (time.perf_counter() - t0))
    per_replica = ctx._engine.lib.f['state_bytes'](ctx._engine.h) / R
    model_bytes = 2.0 * per_replica * n_copy
    ms = float(np.median(times))
    line1 = dict(what='Context.branch() after a %d-day HUS run, %d replicas, %d copied' % (a.day, R, n_copy), card=gpu,
                 calls=a.calls, ms_per_call_median=ms, ms_per_call_min=float(min(times)), ms_per_call_max=float(max(times)),
                 bytes_per_replica=per_replica, model_bytes=model_bytes, model_gbs=model_bytes / (ms / 1e3) / 1e9,
                 hbm_gbs=HBM_GBS, share_of_hbm=model_bytes / (ms / 1e3) / 1e9 / HBM_GBS,
                 model_ms_at_hbm=model_bytes / (HBM_GBS * 1e9) * 1e3, agents=ctx.n_agents)
    ctx.close()

    # ---- a particle filter against a plain run
    truth = make(model, inputs, 1, 987654321, a.days + 1)
    truth.run(a.days)
    rows = truth.series(0, a.days)
    obs_days = list(range(7, a.days, 7))
    obs = {d: {n: int(ensemble._model_counts(truth, rows[:, d], n)[0]) for n in ('in_ward', 'in_icu')} for d in obs_days}
    truth.close()
    plain = make(model, inputs, R, 1, a.days + 1)
    plain.run(1)                                             # warm-up: graphs
    plain.reset(1)
    t0 = time.perf_counter()
    plain.run(a.days)
    plain_ms = 1e3 * (time.perf_counter() - t0)
    plain.close()
    filt = make(model, inputs, R, 1, a.days + 1)
    filt.run(1)
    filt.reset(1)
    t0 = time.perf_counter()
    out = ensemble.particle_filter(filt, obs, seed=0)
    filt.run(a.days - filt.day)
    filter_ms = 1e3 * (time.perf_counter() - t0)
    filt.close()
    line2 = dict(what='%d-day HUS run, %d replicas: particle filter with weekly in_ward / in_icu (%d observation days) '
                      'against a plain run' % (a.days, R, len(obs_days)), card=gpu, plain_ms=plain_ms, filter_ms=filter_ms,
                 filter_over_plain=filter_ms / plain_ms, resamplings=int(out['resampled'].sum()),
                 branch_ms_share_of_filter=int(out['resampled'].sum()) * ms / filter_ms,
                 log_evidence=float(out['log_evidence']), mean_ess=float(out['ess'].mean()))
    lines = [json.dumps(line1), json.dumps(line2)]
    print('\n'.join(lines), flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
