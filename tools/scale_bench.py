#!/usr/bin/env python
"""Cost of the per-replica transmission scale and of filtering it: full HUS (1,685,983 agents), default interventions.

    python tools/scale_bench.py [--replicas 256] [--days 180] [--out FILE]

Line 1: k_expose device time summed over a 180-day run (rb_step_profiled: one kernel at a time, events around each), with
every scale 1 against heterogeneous scales (log-normal, median 1, log sd 0.3, in [0.5, 2]), and the whole step's device
time for both.  The heterogeneous run infects more or fewer people, so its time differs by the work as well as by the
multiply; the scale-1 figure is the one to hold against the parent commit.
Line 2: a 180-day run under ensemble.particle_filter (weekly in_ward / in_icu of a synthetic truth with scale 1.3), with
and without transmission_prior=(1, 0.5) and volatility 0.05, against a plain run: wall time (host clock around work that
ends in a synchronise) and the number of resamplings, and the final 90 % band of the filtered scale.
Every Context is made with contact_capacity 4 (--contact-capacity): at the scales a prior reaches, a replica's peak day
holds more contacts and transmissions than the default lists, and a run that overflows them stops with SimulationFailed.
The capacity sizes buffers only; the work done is the same.
The card's name and power limit are read in the same process.
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

from transmission_bench import card  # noqa: E402


def make(model, inputs, replicas, seed, max_days, contact_capacity):
    v = inputs.default_variables()
    args = inputs.build_context_args(v, area='HUS')
    args['random_seed'] = seed
    ctx = model.Context(n_replicas=replicas, max_days=max_days, contact_capacity=contact_capacity, **args)
    for iv in inputs.active_interventions(v, None):
        ctx.add_intervention(iv)
    return ctx


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--replicas', type=int, default=256)
    ap.add_argument('--days', type=int, default=180)
    ap.add_argument('--contact-capacity', type=float, default=4.0,
                    help='Context contact_capacity: replicas at scales of 4 and more hold several times the default day\'s contacts')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    from reina_b200 import ensemble, inputs, model
    R, gpu = a.replicas, card()

    # ---- k_expose per run, scales 1 and heterogeneous
    rng = np.random.default_rng(0)
    hetero = np.clip(np.exp(rng.normal(0.0, 0.3, R)), 0.5, 2.0).astype(np.float32)
    ctx = make(model, inputs, R, 1, a.days + 1, a.contact_capacity)
    ctx.run(1)                                                # warm-up: modules, first launches
    res = {}
    for name, f in (('ones', np.ones(R, np.float32)), ('hetero', hetero), ('ones_again', np.ones(R, np.float32))):
        ctx.reset(1)
        ctx.set_transmission_scale(f)
        ctx._prepare_run(a.days)
        ms = ctx._engine.step_profiled(a.days)
        ctx.day += a.days
        ctx._finish_run()
        res[name] = dict(expose_ms=float(ms[2]), step_ms=float(ms.sum()),
                         infected=float(ctx.series(0, a.days)[:, -1, 3 * len(ctx.age_group_labels):4 * len(ctx.age_group_labels)].sum() / R))
    ctx.close()
    line1 = dict(what='k_expose ms per %d-day run (rb_step_profiled), %d HUS replicas: scales all 1 vs heterogeneous' % (a.days, R),
                 card=gpu, **{'%s_%s' % (n, k): v for n, d in res.items() for k, v in d.items()})

    # ---- 180-day filtered runs
    truth = make(model, inputs, 1, 987654321, a.days + 1, a.contact_capacity)
    truth.set_transmission_scale(1.3)
    truth.run(a.days)
    rows = truth.series(0, a.days)
    obs_days = list(range(7, a.days, 7))
    obs = {d: {n: int(ensemble._model_counts(truth, rows[:, d], n)[0]) for n in ('in_ward', 'in_icu')} for d in obs_days}
    truth.close()

    def run(filtered, **kw):
        c = make(model, inputs, R, 1, a.days + 1, a.contact_capacity)
        c.run(1)                                              # warm-up: graphs
        c.reset(1)
        t0 = time.perf_counter()
        out = ensemble.particle_filter(c, obs, seed=0, **kw) if filtered else None
        c.run(a.days - c.day)
        ms = 1e3 * (time.perf_counter() - t0)
        c.close()
        return ms, out

    plain_ms, _ = run(False)
    base_ms, o0 = run(True)
    prior_ms, o1 = run(True, transmission_prior=(1.0, 0.5), transmission_volatility=0.05)
    lo, med, hi = ensemble.weighted_quantiles(o1['transmission_scale'][-1], o1['weights'][-1], [0.05, 0.5, 0.95])
    line2 = dict(what='%d-day HUS run of %d replicas, particle filter with weekly in_ward / in_icu (%d observation days) of a '
                      'truth at scale 1.3: without and with transmission_prior=(1, 0.5), volatility 0.05, against a plain run'
                      % (a.days, R, len(obs_days)), card=gpu,
                 plain_ms=plain_ms, filter_ms=base_ms, filter_prior_ms=prior_ms, resamplings=int(o0['resampled'].sum()),
                 resamplings_prior=int(o1['resampled'].sum()), log_evidence=float(o0['log_evidence']),
                 log_evidence_prior=float(o1['log_evidence']), final_scale_band_5_50_95=[float(lo), float(med), float(hi)])
    lines = [json.dumps(line1), json.dumps(line2)]
    print('\n'.join(lines), flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
