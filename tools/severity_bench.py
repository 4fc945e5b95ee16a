#!/usr/bin/env python
"""Cost of the per-replica severity scales and what filtering them buys: full HUS (1,685,983 agents), default
interventions.

    python tools/severity_bench.py [--replicas 256] [--days 180] [--out FILE] [--resolve-only]

Line 1: k_resolve device time summed over a 180-day run (rb_step_profiled: one kernel at a time, events around each),
with every severity scale 1 against heterogeneous scales (each of severe, critical, fatal log-normal, median 1, log sd
0.3, in [0.5, 2]), and the whole step's device time for both.  Run it with the parent commit's library as well
(--resolve-only, which needs no severity entry point) for the comparison with scales of 1.  The heterogeneous run moves
people through hospital differently, so its time differs by the work as well as by the products.
Line 2: 180-day runs under ensemble.particle_filter against weekly in_ward / in_icu / dead / all_detected of a
synthetic truth at transmission 1.3 and severity scales (0.7, 1.3, 0.8): with the transmission prior (1, 0.5) alone, and
with it plus severity priors (1, 0.5) on all three, volatility 0.05 each.  Wall time (host clock around work that ends
in a synchronise), resamplings, log evidence, and the final 5 / 50 / 95 % band of every filtered scale.
Every Context is made with contact_capacity 4 (as tools/scale_bench.py): the scales a prior reaches can overflow the
default lists on a peak day.  The capacity sizes buffers only; the work done is the same.
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

from scale_bench import make  # noqa: E402
from transmission_bench import card  # noqa: E402

TRUTH_F, TRUTH_SEV = 1.3, (0.7, 1.3, 0.8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--replicas', type=int, default=256)
    ap.add_argument('--days', type=int, default=180)
    ap.add_argument('--contact-capacity', type=float, default=4.0)
    ap.add_argument('--resolve-only', action='store_true', help='line 1 with scales 1 only (a library without severity scales)')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    from reina_b200 import ensemble, inputs, model
    R, gpu = a.replicas, card()

    # ---- k_resolve per run (rb_step_profiled: ms per kernel in the order pre, sweep, expose, resolve, post)
    rng = np.random.default_rng(0)
    hetero = np.clip(np.exp(rng.normal(0.0, 0.3, (R, 3))), 0.5, 2.0).astype(np.float32)
    ctx = make(model, inputs, R, 1, a.days + 1, a.contact_capacity)
    ctx.run(1)                                                # warm-up: modules, first launches
    res = {}
    cases = [('ones', None)] if a.resolve_only else [('ones', np.ones((R, 3), np.float32)), ('hetero', hetero),
                                                      ('ones_again', np.ones((R, 3), np.float32))]
    for name, s in cases:
        ctx.reset(1)
        if s is not None:
            ctx.set_severity_scale(s[:, 0], s[:, 1], s[:, 2])
        ctx._prepare_run(a.days)
        ms = ctx._engine.step_profiled(a.days)
        ctx.day += a.days
        ctx._finish_run()
        rows = ctx.series(0, a.days)
        res[name] = dict(resolve_ms=float(ms[3]), step_ms=float(ms.sum()),
                         in_ward_days=float(ensemble._model_counts(ctx, rows.reshape(-1, rows.shape[-1]), 'in_ward').sum() / R))
    ctx.close()
    lines = [json.dumps(dict(what='k_resolve ms per %d-day run (rb_step_profiled), %d HUS replicas: severity scales all 1 vs '
                                  'heterogeneous' % (a.days, R), card=gpu,
                             **{'%s_%s' % (n, k): v for n, d in res.items() for k, v in d.items()}))]

    if not a.resolve_only:
        truth = make(model, inputs, 1, 987654321, a.days + 1, a.contact_capacity)
        truth.set_transmission_scale(TRUTH_F)
        truth.set_severity_scale(*TRUTH_SEV)
        truth.run(a.days)
        rows = truth.series(0, a.days)
        obs_days = list(range(7, a.days, 7))
        names = ('in_ward', 'in_icu', 'dead', 'all_detected')
        obs = {d: {n: int(ensemble._model_counts(truth, rows[:, d], n)[0]) for n in names} for d in obs_days}
        truth.close()

        def run(**kw):
            c = make(model, inputs, R, 1, a.days + 1, a.contact_capacity)
            c.run(1)                                          # warm-up: graphs
            c.reset(1)
            t0 = time.perf_counter()
            out = ensemble.particle_filter(c, obs, seed=0, transmission_prior=(1.0, 0.5), transmission_volatility=0.05, **kw)
            c.run(a.days - c.day)
            ms = 1e3 * (time.perf_counter() - t0)
            c.close()
            bands = {'transmission': out['transmission_scale']}
            bands.update(out['severity_scale'] or {})
            q = {n: [float(x) for x in ensemble.weighted_quantiles(v[-1], out['weights'][-1], [0.05, 0.5, 0.95])]
                 for n, v in bands.items()}
            return dict(ms=ms, resamplings=int(out['resampled'].sum()), log_evidence=float(out['log_evidence']),
                        final_band_5_50_95=q)

        t_only = run()
        both = run(severity_prior={n: (1.0, 0.5) for n in model.SEVERITY_SCALES}, severity_volatility=0.05)
        lines.append(json.dumps(dict(
            what='%d-day HUS run of %d replicas, particle filter with weekly %s (%d observation days) of a truth at '
                 'transmission %.1f and severity (severe, critical, fatal) %s: transmission prior alone vs transmission '
                 'and severity priors' % (a.days, R, ' / '.join(names), len(obs_days), TRUTH_F, TRUTH_SEV),
            card=gpu, transmission_only=t_only, transmission_and_severity=both)))
    print('\n'.join(lines), flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
