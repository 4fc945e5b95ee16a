#!/usr/bin/env python
"""Cost of moving replicas between engines, and of one particle filter over two engines: full HUS (1,685,983 agents),
default interventions.

    python tools/migrate_bench.py [--replicas 128] [--day 60] [--moves 32] [--out FILE]

Line 1: Context.export_replicas / import_replicas of one replica (host round trip), median of repeated calls (host clock
around calls that end in a stream synchronise).
Line 2: Context.copy_replicas_from of `--moves` replicas between two engines on device 0, median of repeated calls,
with its byte model: 2 x record bytes per replica (read once, written once) against the project's measured HBM
bandwidth.  The flush of the source's active lists and the list rebuild of the written slots are inside the time.
Line 3: a 180-day run of 2 engines x R replicas under ensemble.particle_filter (weekly in_ward / in_icu of a synthetic
truth), against the filter over one engine of 2 R replicas and a plain run of that engine.
The card's name and power limit are read in the same process.  With two GPUs, the NCCL move is measured by the two-rank
test of tests/test_migrate.py, not here.
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

from branch_bench import make  # noqa: E402
from transmission_bench import HBM_GBS, card  # noqa: E402


def timed(f, calls):
    f()                                                      # warm-up: module load, argument buffers
    t = []
    for _ in range(calls):
        t0 = time.perf_counter()
        f()
        t.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(t)), float(min(t)), float(max(t))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--replicas', type=int, default=128)
    ap.add_argument('--day', type=int, default=60)
    ap.add_argument('--days', type=int, default=180)
    ap.add_argument('--moves', type=int, default=32)
    ap.add_argument('--calls', type=int, default=10)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    from reina_b200 import ensemble, inputs, model
    R, gpu = a.replicas, card()

    # ---- host round trip and device copy after `day` days
    A = make(model, inputs, R, 1, a.days + 1)
    B = make(model, inputs, R, 1 + R, a.days + 1)
    A.run(a.day)
    B.run(a.day)
    rb = A._engine.replica_bytes()
    seeds = A.replica_seeds()
    rec = A.export_replicas([0])
    exp = timed(lambda: A.export_replicas([0]), a.calls)
    imp = timed(lambda: B.import_replicas([0], rec, seeds[:1]), a.calls)
    line1 = dict(what='host export / import of one HUS replica after %d days' % a.day, card=gpu, record_bytes=rb,
                 export_ms_median=exp[0], export_ms_min=exp[1], import_ms_median=imp[0], import_ms_min=imp[1],
                 export_gbs=rb / (exp[0] / 1e3) / 1e9, import_gbs=rb / (imp[0] / 1e3) / 1e9)
    idx = np.arange(a.moves)
    cp = timed(lambda: B.copy_replicas_from(A, idx, idx, seeds[idx]), a.calls)
    model_bytes = 2.0 * rb * a.moves
    line2 = dict(what='copy_replicas_from: %d HUS replicas between two engines on one device' % a.moves, card=gpu,
                 ms_median=cp[0], ms_min=cp[1], ms_max=cp[2], us_per_replica=1e3 * cp[0] / a.moves,
                 model_bytes=model_bytes, model_gbs=model_bytes / (cp[0] / 1e3) / 1e9, hbm_gbs=HBM_GBS,
                 share_of_hbm=model_bytes / (cp[0] / 1e3) / 1e9 / HBM_GBS,
                 model_us_per_replica_at_hbm=2.0 * rb / (HBM_GBS * 1e9) * 1e6)
    A.close()
    B.close()

    # ---- 180-day filtered runs
    truth = make(model, inputs, 1, 987654321, a.days + 1)
    truth.run(a.days)
    rows = truth.series(0, a.days)
    obs_days = list(range(7, a.days, 7))
    obs = {d: {n: int(ensemble._model_counts(truth, rows[:, d], n)[0]) for n in ('in_ward', 'in_icu')} for d in obs_days}
    truth.close()

    def run(make_ctxs, filtered):
        ctxs = make_ctxs()
        for c in ctxs:                                       # warm-up: graphs
            c.run(1)
            c.reset(c._engine.cfg.seed)
        t0 = time.perf_counter()
        out = ensemble.particle_filter(ctxs if len(ctxs) > 1 else ctxs[0], obs, seed=0) if filtered else None
        for c in ctxs:
            c.run(a.days - c.day)
        ms = 1e3 * (time.perf_counter() - t0)
        for c in ctxs:
            c.close()
        return ms, out

    plain_ms, _ = run(lambda: [make(model, inputs, 2 * R, 1, a.days + 1)], False)
    one_ms, o1 = run(lambda: [make(model, inputs, 2 * R, 1, a.days + 1)], True)
    two_ms, o2 = run(lambda: [make(model, inputs, R, 1, a.days + 1), make(model, inputs, R, 1 + R, a.days + 1)], True)
    g = np.arange(2 * R)
    line3 = dict(what='%d-day HUS run, particle filter with weekly in_ward / in_icu (%d observation days): 2 engines x %d '
                      'replicas against 1 engine x %d and a plain run of it' % (a.days, len(obs_days), R, 2 * R), card=gpu,
                 plain_ms=plain_ms, filter_one_engine_ms=one_ms, filter_two_engines_ms=two_ms,
                 one_engine_over_plain=one_ms / plain_ms, two_engines_over_plain=two_ms / plain_ms,
                 two_over_one=two_ms / one_ms, resamplings=int(o2['resampled'].sum()),
                 replicas_moved_between_engines=int(((o2['ancestors'] // R) != (g // R)[None]).sum()),
                 log_evidence_two=float(o2['log_evidence']), log_evidence_one=float(o1['log_evidence']))
    lines = [json.dumps(line1), json.dumps(line2), json.dumps(line3)]
    print('\n'.join(lines), flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
