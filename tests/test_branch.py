"""Branching replicas from the current state (rb_branch / rb_read_seeds, Context.branch / replica_seeds) and conditioning
an ensemble on observed counts (ensemble.systematic_resample / assign_slots / log_likelihood / particle_filter).

CPU: the reference branch copies state, a copy with its source's seed continues as the source, the identity branch is a
no-op, the resampling helpers hold their properties, the likelihoods match scipy, the filter is deterministic, refuses a
collapse and conditions.  GPU: the CUDA engine equals the reference through branches on the every-intervention schedule
and at the bench geometry (256 HUS replicas, four replica groups), the identity branch changes nothing, branched states
survive save / load (and version-2 blobs still load), bad sources are refused, and the filter gives the same answer on
both engines.

The CPU reference is tests/oracle_branch.c over the instrumented oracle of test_transmission_settings.py (the probes
record the place of every infection where the oracle makes it), compiled into a library of its own in the temporary
directory, keyed by the hash of the sources."""
import hashlib
import multiprocessing
import os
import shutil
import subprocess
import tempfile
import traceback
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

import helpers
from reina_b200 import _abi, ensemble
from test_transmission import stress_kw
from test_transmission_settings import ORACLE_PROBES, SETTINGS

_br_oracle = None


def br_oracle_library():
    """The probed oracle plus the transmission, settings and branch entry points, built once per source state."""
    global _br_oracle
    if _br_oracle is None:
        files = [('oracle', 'reina_oracle.c'), ('tests', 'oracle_transmission.c'), ('tests', 'oracle_settings.c'),
                 ('tests', 'oracle_branch.c'), ('include', 'reina_b200.h')]
        src = {f: open(os.path.join(helpers.ROOT, *f), 'rb').read().decode() for f in files}
        key = hashlib.sha1(''.join(src[f] for f in files).encode() + repr(ORACLE_PROBES).encode()).hexdigest()[:16]
        lib = os.path.join(tempfile.gettempdir(), 'reina_br_oracle_%d_%s.so' % (os.getuid(), key))
        if not os.path.exists(lib):
            text = src[('oracle', 'reina_oracle.c')]
            for anchor, line in ORACLE_PROBES:
                assert text.count(anchor) == 1, 'oracle probe anchor not found exactly once: %r' % anchor
                text = text.replace(anchor, anchor + line)
            src[('oracle', 'reina_oracle.c')] = text
            tree = tempfile.mkdtemp(prefix='reina_br_oracle_')
            try:
                for f in files:
                    os.makedirs(os.path.join(tree, f[0]), exist_ok=True)
                    with open(os.path.join(tree, *f), 'w') as fh:
                        fh.write(src[f])
                tmp = '%s.%d.tmp' % (lib, os.getpid())
                subprocess.run([os.environ.get('CC', 'gcc'), '-O2', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math',
                                '-shared', '-o', tmp, os.path.join(tree, 'tests', 'oracle_branch.c'), '-lm'], check=True)
                os.replace(tmp, lib)
            finally:
                shutil.rmtree(tree, ignore_errors=True)
        _br_oracle = _abi.Library(lib, 'ro_')
        _br_oracle.bind_transmission()
        _br_oracle.bind_settings()
        _br_oracle.bind_branch()
    return _br_oracle


@pytest.fixture(scope='module')
def br_oracle():
    return br_oracle_library()


def replica_state(ctx, r):
    """Everything of replica r a test compares: rows so far, agents, queue, free beds / ICU, seed history up to today."""
    return dict(rows=ctx.series(0, ctx.day)[r], agents=ctx._engine.read_agents(r), queue=np.sort(ctx._engine.read_queue(r)),
                avail=ctx._engine.read_available(r), seeds=ctx._engine.read_seeds()[r, :ctx.day + 1])


def assert_same_state(a, b, what):
    for k in a:
        assert np.array_equal(a[k], b[k]), (what, k)


def assert_same_ensemble(gpu, cpu, what):
    rep = helpers.diff_report(gpu, cpu, gpu.day)
    assert not rep, '%s:\n%s' % (what, '\n'.join(rep))
    assert np.array_equal(gpu._engine.read_seeds(), cpu._engine.read_seeds()), what
    t, tc = gpu.transmission_stats(), cpu.transmission_stats()
    assert all(np.array_equal(t[k], tc[k]) for k in t), what
    s, sc = gpu.transmission_settings(), cpu.transmission_settings()
    assert all(np.array_equal(s[k], sc[k]) for k in SETTINGS), what
    for r in range(gpu.n_replicas):
        assert np.array_equal(gpu.infection_places(r), cpu.infection_places(r)), (what, r)


# ---------------------------------------------------------------- CPU (oracle)
def test_oracle_branch_copies_state(br_oracle):
    """After a branch, replica j up to today is replica src[j]: rows, agents, queue, capacity, seed history, places."""
    ctx = helpers.make_context(br_oracle, seed=40, n_replicas=4, max_days=80, **stress_kw(30000))
    ctx.run(45)
    before = {r: replica_state(ctx, r) for r in range(4)}
    places = {r: ctx.infection_places(r) for r in range(4)}
    seeds = ctx.branch([0, 0, 2, 0], [40, 900, 901, 902])
    assert seeds.tolist() == [40, 900, 901, 902] and ctx.replica_seeds().tolist() == [40, 900, 901, 902]
    for j, s in enumerate([0, 0, 2, 0]):
        after = replica_state(ctx, j)
        assert np.array_equal(after['seeds'][:45], before[s]['seeds'][:45]) and after['seeds'][45] == seeds[j]
        after['seeds'], b = after['seeds'][:45], dict(before[s], seeds=before[s]['seeds'][:45])
        assert_same_state(after, b, j)
        assert np.array_equal(ctx.infection_places(j), places[s]), j
    assert before[0]['queue'].size > 0                       # contact tracing is on: the queue is part of the copy
    ctx.run(30)                                              # the copies drew different futures
    rows = ctx.series(0, 75)
    assert not np.array_equal(rows[1, 46:], rows[0, 46:]) and not np.array_equal(rows[3, 46:], rows[1, 46:])


def test_oracle_copy_with_the_source_seed_continues_as_the_source(br_oracle):
    ctx = helpers.make_context(br_oracle, seed=60, n_replicas=3, max_days=80, **stress_kw(30000))
    ctx.run(38)
    ctx.branch([0, 0, 0], [60, 60, 61])
    ctx.run(30)
    assert_same_state(replica_state(ctx, 1), replica_state(ctx, 0), 'same seed')
    assert not np.array_equal(ctx.series(0, 68)[2], ctx.series(0, 68)[0])


def test_oracle_identity_branch_is_a_no_op(br_oracle):
    kw = dict(seed=70, n_replicas=3, max_days=80, **stress_kw(30000))
    a, b = helpers.make_context(br_oracle, **kw), helpers.make_context(br_oracle, **kw)
    a.run(33)
    b.run(33)
    a.branch(np.arange(3), a.replica_seeds())
    assert a.branch(np.arange(3)).tolist() == [70, 71, 72]   # no state changes: nobody gets a new seed
    a.run(30)
    b.run(30)
    for r in range(3):
        assert_same_state(replica_state(a, r), replica_state(b, r), r)


def test_fresh_seeds_are_unused(br_oracle):
    ctx = helpers.make_context(br_oracle, seed=5, n_replicas=4, max_days=40, age_count_override=helpers.small_population(5000))
    ctx.run(10)
    s1 = ctx.branch(0)
    assert s1[0] == 5 and len(set(s1.tolist()) | {6, 7, 8}) == 7
    ctx.run(5)
    s2 = ctx.branch([1, 1, 2, 3])
    hist = ctx._engine.read_seeds()
    assert s2[0] not in set(hist[:, :15].ravel().tolist()) | set(s1.tolist())
    assert (hist[:, :10] == 5).all() and (hist[:, 10:15] == s1[[1, 1, 2, 3], None]).all() and (hist[:, 15:] == s2[:, None]).all()
    for bad in ([0, 0, 0, 4], [-1, 1, 2, 3], [1, 2, 2, 3]):
        with pytest.raises(_abi.EngineError):
            ctx.branch(bad)
    with pytest.raises(ValueError):
        ctx.branch([0, 1])


@pytest.mark.parametrize('seed', range(6))
def test_resample_and_assign_slots(seed):
    rng = np.random.default_rng(seed)
    for R in (1, 2, 7, 64, 256):
        w = rng.random(R) ** 8
        w[rng.random(R) < 0.3] = 0
        if not w.sum() > 0:
            w[0] = 1
        c = ensemble.systematic_resample(w, rng)
        assert c.sum() == R and (c >= 0).all() and (c[w == 0] == 0).all()
        assert (np.abs(c - R * w / w.sum()) < 1 + 1e-9).all()        # systematic: within one of the expected count
        src = ensemble.assign_slots(c)
        assert (src[src] == src).all() and ((0 <= src) & (src < R)).all()
        assert np.array_equal(np.bincount(src, minlength=R), c)
        assert (src[c > 0] == np.flatnonzero(c > 0)).all()
    assert ensemble.assign_slots([0, 3, 0, 1]).tolist() == [1, 1, 1, 3]
    with pytest.raises(ValueError):
        ensemble.assign_slots([2, 0, 0])
    with pytest.raises(ValueError):
        ensemble.systematic_resample([0.0, 0.0], rng)


def test_likelihood_matches_scipy():
    from scipy import stats
    mu = np.array([0.0, 0.4, 3.0, 17.5, 250.0])
    for y in (0, 1, 5, 40):
        for k in (0.5, 10.0, 300.0):
            want = stats.nbinom.logpmf(y, k, k / (k + mu))
            got = ensemble.log_likelihood(mu, y, 'negbin', k)
            np.testing.assert_allclose(got[1:], want[1:], rtol=1e-10)
            assert got[0] == (0.0 if y == 0 else -np.inf)
        np.testing.assert_allclose(ensemble.log_likelihood(mu[1:], y, 'poisson'), stats.poisson.logpmf(y, mu[1:]), rtol=1e-10)
        assert ensemble.log_likelihood([0.0], y, 'poisson')[0] == (0.0 if y == 0 else -np.inf)


def test_empty_observations_leave_a_plain_run(br_oracle):
    kw = dict(seed=3, n_replicas=3, max_days=40, age_count_override=helpers.small_population(8000))
    a, b = helpers.make_context(br_oracle, **kw), helpers.make_context(br_oracle, **kw)
    out = ensemble.particle_filter(a, {})
    assert out['log_evidence'] == 0.0 and out['ancestors'].shape == (0, 3) and a.day == 0
    a.run(30)
    b.run(30)
    assert np.array_equal(a.series(), b.series())


def test_collapse_raises(br_oracle):
    ctx = helpers.make_context(br_oracle, seed=3, n_replicas=3, max_days=40, age_count_override=helpers.small_population(8000))
    with pytest.raises(ValueError, match='day 4'):
        ensemble.particle_filter(ctx, {4: {'dead': 3}}, model='poisson')


def _filter_case(lib, n_agents, R, seed0, truth_seed, days, names):
    kw = dict(age_count_override=helpers.small_population(n_agents), max_days=days[-1] + 30)
    truth = helpers.make_context(br_oracle_library(), seed=truth_seed, **kw)
    truth.run(days[-1] + 1)
    t = truth.series(0, days[-1] + 1)
    obs = {d: {n: int(ensemble._model_counts(truth, t[:, d], n)[0]) for n in names} for d in days}
    ctx = helpers.make_context(lib, seed=seed0, n_replicas=R, **kw)
    return ctx, obs, kw


def test_filter_is_deterministic(br_oracle):
    outs = []
    for _ in range(2):
        ctx, obs, _ = _filter_case(br_oracle, 10000, 8, 100, 999, [10, 20, 30], ['in_ward', 'all_detected'])
        out = ensemble.particle_filter(ctx, obs, seed=4, ess_threshold=0.9)
        ctx.run(10)
        outs.append((out, ctx.series()))
    (a, ra), (b, rb) = outs
    assert all(np.array_equal(a[k], b[k]) for k in a) and np.array_equal(ra, rb)
    assert a['resampled'][-1] and a['ancestors'].shape == (3, 8)


def test_filter_conditions_on_the_observations(br_oracle):
    """The truth is an oracle run with a seed outside the ensemble's (40k agents, 16 replicas); in_ward and all_detected
    are observed weekly from day 7 to day 112.  At the observation days the filtered ensemble's paths are closer to the
    truth than those of the same ensemble run unconditioned.  Measured (deterministic), the mean absolute error over
    replicas and observation days, filtered / unconditioned: all_detected 0.572, in_ward 0.890 (a few dozen beds, where
    the counting noise of the truth is as large as the spread of the ensemble).  The bounds 0.7 and 1.0 leave room for
    changes of the resampling details."""
    days = list(range(7, 113, 7))
    ctx, obs, kw = _filter_case(br_oracle, 40000, 16, 100, 7777, days, ['in_ward', 'all_detected'])
    ensemble.particle_filter(ctx, obs, seed=1)
    plain = helpers.make_context(br_oracle, seed=100, n_replicas=16, **kw)
    plain.run(days[-1] + 1)
    f, p = ctx.series(0, days[-1] + 1), plain.series(0, days[-1] + 1)
    for n, bound in (('all_detected', 0.7), ('in_ward', 1.0)):
        truth = np.array([obs[d][n] for d in days], dtype=np.float64)
        err = lambda rows: np.abs(np.array([ensemble._model_counts(ctx, rows[:, d], n) for d in days]) - truth[:, None]).mean()
        ratio = err(f) / err(p)
        assert ratio < bound, (n, ratio)


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_small_population_all_replicas_equal_oracle(cuda_lib, br_oracle):
    """80k agents, every intervention type, 8 replicas, two rounds of branches: CUDA == reference in every series, agent
    field, queue entry, capacity counter, seed, transmission table and infection place."""
    kw = dict(stress_kw(), seed=11, n_replicas=8, max_days=130)
    gpu, cpu = helpers.make_context(cuda_lib, **kw), helpers.make_context(br_oracle, **kw)
    plan = [(30, [0, 0, 2, 2, 4, 0, 6, 2], [11, 500, 13, 501, 15, 502, 17, 503]),
            (60, [0, 1, 1, 3, 1, 5, 3, 0], [600, 601, 602, 603, 604, 605, 606, 607])]
    for day, src, seeds in plan:
        gpu.run(day - gpu.day)
        cpu.run(day - cpu.day)
        gpu.branch(src, seeds)
        cpu.branch(src, seeds)
        assert_same_ensemble(gpu, cpu, 'day %d' % day)
    gpu.run(60)
    cpu.run(60)
    assert_same_ensemble(gpu, cpu, 'day 120')


def _oracle_one_branched(args):
    seed, day, new_seed, days = args
    cpu = helpers.make_context(br_oracle_library(), seed=seed, max_days=181)
    cpu.run(day)
    cpu.branch([0], [new_seed])
    cpu.run(days - day)
    return cpu.series(0, days)[0], cpu._engine.read_agents(0), np.sort(cpu._engine.read_queue(0)), cpu._engine.read_available(0)


@pytest.mark.gpu
def test_bench_geometry_branch_equals_oracle(cuda_lib):
    """Full HUS, 256 replicas (four replica groups), half of the slots copied at day 60 and every slot re-seeded, run to
    180: a copied slot, its source and a slot copied across a group boundary against one-replica references."""
    R, seed0 = 256, 424242
    gpu = helpers.make_context(cuda_lib, seed=seed0, n_replicas=R, max_days=181)
    gpu.run(60)
    src = np.arange(R)
    src[1::2] = (np.arange(1, R, 2) * 7 + 40) % R & ~1      # odd slots copy an even one, often in another group
    seeds = 7000000 + np.arange(R)
    gpu.branch(src, seeds)
    gpu.run(120)
    rows = gpu.series(0, 180)
    j_same = next(j for j in range(1, R, 2) if src[j] // 64 == j // 64)
    j_cross = next(j for j in range(1, R, 2) if src[j] // 64 != j // 64)
    check = [j_same, src[j_same], j_cross]
    args = [(seed0 + src[j], 60, int(seeds[j]), 180) for j in check]
    with ProcessPoolExecutor(3, mp_context=multiprocessing.get_context('spawn')) as ex:
        refs = list(ex.map(_oracle_one_branched, args))
    for j, (r_rows, r_agents, r_queue, r_avail) in zip(check, refs):
        assert np.array_equal(rows[j], r_rows), j
        assert np.array_equal(gpu._engine.read_agents(j), r_agents), j
        assert np.array_equal(np.sort(gpu._engine.read_queue(j)), r_queue), j
        assert np.array_equal(gpu._engine.read_available(j), r_avail), j
    assert np.array_equal(rows[j_same, :60], rows[src[j_same], :60]) and not np.array_equal(rows[j_same, 61:], rows[src[j_same], 61:])
    gpu.close()


@pytest.mark.gpu
def test_identity_branch_changes_nothing_at_256_replicas(cuda_lib):
    kw = dict(seed=31000, n_replicas=256, max_days=181)
    a = helpers.make_context(cuda_lib, **kw)
    a.run(60)
    a.branch(np.arange(256), a.replica_seeds())
    a.run(120)
    b = helpers.make_context(cuda_lib, **kw)
    b.run(180)
    assert np.array_equal(a.series(0, 180), b.series(0, 180))
    for r in range(256):
        assert np.array_equal(a._engine.read_agents(r), b._engine.read_agents(r)), r
    a.close()
    b.close()


@pytest.mark.gpu
def test_branched_state_survives_save_load(cuda_lib):
    kw = dict(stress_kw(60000), seed=21, n_replicas=4, max_days=100)
    a = helpers.make_context(cuda_lib, **kw)
    a.run(35)
    a.branch([0, 0, 2, 0])
    a.run(12)
    blob = a.save_state()
    b = helpers.make_context(cuda_lib, **kw)
    b.load_state(blob)
    assert np.array_equal(b._engine.read_seeds(), a._engine.read_seeds())
    a.run(40)
    b.run(40)
    assert np.array_equal(a.series(), b.series())
    for r in range(4):
        assert np.array_equal(a._engine.read_agents(r), b._engine.read_agents(r)), r
    sa, sb = a.transmission_settings(), b.transmission_settings()
    assert all(np.array_equal(sa[k], sb[k]) for k in SETTINGS)
    # a version-2 blob (no seed history) of an unbranched state still loads and continues identically
    c = helpers.make_context(cuda_lib, **kw)
    c.run(30)
    v3 = c.save_state()
    v2 = v3[:v3.size - 4 * 4 * 101].copy()
    assert int(v3[8:12].view(np.int32)[0]) == 3
    v2[8:12] = np.array([2], dtype=np.int32).view(np.uint8)
    d = helpers.make_context(cuda_lib, **kw)
    d.load_state(v2)
    assert np.array_equal(d._engine.read_seeds(), c._engine.read_seeds())
    c.run(30)
    d.run(30)
    assert np.array_equal(c.series(), d.series())
    sc, sd = c.transmission_settings(), d.transmission_settings()
    assert all(np.array_equal(sc[k], sd[k]) for k in SETTINGS)
    with pytest.raises(_abi.EngineError):
        d.load_state(v3[:-4])


@pytest.mark.gpu
def test_bad_sources_are_refused(cuda_lib, br_oracle):
    kw = dict(stress_kw(20000), seed=9, n_replicas=4, max_days=60)
    gpu, cpu = helpers.make_context(cuda_lib, **kw), helpers.make_context(br_oracle, **kw)
    gpu.run(20)
    cpu.run(20)
    for bad in ([0, 1, 2, 4], [0, 1, 2, -1], [0, 0, 1, 3], [1, 2, 3, 0]):
        with pytest.raises(_abi.EngineError):
            gpu.branch(bad)
    gpu.run(20)                                              # the engine is fine afterwards
    cpu.run(20)
    assert not helpers.diff_report(gpu, cpu, 40)


def _sharded_worker(q):
    try:
        from reina_b200 import sharded
        kw = dict(stress_kw(20000), seed=9, max_days=60)
        ctxs = [helpers.make_context(helpers.cuda_library(), device=0, **kw) for _ in range(2)]
        sharded.join_local(ctxs)
        refused = 0
        for c in ctxs:
            try:
                c.branch([0], [5])
            except _abi.EngineError:
                refused += 1
        sharded.run_local(ctxs, 20)
        q.put((refused, [c.series(0, 20) for c in ctxs]))
    except Exception:
        q.put(traceback.format_exc())


@pytest.mark.gpu
def test_sharded_engine_refuses_to_branch(cuda_lib, oracle_lib, monkeypatch):
    monkeypatch.setenv('CUDA_DEVICE_MAX_CONNECTIONS', '32')
    monkeypatch.setenv('CUDA_MODULE_LOADING', 'EAGER')
    mpc = multiprocessing.get_context('spawn')
    q = mpc.Queue()
    p = mpc.Process(target=_sharded_worker, args=(q,))
    p.start()
    try:
        out = q.get(timeout=300)
    finally:
        p.join(timeout=30)
        if p.is_alive():
            p.kill()
    assert not isinstance(out, str), 'local ranks failed:\n%s' % out
    refused, rows = out
    assert refused == 2
    ref = helpers.make_context(oracle_lib, **dict(stress_kw(20000), seed=9, max_days=60))
    ref.run(20)
    for r in rows:
        assert np.array_equal(r, ref.series(0, 20))


@pytest.mark.gpu
def test_particle_filter_equals_oracle(cuda_lib, br_oracle):
    """80k agents, 16 replicas, weekly in_ward / all_detected of a truth run: the same ancestors, likelihoods, evidence
    and final rows on the CUDA engine and on the reference."""
    days = list(range(7, 85, 7))
    outs = []
    for lib in (cuda_lib, br_oracle):
        ctx, obs, _ = _filter_case(lib, 80000, 16, 300, 8888, days, ['in_ward', 'all_detected'])
        out = ensemble.particle_filter(ctx, obs, seed=2)
        ctx.run(20)
        outs.append((out, ctx.series(), ctx._engine.read_seeds()))
    (a, ra, sa), (b, rb, sb) = outs
    assert a['resampled'].sum() >= 2 and (a['ancestors'] != np.arange(16)).any()
    for k in ('ancestors', 'loglik', 'ess', 'resampled'):
        assert np.array_equal(a[k], b[k]), k
    assert a['log_evidence'] == b['log_evidence']
    assert np.array_equal(ra, rb) and np.array_equal(sa, sb)
