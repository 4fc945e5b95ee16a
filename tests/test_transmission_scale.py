"""The per-replica transmission scale (rb_set_transmission_scale / rb_read_transmission_scale,
Context.set_transmission_scale / transmission_scale) and a particle filter that estimates it from observed counts
(ensemble.particle_filter's transmission_prior / transmission_volatility, ensemble.weighted_quantiles).

CPU: a scale of exactly 1 is the unscaled reference; cohort R grows with the scale; branches, records and copies carry
it; bad values are refused and change nothing; the filter without a prior makes no new call, with one it is
deterministic, recovers a constant scale and follows a drop; the two-Context filter equals a replay on one Context.
GPU: heterogeneous scales equal the reference on small populations and at the bench geometry, survive every way a
replica moves, return to 1 on reset, hold on every rank of a population-sharded run, and the CUDA filter with a prior
equals the reference's.

The CPU reference is tests/oracle_tscale.c over the reference of test_migrate.py, compiled together with an instrumented
copy of the sequential oracle: the probes of test_transmission_settings.py plus TSCALE_PROBES below, which add the scale
to the copy's Replica and multiply p_upper and did_infect's p by it.  oracle/ itself stays as it is."""
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
from test_branch import assert_same_ensemble
from test_migrate import full_state, mg_oracle_library
from test_transmission import stress_kw
from test_transmission_settings import ORACLE_PROBES

# (anchor in oracle/reina_oracle.c, line inserted after it): the scale, applied where the CUDA engine applies it
TSCALE_PROBES = [
    ('    int32_t epoch;\n', '    float tscale_m1;             /* test build: the transmission scale f - 1 */\n'),
    ('    float p_upper = (si * v->reserved[0]) * v->infectiousness_multiplier;\n', '    p_upper = p_upper * (1.0f + r->tscale_m1);\n'),
    ('        float pr = (si * v->tab[RB_T_SUSCEPTIBILITY][t->age]) * v->infectiousness_multiplier;\n',
     '        pr = pr * (1.0f + r->tscale_m1);\n'),
]

_ts_oracle = None


def ts_oracle_library():
    """The probed oracle plus the transmission, settings, branch, migration and scale entry points, built once per source
    state."""
    global _ts_oracle
    if _ts_oracle is None:
        files = [('oracle', 'reina_oracle.c'), ('tests', 'oracle_transmission.c'), ('tests', 'oracle_settings.c'),
                 ('tests', 'oracle_branch.c'), ('tests', 'oracle_migrate.c'), ('tests', 'oracle_tscale.c'),
                 ('include', 'reina_b200.h')]
        probes = ORACLE_PROBES + TSCALE_PROBES
        src = {f: open(os.path.join(helpers.ROOT, *f), 'rb').read().decode() for f in files}
        key = hashlib.sha1(''.join(src[f] for f in files).encode() + repr(probes).encode()).hexdigest()[:16]
        lib = os.path.join(tempfile.gettempdir(), 'reina_ts_oracle_%d_%s.so' % (os.getuid(), key))
        if not os.path.exists(lib):
            text = src[('oracle', 'reina_oracle.c')]
            for anchor, line in probes:
                assert text.count(anchor) == 1, 'oracle probe anchor not found exactly once: %r' % anchor
                text = text.replace(anchor, anchor + line)
            src[('oracle', 'reina_oracle.c')] = text
            tree = tempfile.mkdtemp(prefix='reina_ts_oracle_')
            try:
                for f in files:
                    os.makedirs(os.path.join(tree, f[0]), exist_ok=True)
                    with open(os.path.join(tree, *f), 'w') as fh:
                        fh.write(src[f])
                tmp = '%s.%d.tmp' % (lib, os.getpid())
                subprocess.run([os.environ.get('CC', 'gcc'), '-O2', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math',
                                '-shared', '-o', tmp, os.path.join(tree, 'tests', 'oracle_tscale.c'), '-lm'], check=True)
                os.replace(tmp, lib)
            finally:
                shutil.rmtree(tree, ignore_errors=True)
        _ts_oracle = _abi.Library(lib, 'ro_')
        _ts_oracle.bind_transmission()
        _ts_oracle.bind_settings()
        _ts_oracle.bind_branch()
        _ts_oracle.bind_migrate()
        _ts_oracle.bind_tscale()
    return _ts_oracle


@pytest.fixture(scope='module')
def ts_oracle():
    return ts_oracle_library()


HETERO = [0.25, 0.5, 1.0, 1.7, 4.0]


def _truth_obs(lib, scale_of_day, days, names, n_agents, seed=4242, max_days=None):
    """Observations {day: {name: count}} of one replica run with the transmission scale scale_of_day(d) on day d."""
    truth = helpers.make_context(lib, seed=seed, age_count_override=helpers.small_population(n_agents),
                                 max_days=max_days or days[-1] + 20)
    for d in range(days[-1] + 1):
        f = scale_of_day(d)
        if d == 0 or f != scale_of_day(d - 1):
            truth.set_transmission_scale(f)
        truth.run(1)
    t = truth.series(0, days[-1] + 1)
    return {d: {n: int(ensemble._model_counts(truth, t[:, d], n)[0]) for n in names} for d in days}


def _final_band(out, q=(0.05, 0.95)):
    return ensemble.weighted_quantiles(out['transmission_scale'][-1], out['weights'][-1], list(q))


def _replay(lib, out, R_total, seed0, kw, end, volatility):
    """One Context holding every replica, driven by the filter's output: its initial scales, at each observation day its
    ancestors and seeds where it resampled, then the scales it set for the next stretch."""
    one = helpers.make_context(lib, seed=seed0, n_replicas=R_total, **kw)
    one.set_transmission_scale(out['transmission_scale'][0])
    days = out['days']
    for k, d in enumerate(days):
        one.run(int(d) - one.day)
        if out['resampled'][k]:
            one.branch(out['ancestors'][k], out['seeds'][k])
        if k < len(days) - 1 and volatility > 0:
            one.set_transmission_scale(out['transmission_scale'][k + 1])
    one.run(end - one.day)
    return one


# ---------------------------------------------------------------- CPU (oracle)
def test_oracle_scale_one_is_the_unscaled_reference(ts_oracle):
    """Scale 1 set explicitly: every row, agent, queue, capacity counter and table equals the unprobed oracle's."""
    kw = dict(stress_kw(30000), seed=13, n_replicas=3, max_days=70)
    a = helpers.make_context(ts_oracle, **kw)
    b = helpers.make_context(helpers.oracle_library(), **kw)
    a.set_transmission_scale(1.0)
    assert a.transmission_scale().tolist() == [1.0] * 3
    a.run(60)
    b.run(60)
    assert not helpers.diff_report(a, b, 60)


def test_oracle_cohort_R_grows_with_the_scale(ts_oracle):
    R = {}
    for f in (0.5, 1.0, 2.0):
        ctx = helpers.make_context(ts_oracle, seed=70, n_replicas=4, max_days=60, age_count_override=helpers.small_population(20000))
        ctx.set_transmission_scale(f)
        ctx.run(50)
        t = ctx.transmission_stats()
        R[f] = t['cohort_offspring'][:, :21].sum() / t['cohort_infected'][:, :21].sum()
    assert R[0.5] < R[1.0] < R[2.0], R


def test_oracle_branch_records_and_copies_carry_the_scale(ts_oracle):
    """A copy given its source's seed continues exactly as the source, which it can only do with the source's scale."""
    kw = dict(stress_kw(30000), max_days=80)
    a = helpers.make_context(ts_oracle, seed=40, n_replicas=3, **kw)
    b = helpers.make_context(ts_oracle, seed=90, n_replicas=3, **kw)
    a.set_transmission_scale([2.0, 0.6, 1.3])
    a.run(30)
    b.run(30)
    seeds = a.replica_seeds()
    b.import_replicas([0], a.export_replicas([0]), seeds[[0]])
    b.copy_replicas_from(a, [2], [1], seeds[[2]])
    a.branch([0, 0, 2], seeds[[0, 0, 2]])
    assert a.transmission_scale().tolist() == pytest.approx([2.0, 2.0, 1.3])
    assert b.transmission_scale().tolist() == pytest.approx([2.0, 1.3, 1.0])
    a.run(20)
    b.run(20)
    for (x, rx), (y, ry) in (((a, 1), (a, 0)), ((b, 0), (a, 0)), ((b, 1), (a, 2))):
        sx, sy = full_state(x, rx), full_state(y, ry)
        for k in sx:
            assert np.array_equal(sx[k], sy[k]), (rx, ry, k)


def test_oracle_bad_scales_are_refused(ts_oracle):
    ctx = helpers.make_context(ts_oracle, seed=5, n_replicas=3, max_days=20, age_count_override=helpers.small_population(4000))
    ctx.set_transmission_scale([0.5, 1.0, 16.0])
    before = ctx.transmission_scale().copy()
    for bad in ([np.nan, 1, 1], [1, 0.0, 1], [1, 1, -2], [16.5, 1, 1], [1, np.inf, 1], 1e300):
        with pytest.raises(_abi.EngineError):
            ctx.set_transmission_scale(bad)
        assert np.array_equal(ctx.transmission_scale(), before)
    for bad in ([1.0, 1.0], np.ones((3, 1))):
        with pytest.raises(ValueError):
            ctx.set_transmission_scale(bad)
    assert np.array_equal(ctx.transmission_scale(), before)


def test_weighted_quantiles():
    rng = np.random.default_rng(3)
    x = rng.random((4, 33))
    for q in (0.0, 0.05, 0.5, 0.9, 1.0):
        np.testing.assert_array_equal(ensemble.weighted_quantiles(x, np.ones_like(x), q),
                                      np.quantile(x, q, axis=-1, method='inverted_cdf'))
    # integer weights are repeated samples
    w = rng.integers(0, 4, 33)
    w[0] = 1
    xr = np.repeat(x[0], w)
    assert ensemble.weighted_quantiles(x[0], w, [0.1, 0.5, 0.95]).tolist() == \
        np.quantile(xr, [0.1, 0.5, 0.95], method='inverted_cdf').tolist()
    assert ensemble.weighted_quantiles([3.0, 1.0, 2.0], [0.0, 0.0, 1.0], 0.5) == 2.0
    for bad in (([1.0], [0.0]), ([1.0, 2.0], [1.0, -1.0]), ([1.0], [np.nan])):
        with pytest.raises(ValueError):
            ensemble.weighted_quantiles(*bad, 0.5)
    with pytest.raises(ValueError):
        ensemble.weighted_quantiles([1.0], [1.0], 1.5)


def _filter_case(lib, R=8, n_agents=20000, seed0=500, days=(6, 12, 18, 24, 30)):
    kw = dict(age_count_override=helpers.small_population(n_agents), max_days=days[-1] + 20)
    obs = _truth_obs(lib, lambda d: 1.0, list(days), ('in_ward', 'all_detected'), n_agents)
    return kw, obs


def test_oracle_filter_without_prior_makes_no_new_call(ts_oracle):
    """transmission_prior None: the outputs equal those over a reference that has no scale entry points at all (a call
    would fail there), the scales stay 1 and the new weights are the normalised weights of the log-likelihoods."""
    kw, obs = _filter_case(ts_oracle)
    outs = []
    for lib in (ts_oracle, mg_oracle_library()):
        ctx = helpers.make_context(lib, seed=500, n_replicas=8, **kw)
        outs.append(ensemble.particle_filter(ctx, obs, seed=3, ess_threshold=0.9))
        ctx.run(40 - ctx.day)
        outs.append(ctx.series(0, 40))
        if lib is ts_oracle:
            assert ctx.transmission_scale().tolist() == [1.0] * 8
    (a, ra, b, rb) = outs
    assert a['transmission_scale'] is None and np.array_equal(ra, rb)
    for k in a:
        if k != 'transmission_scale':
            assert np.array_equal(a[k], b[k]), k
    w0 = np.exp(a['loglik'][0] - a['loglik'][0].max())
    np.testing.assert_allclose(a['weights'][0], w0 / w0.sum(), rtol=1e-12)


def test_oracle_filter_with_prior_is_deterministic_and_equals_replay(ts_oracle):
    """Twice the same; and the filter over two Contexts equals a replay of its scales, ancestors and seeds on one Context
    holding all replicas."""
    kw, obs = _filter_case(ts_oracle)
    res = []
    for _ in range(2):
        parts = [helpers.make_context(ts_oracle, seed=500 + k * 6, n_replicas=6, **kw) for k in range(2)]
        out = ensemble.particle_filter(parts, obs, seed=3, ess_threshold=0.9, transmission_prior=(1.0, 0.5),
                                       transmission_volatility=0.05)
        for p in parts:
            p.run(40 - p.day)
        res.append((out, parts))
    (a, pa), (b, _) = res
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    ts = a['transmission_scale']
    assert ts.shape == (5, 12) and len(np.unique(ts[0])) == 12 and (ts[1:] != ts[:-1]).any()
    one = _replay(ts_oracle, a, 12, 500, kw, 40, 0.05)
    for g in range(12):
        x, y = full_state(pa[g // 6], g % 6), full_state(one, g)
        for k in x:
            assert np.array_equal(x[k], y[k]), (g, k)
    assert np.array_equal(np.concatenate([p.transmission_scale() for p in pa]), one.transmission_scale())


def test_oracle_filter_recovers_a_constant_scale(ts_oracle):
    """Truth at f* = 1.6, weekly in_ward and all_detected: the final 90 % weighted interval of the scale holds 1.6, and
    the prior's median 1 lies below it."""
    days = list(range(7, 71, 7))
    obs = _truth_obs(ts_oracle, lambda d: 1.6, days, ('in_ward', 'all_detected'), 30000, max_days=80)
    ctx = helpers.make_context(ts_oracle, seed=900, n_replicas=64, max_days=80, age_count_override=helpers.small_population(30000))
    out = ensemble.particle_filter(ctx, obs, seed=1, transmission_prior=(1.0, 0.5), transmission_volatility=0.02)
    lo, hi = _final_band(out)
    assert lo <= 1.6 <= hi and lo > 1.0, (lo, hi)


def test_oracle_filter_follows_a_drop(ts_oracle):
    """Truth at 1.0 until day 50, 0.6 after, weekly to day 91 while the epidemic is still large: with a volatility the
    filter does not raise, its median falls, and the final 90 % interval holds 0.6 and lies below 1."""
    days = list(range(7, 92, 7))
    n, kw = 100000, dict(max_days=100)
    obs = _truth_obs(ts_oracle, lambda d: 1.0 if d < 50 else 0.6, days, ('in_ward', 'all_detected'), n, **kw)
    ctx = helpers.make_context(ts_oracle, seed=901, n_replicas=64, age_count_override=helpers.small_population(n), **kw)
    out = ensemble.particle_filter(ctx, obs, seed=2, dispersion=100.0, transmission_prior=(1.0, 0.5),
                                   transmission_volatility=0.1)
    med = ensemble.weighted_quantiles(out['transmission_scale'], out['weights'], 0.5)
    lo, hi = _final_band(out)
    assert lo <= 0.6 <= hi and hi < 1.0 and med[-1] < med[days.index(49)], (lo, hi, med)


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_heterogeneous_scales_equal_oracle(cuda_lib, ts_oracle):
    """0.25 .. 4.0 across five replicas of the every-intervention schedule (tracing, saturated beds and ICU): every
    series, agent field, queue, capacity counter, seed, transmission and settings table equals the reference.  At 4.0 the
    imported variant's contacts reach kq = 256 with p >= 1."""
    from reina_b200 import inputs, model
    v = stress_kw()['variables']
    dp = inputs.build_context_args(v, area='HUS')['disease_params']
    var = model.make_variant(dict(dp, **dp['variants'][0]), 100)
    top = np.float32(np.float32(max(var.iot)) * np.float32(var.reserved[0])) * np.float32(var.infectiousness_multiplier)
    assert top * np.float32(4.0) >= 1.0
    kw = dict(stress_kw(), max_days=130, contact_capacity=2.0)    # at 4.0 the peak days hold more contacts than the default lists
    gpu = helpers.make_context(cuda_lib, seed=11, n_replicas=5, **kw)
    cpu = helpers.make_context(ts_oracle, seed=11, n_replicas=5, **kw)
    for c in (gpu, cpu):
        c.set_transmission_scale(HETERO)
        c.run(60)
        c.set_transmission_scale(HETERO[::-1])       # a change takes effect from the next day
        c.run(60)
    assert np.array_equal(gpu.transmission_scale(), cpu.transmission_scale())
    assert_same_ensemble(gpu, cpu, 'heterogeneous scales')


def _oracle_full_hus(args):
    seed, f = args
    ctx = helpers.make_context(ts_oracle_library(), area='HUS', seed=seed, max_days=181)
    ctx.set_transmission_scale(f)
    ctx.run(180)
    return ctx.series(0, 180)[0], ctx._engine.read_agents(0), np.sort(ctx._engine.read_queue(0)), ctx._engine.read_available(0)


@pytest.mark.gpu
def test_gpu_bench_geometry_with_scales_equals_oracle(cuda_lib):
    """256 HUS replicas, 180 days, a third of them at 1.4 and replica 100 at 0.7: replicas 0, 100 and 255 against the
    reference with the same seeds and scales."""
    seed = 616161
    f = np.ones(256, dtype=np.float32)
    f[::3] = 1.4
    f[100] = 0.7
    assert (f[0], f[255]) == (np.float32(1.4), np.float32(1.4)) and f[1] == 1.0
    gpu = helpers.make_context(cuda_lib, area='HUS', seed=seed, n_replicas=256, max_days=181)
    gpu.set_transmission_scale(f)
    gpu.run(180)
    rows = gpu.series(0, 180)
    mine = {r: (rows[r], gpu._engine.read_agents(r), np.sort(gpu._engine.read_queue(r)), gpu._engine.read_available(r))
            for r in (0, 100, 255)}
    gpu.close()
    with ProcessPoolExecutor(3, mp_context=multiprocessing.get_context('spawn')) as ex:
        ref = dict(zip((0, 100, 255), ex.map(_oracle_full_hus, [(seed + r, float(f[r])) for r in (0, 100, 255)])))
    for r in (0, 100, 255):
        for a, b in zip(mine[r], ref[r]):
            assert np.array_equal(a, b), r
    assert not np.array_equal(rows[0], rows[1])


@pytest.mark.gpu
def test_gpu_scale_survives_every_move(cuda_lib, ts_oracle):
    """branch, export / import, copy_replicas_from and save_state / load_state into a fresh Context: 30 days later the
    CUDA engines equal the reference that made the same moves."""
    kw = dict(stress_kw(), max_days=100, contact_capacity=2.0)
    side = {}
    for name, lib in (('gpu', cuda_lib), ('cpu', ts_oracle)):
        a = helpers.make_context(lib, seed=21, n_replicas=4, **kw)
        b = helpers.make_context(lib, seed=61, n_replicas=4, **kw)
        a.set_transmission_scale([0.5, 1.7, 4.0, 1.0])
        for x in (a, b):
            x.run(40)
        a.branch([0, 1, 1, 3], [501, 502, 503, 504])
        b.import_replicas([0], a.export_replicas([2]), [601])
        b.copy_replicas_from(a, [1], [3], [602])
        side[name] = (a, b)
    (ga, gb), (ca, cb) = side['gpu'], side['cpu']
    c = helpers.make_context(cuda_lib, seed=0, n_replicas=4, **kw)
    assert c.transmission_scale().tolist() == [1.0] * 4
    c.load_state(ga.save_state())
    for x in (ga, gb, c, ca, cb):
        x.run(30)
    assert ga.transmission_scale().tolist() == pytest.approx([0.5, 1.7, 1.7, 1.0])
    assert gb.transmission_scale().tolist() == pytest.approx([1.7, 1.0, 1.0, 1.7])
    assert np.array_equal(c.transmission_scale(), ga.transmission_scale())
    assert_same_ensemble(ga, ca, 'branched')
    assert_same_ensemble(gb, cb, 'imported and copied')
    assert_same_ensemble(c, ca, 'loaded')


@pytest.mark.gpu
def test_gpu_reset_returns_the_scales_to_one(cuda_lib, ts_oracle):
    kw = dict(stress_kw(40000), seed=8, n_replicas=2, max_days=60)
    gpu = helpers.make_context(cuda_lib, **kw)
    gpu.set_transmission_scale([3.0, 0.4])
    gpu.run(20)
    gpu.reset(8)
    assert gpu.transmission_scale().tolist() == [1.0, 1.0]
    gpu.run(40)
    cpu = helpers.make_context(ts_oracle, **kw)
    cpu.run(40)
    assert_same_ensemble(gpu, cpu, 'after reset')


def _local_worker(world, q):
    try:
        from reina_b200 import sharded
        kw = dict(stress_kw(), seed=11, max_days=130)
        ctxs = [helpers.make_context(helpers.cuda_library(), device=0, **kw) for _ in range(world)]
        sharded.join_local(ctxs)
        for c in ctxs:
            c.set_transmission_scale(1.6)
        sharded.run_local(ctxs, 50)
        for c in ctxs:
            c.set_transmission_scale(0.7)
        sharded.run_local(ctxs, 50)
        q.put([(c.series(0, 100), c.transmission_scale()) for c in ctxs])
    except Exception:
        q.put(traceback.format_exc())


@pytest.mark.gpu
@pytest.mark.parametrize('world', [2, 4])
def test_gpu_local_ranks_with_a_scale_equal_the_single_engine(cuda_lib, ts_oracle, monkeypatch, world):
    monkeypatch.setenv('CUDA_DEVICE_MAX_CONNECTIONS', '32')
    monkeypatch.setenv('CUDA_MODULE_LOADING', 'EAGER')
    mpc = multiprocessing.get_context('spawn')
    q = mpc.Queue()
    p = mpc.Process(target=_local_worker, args=(world, q))
    p.start()
    try:
        out = q.get(timeout=300)
    finally:
        p.join(timeout=30)
        if p.is_alive():
            p.kill()
    assert not isinstance(out, str), 'local ranks failed:\n%s' % out
    ref = helpers.make_context(ts_oracle, **dict(stress_kw(), seed=11, max_days=130))
    ref.set_transmission_scale(1.6)
    ref.run(50)
    ref.set_transmission_scale(0.7)
    ref.run(50)
    for rank, (rows, f) in enumerate(out):
        assert np.array_equal(rows, ref.series(0, 100)), rank
        assert np.array_equal(f, ref.transmission_scale()), rank


def _gpu_filter_case(lib, R, days=(14, 21, 28, 35, 42, 49), **extra):
    kw = dict(age_count_override=helpers.small_population(80000), max_days=days[-1] + 20,
              variables=stress_kw()['variables'], interventions=helpers.stress_interventions(), **extra)
    obs = _truth_obs(lib, lambda d: 1.3, list(days), ('in_ward', 'all_detected'), 80000, seed=8888, max_days=kw['max_days'])
    return kw, obs


@pytest.mark.gpu
def test_gpu_filter_with_prior_equals_oracle_and_replay(cuda_lib, ts_oracle):
    """Two engines x 8 replicas with a prior and a volatility: ancestors, seeds, scales, weights and evidence equal the
    reference's filter, every replica equals it afterwards, and the split run equals its replay on one 16-replica engine."""
    R, seed0 = 8, 11
    outs = []
    for lib in (cuda_lib, ts_oracle):
        kw, obs = _gpu_filter_case(lib, R)
        parts = [helpers.make_context(lib, seed=seed0 + k * R, n_replicas=R, **kw) for k in range(2)]
        out = ensemble.particle_filter(parts, obs, seed=2, ess_threshold=0.9, transmission_prior=(1.0, 0.5),
                                       transmission_volatility=0.05)
        for p in parts:
            p.run(kw['max_days'] - p.day)
        outs.append((out, parts))
    (a, pa), (b, pb) = outs
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    for g, c in zip(pa, pb):
        assert_same_ensemble(g, c, 'gpu vs oracle')
    one = _replay(cuda_lib, a, 2 * R, seed0, kw, kw['max_days'], 0.05)
    for g in range(2 * R):
        x, y = full_state(pa[g // R], g % R), full_state(one, g)
        for k in x:
            assert np.array_equal(x[k], y[k]), (g, k)


def _nccl_worker(rank, world, uid, q):
    try:
        from reina_b200 import comm as _comm
        R, seed0 = 8, 11
        kw, obs = _gpu_filter_case(helpers.cuda_library(), R, device=rank)
        ctx = helpers.make_context(helpers.cuda_library(), seed=seed0 + rank * R, n_replicas=R, **kw)
        c = _comm.connect(ctx._engine, rank=rank, size=world, unique_id=uid)
        out = ensemble.particle_filter(ctx, obs, seed=2, ess_threshold=0.9, transmission_prior=(1.0, 0.5),
                                       transmission_volatility=0.05, comm=c)
        ctx.run(kw['max_days'] - ctx.day)
        q.put((rank, dict(out=out, rows=ctx.series(0, kw['max_days']), scale=ctx.transmission_scale())))
    except Exception:
        q.put((rank, traceback.format_exc()))


@pytest.mark.gpu
def test_gpu_nccl_filter_with_prior_equals_replay(cuda_lib):
    """The filter above over two NCCL ranks, one GPU each: the same outputs on both ranks, and the rows and scales of the
    replay on one 16-replica engine.  Needs two GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    uid = _abi.shard_unique_id()
    mpc = multiprocessing.get_context('spawn')
    q = mpc.Queue()
    procs = [mpc.Process(target=_nccl_worker, args=(r, 2, uid, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = {}
    try:
        for _ in range(2):
            rank, r = q.get(timeout=900)
            assert not isinstance(r, str), 'rank %d failed:\n%s' % (rank, r)
            res[rank] = r
    finally:
        for p in procs:
            p.join(timeout=30)
            if p.is_alive():
                p.kill()
    R, seed0 = 8, 11
    out = res[0]['out']
    for k in ('ancestors', 'loglik', 'seeds', 'transmission_scale', 'weights'):
        assert np.array_equal(out[k], res[1]['out'][k]), k
    kw, _ = _gpu_filter_case(cuda_lib, R)
    one = _replay(cuda_lib, out, 2 * R, seed0, kw, kw['max_days'], 0.05)
    rows, f = one.series(0, kw['max_days']), one.transmission_scale()
    for k in range(2):
        assert np.array_equal(res[k]['rows'], rows[k * R:(k + 1) * R]), k
        assert np.array_equal(res[k]['scale'], f[k * R:(k + 1) * R]), k
