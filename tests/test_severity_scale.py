"""The per-replica severity scales (rb_set_severity_scale / rb_read_severity_scale, Context.set_severity_scale /
severity_scale) and the particle filter that estimates them from observed counts (ensemble.particle_filter's
severity_prior / severity_volatility).

CPU: scales of exactly 1 are the unscaled reference; the severity shares by age of every infected agent follow the
scaled tables (clamped at 1 included); in_ward, in_icu and dead per infection move the way each scale says; dohc' = 1
makes every effectively vaccinated symptomatic case FATAL; branches, records and copies carry the scales, reset() gives
1, bad values are refused and change nothing; the filter without severity_prior makes no severity call, with one it is
deterministic, equals a replay on one Context, and recovers a severity scale alone and jointly with transmission.
GPU: heterogeneous scales equal the reference on the every-intervention schedule and at the bench geometry, survive every
way a replica moves, return to 1 on reset, reach the initial state, hold on every rank of a population-sharded run, and
the CUDA filter with severity and transmission priors equals the reference's and its replay.

The CPU reference is tests/oracle_sscale.c over the reference of test_transmission_scale.py, compiled together with an
instrumented copy of the sequential oracle: the probes of test_transmission_settings.py and test_transmission_scale.py
plus SEVERITY_PROBES below, which add the scales to the copy's Replica and apply the engine's four clamped products where
the copy's symptom_severity reads its tables, for person_infect's draws only.  oracle/ itself stays as it is."""
import hashlib
import math
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
from reina_b200 import _abi, ensemble, inputs, model
from test_branch import assert_same_ensemble
from test_migrate import full_state
from test_transmission import stress_kw
from test_transmission_scale import TSCALE_PROBES, ts_oracle_library
from test_transmission_settings import ORACLE_PROBES

_SCALED = ('{\n'
           '        const float *m = sscale_m1_now;\n'
           '        sc = fminf(sc * (1.0f + m[0]), fmaxf(sc, 1.0f));\n'
           '        cc = fminf(cc * (1.0f + m[1]), fmaxf(cc, 1.0f));\n'
           '        fc = fminf(fc * (1.0f + m[2]), fmaxf(fc, 1.0f));\n'
           '    }\n')
# (anchor in oracle/reina_oracle.c, line inserted after it): the scales, applied where the CUDA engine applies them
SEVERITY_PROBES = [
    ('    int32_t epoch;\n', '    float sscale_m1[3];          /* test build: severe, critical, fatal scale - 1 */\n'),
    (' * first marks DEATH_OUTSIDE_HOSPITAL, so every FATAL case dies outside hospital: place of death is implied). */\n',
     'static const float *sscale_m1_now;     /* test build: the infecting replica\'s scales; NULL (unscaled) in the sampler */\n'),
    ('    float dohc = v->tab[RB_T_DEATH_OUTSIDE_HOSPITAL][age];\n',
     '    if (sscale_m1_now) dohc = fminf(dohc * (1.0f + sscale_m1_now[2]), fmaxf(dohc, 1.0f));\n'),
    ('    float sc = v->tab[RB_T_SEVERE][age], cc = v->tab[RB_T_CRITICAL][age], fc = v->tab[RB_T_FATAL][age];\n',
     '    if (sscale_m1_now) ' + _SCALED),
    ('    int vacc_eff = t->day_of_vaccination >= 0 && (e->day - t->day_of_vaccination) > 14;\n',
     '    sscale_m1_now = r->sscale_m1;\n'),
    ('    t->severity = (uint8_t)symptom_severity(v0, t->age, u01f(x[0]), vacc_eff);\n', '    sscale_m1_now = NULL;\n'),
]

_ss_oracle = None


def ss_oracle_library():
    """The probed oracle plus the transmission, settings, branch, migration, transmission-scale and severity-scale entry
    points, built once per source state."""
    global _ss_oracle
    if _ss_oracle is None:
        files = [('oracle', 'reina_oracle.c'), ('tests', 'oracle_transmission.c'), ('tests', 'oracle_settings.c'),
                 ('tests', 'oracle_branch.c'), ('tests', 'oracle_migrate.c'), ('tests', 'oracle_tscale.c'),
                 ('tests', 'oracle_sscale.c'), ('include', 'reina_b200.h')]
        probes = ORACLE_PROBES + TSCALE_PROBES + SEVERITY_PROBES
        src = {f: open(os.path.join(helpers.ROOT, *f), 'rb').read().decode() for f in files}
        key = hashlib.sha1(''.join(src[f] for f in files).encode() + repr(probes).encode()).hexdigest()[:16]
        lib = os.path.join(tempfile.gettempdir(), 'reina_ss_oracle_%d_%s.so' % (os.getuid(), key))
        if not os.path.exists(lib):
            text = src[('oracle', 'reina_oracle.c')]
            for anchor, line in probes:
                assert text.count(anchor) == 1, 'oracle probe anchor not found exactly once: %r' % anchor
                text = text.replace(anchor, anchor + line)
            src[('oracle', 'reina_oracle.c')] = text
            tree = tempfile.mkdtemp(prefix='reina_ss_oracle_')
            try:
                for f in files:
                    os.makedirs(os.path.join(tree, f[0]), exist_ok=True)
                    with open(os.path.join(tree, *f), 'w') as fh:
                        fh.write(src[f])
                tmp = '%s.%d.tmp' % (lib, os.getpid())
                subprocess.run([os.environ.get('CC', 'gcc'), '-O2', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math',
                                '-shared', '-o', tmp, os.path.join(tree, 'tests', 'oracle_sscale.c'), '-lm'], check=True)
                os.replace(tmp, lib)
            finally:
                shutil.rmtree(tree, ignore_errors=True)
        _ss_oracle = _abi.Library(lib, 'ro_')
        _ss_oracle.bind_transmission()
        _ss_oracle.bind_settings()
        _ss_oracle.bind_branch()
        _ss_oracle.bind_migrate()
        _ss_oracle.bind_tscale()
        _ss_oracle.bind_sscale()
    return _ss_oracle


@pytest.fixture(scope='module')
def ss_oracle():
    return ss_oracle_library()


def _set(ctx, triples):
    t = np.asarray(triples, dtype=np.float64).reshape(-1, 3)
    ctx.set_severity_scale(t[:, 0], t[:, 1], t[:, 2])


def _wild_type(ctx, ctx_kw):
    """The wild-type variant the Context was built with (Context.__init__)."""
    dp = inputs.build_context_args(ctx_kw.get('variables') or inputs.default_variables(), area='HUS',
                                   age_count_override=ctx_kw.get('age_count_override'))['disease_params']
    return model.make_variant(dp, ctx.n_ages)


def severity_probabilities(var, n_ages, scales):
    """[n_ages, 5] P(ASYMPTOMATIC .. FATAL) of an unvaccinated infection (vmod = 1) with a uniform draw in [0, 1), from
    the wild-type tables and the scales through the engine's clamped products (in float32, as the engine forms them)."""
    f32 = np.float32
    s, c, q = (f32(x) for x in scales)
    out = np.zeros((n_ages, 5))
    for age in range(n_ages):
        syc = float(f32(var.tab[_abi.T_SYMPTOMATIC][age]))
        tab = [f32(var.tab[t][age]) for t in (_abi.T_SEVERE, _abi.T_CRITICAL, _abi.T_FATAL, _abi.T_DEATH_OUTSIDE_HOSPITAL)]
        sc, cc, fc, d = (min(x * k, max(x, f32(1.0))) for x, k in zip(tab, (s, c, q, q)))
        sc, cc, fc, d = float(sc), float(cc), float(fc), float(d)
        seg = lambda a, b, lo, hi: max(0.0, min(b, hi) - max(a, lo))
        out[age, 0] = 1.0 - syc
        lo = d * syc if d != 0.0 else 0.0
        fatal = lo
        if d < 1.0:
            x = lambda t: d + (1.0 - d) * t           # val2 < t  <=>  val < d + (1 - d) t
            tF, tC, tS = x(fc * cc * sc * syc), x(cc * sc * syc), x(sc * syc)
            fatal += seg(0.0, tF, lo, syc)
            out[age, 3] = seg(tF, tC, lo, syc)
            out[age, 2] = seg(tC, tS, lo, syc)
            out[age, 1] = seg(tS, syc, lo, syc)
        out[age, 4] = fatal
    return out


# ---------------------------------------------------------------- CPU (oracle)
def test_oracle_scale_one_is_the_unscaled_reference(ss_oracle):
    """Scales of 1 set explicitly on the every-intervention schedule: every row, agent, queue and capacity counter
    equals the unprobed oracle's."""
    kw = dict(stress_kw(30000), seed=13, n_replicas=3, max_days=70)
    a = helpers.make_context(ss_oracle, **kw)
    b = helpers.make_context(helpers.oracle_library(), **kw)
    a.set_severity_scale(1.0, 1.0, 1.0)
    assert a.severity_scale().tolist() == [[1.0] * 3] * 3
    a.run(60)
    b.run(60)
    assert not helpers.diff_report(a, b, 60)


SHARE_CASES = [(1.0, 1.0, 1.0), (0.5, 2.0, 1.5),
               (16.0, 1.0, 16.0)]     # p_severe / p_symptomatic * 16 and p_death_outside_hospital * 16 clamp at 1 in old age


@pytest.mark.parametrize('scales', SHARE_CASES)
def test_oracle_severity_shares_follow_the_scaled_tables(ss_oracle, scales):
    """One run of 4 x 60000 agents over 80 days without vaccination: for every decade of age and every severity, the
    count among all infected agents is within 4 standard errors of what the scaled tables give."""
    kw = dict(age_count_override=helpers.small_population(60000))
    ctx = helpers.make_context(ss_oracle, seed=31, n_replicas=4, max_days=90, **kw)
    ctx.set_severity_scale(*scales)
    ctx.run(80)
    p = severity_probabilities(_wild_type(ctx, kw), ctx.n_ages, scales)
    if scales[0] == 16.0:
        assert p[85, 4] > 0.99 * (1.0 - p[85, 0])   # dohc' = 1: every symptomatic case of that age is FATAL
    age = np.repeat(np.arange(ctx.n_ages), np.diff(ctx._age_start))
    n_inf, n_sev = np.zeros(ctx.n_ages), np.zeros((ctx.n_ages, 5))
    for r in range(4):
        ag = ctx._engine.read_agents(r)
        assert (ag['day_of_vaccination'] < 0).all()
        inf = ag['state'] != 0
        n_inf += np.bincount(age[inf], minlength=ctx.n_ages)
        np.add.at(n_sev, (age[inf], ag['severity'][inf]), 1)
    assert n_inf.sum() > 50000
    for dec in range(10):
        sel = slice(10 * dec, 10 * dec + 10 if dec < 9 else ctx.n_ages)
        exp = (n_inf[sel, None] * p[sel]).sum(0)
        var = (n_inf[sel, None] * p[sel] * (1 - p[sel])).sum(0)
        obs = n_sev[sel].sum(0)
        assert (np.abs(obs - exp) <= 4 * np.sqrt(var) + 1e-9).all(), (dec, obs, exp, np.sqrt(var))


def test_oracle_each_scale_moves_its_series(ss_oracle):
    """Ward-days, ICU-days and deaths per infection over 70 days: severe raises in_ward, critical in_icu, fatal dead;
    fatal alone lowers in_icu (critical cases become deaths outside hospital)."""
    res = {}
    for scales in ((1, 1, 1), (0.5, 1, 1), (2, 1, 1), (1, 2, 1), (1, 1, 2)):
        ctx = helpers.make_context(ss_oracle, seed=77, n_replicas=4, max_days=80, age_count_override=helpers.small_population(40000))
        ctx.set_severity_scale(*scales)
        ctx.run(70)
        rows = ctx.series(0, 70)
        per = lambda name: sum(ensemble._model_counts(ctx, rows[:, d], name).sum() for d in range(70))
        inf = ensemble._model_counts(ctx, rows[:, 69], 'all_infected').sum()
        res[scales] = dict(ward=per('in_ward') / inf, icu=per('in_icu') / inf,
                           dead=ensemble._model_counts(ctx, rows[:, 69], 'dead').sum() / inf)
    base = res[(1, 1, 1)]
    assert res[(0.5, 1, 1)]['ward'] < base['ward'] < res[(2, 1, 1)]['ward'], res
    assert res[(1, 2, 1)]['icu'] > base['icu'], res
    assert res[(1, 1, 2)]['dead'] > base['dead'] and res[(1, 1, 2)]['icu'] < base['icu'], res


def test_oracle_dohc_at_one_makes_vaccinated_cases_fatal(ss_oracle):
    """fatal = 16 lifts p_death_outside_hospital to 1 in old age: (val - 1) / (1 - 1) = -inf for an effectively vaccinated
    agent whose draw passed dohc' * syc * 0.1, so every symptomatic one of those ages is FATAL, as the reference's
    expression gives."""
    kw = stress_kw(60000)
    ctx = helpers.make_context(ss_oracle, seed=3, n_replicas=2, max_days=90, **kw)
    var = _wild_type(ctx, kw)
    ctx.set_severity_scale(1.0, 1.0, 16.0)
    ctx.run(80)
    dohc = np.array([var.tab[_abi.T_DEATH_OUTSIDE_HOSPITAL][a] for a in range(ctx.n_ages)], dtype=np.float32)
    old = np.flatnonzero(dohc * np.float32(16.0) >= 1.0)
    assert old.size and old.min() >= 80
    age = np.repeat(np.arange(ctx.n_ages), np.diff(ctx._age_start))
    n = 0
    for r in range(2):
        ag = ctx._engine.read_agents(r)
        day = ctx._engine.read_infection_days(r)
        sel = (np.isin(age, old) & (ag['day_of_vaccination'] >= 0) & (day >= 0)
               & (day - ag['day_of_vaccination'] > 14) & (ag['severity'] != 0))
        n += sel.sum()
        assert (ag['severity'][sel] == 4).all(), np.bincount(ag['severity'][sel])
    assert n >= 5, n


def test_oracle_moves_carry_the_scales_and_reset_clears_them(ss_oracle):
    """A copy given its source's seed continues exactly as the source, which it can only do with the source's scales."""
    kw = dict(stress_kw(30000), max_days=80)
    a = helpers.make_context(ss_oracle, seed=40, n_replicas=3, **kw)
    b = helpers.make_context(ss_oracle, seed=90, n_replicas=3, **kw)
    sa = [[3.0, 0.5, 2.0], [0.4, 4.0, 0.7], [1.5, 1.0, 6.0]]
    _set(a, sa)
    a.set_transmission_scale([1.2, 0.8, 1.0])
    a.run(30)
    b.run(30)
    seeds = a.replica_seeds()
    b.import_replicas([0], a.export_replicas([0]), seeds[[0]])
    b.copy_replicas_from(a, [2], [1], seeds[[2]])
    a.branch([0, 0, 2], seeds[[0, 0, 2]])
    np.testing.assert_array_equal(a.severity_scale(), np.float32([sa[0], sa[0], sa[2]]))
    np.testing.assert_array_equal(b.severity_scale(), np.float32([sa[0], sa[2], [1, 1, 1]]))
    a.run(20)
    b.run(20)
    for (x, rx), (y, ry) in (((a, 1), (a, 0)), ((b, 0), (a, 0)), ((b, 1), (a, 2))):
        sx, sy = full_state(x, rx), full_state(y, ry)
        for k in sx:
            assert np.array_equal(sx[k], sy[k]), (rx, ry, k)
    a.reset(40)
    assert a.severity_scale().tolist() == [[1.0] * 3] * 3


def test_oracle_bad_scales_are_refused(ss_oracle):
    ctx = helpers.make_context(ss_oracle, seed=5, n_replicas=3, max_days=20, age_count_override=helpers.small_population(4000))
    _set(ctx, [[0.5, 1.0, 16.0], [2.0, 3.0, 0.25], [1.0, 1.0, 1.0]])
    before = ctx.severity_scale().copy()
    for col in ('severe', 'critical', 'fatal'):
        for bad in (0.0, -1.0, 16.5, np.nan, np.inf, [1, 1, np.nan], 1e300):
            with pytest.raises(_abi.EngineError):
                ctx.set_severity_scale(**{col: bad})
            assert np.array_equal(ctx.severity_scale(), before), (col, bad)
        for bad in ([1.0, 1.0], np.ones((3, 1))):
            with pytest.raises(ValueError):
                ctx.set_severity_scale(**{col: bad})
    # a refused column refuses the whole call: the valid ones given with it are not set either
    with pytest.raises(_abi.EngineError):
        ctx.set_severity_scale(severe=2.0, fatal=0.0)
    with pytest.raises(ValueError):
        ctx.set_severity_scale(severe=2.0, critical=[1.0])
    assert np.array_equal(ctx.severity_scale(), before)
    ctx.set_severity_scale(critical=[5.0, 6.0, 7.0])           # the other columns stay
    assert ctx.severity_scale().tolist() == [[0.5, 5.0, 16.0], [2.0, 6.0, 0.25], [1.0, 7.0, 1.0]]
    with pytest.raises(_abi.EngineError):
        ctx._engine.set_severity_scale(np.full((3, 3), 17.0, np.float32))


def _truth_obs(lib, days, names, n_agents, severe=1.0, f=1.0, seed=4242, max_days=None):
    """Observations {day: {name: count}} of one replica run with constant severe and transmission scales."""
    truth = helpers.make_context(lib, seed=seed, age_count_override=helpers.small_population(n_agents),
                                 max_days=max_days or days[-1] + 20)
    truth.set_severity_scale(severe=severe)
    truth.set_transmission_scale(f)
    truth.run(days[-1] + 1)
    t = truth.series(0, days[-1] + 1)
    return {d: {n: int(ensemble._model_counts(truth, t[:, d], n)[0]) for n in names} for d in days}


def _band(out, name, q=(0.05, 0.95)):
    v = out['transmission_scale'] if name == 'transmission' else out['severity_scale'][name]
    return ensemble.weighted_quantiles(v[-1], out['weights'][-1], list(q))


SEV_PRIOR = {'severe': (1.0, 0.5), 'fatal': (1.0, 0.3)}


def _replay(lib, out, R_total, seed0, kw, end):
    """One Context holding every replica, driven by the filter's output: its initial scales, at each observation day its
    ancestors and seeds where it resampled, then the scales it set for the next stretch."""
    one = helpers.make_context(lib, seed=seed0, n_replicas=R_total, **kw)
    sev = out['severity_scale'] or {}

    def put(k):
        if out['transmission_scale'] is not None:
            one.set_transmission_scale(out['transmission_scale'][k])
        if sev:
            one.set_severity_scale(**{n: v[k] for n, v in sev.items()})
    put(0)
    days = out['days']
    for k, d in enumerate(days):
        one.run(int(d) - one.day)
        if out['resampled'][k]:
            one.branch(out['ancestors'][k], out['seeds'][k])
        if k < len(days) - 1:
            put(k + 1)
    one.run(end - one.day)
    return one


def _filter_case(lib, n_agents=20000, days=(6, 12, 18, 24, 30)):
    kw = dict(age_count_override=helpers.small_population(n_agents), max_days=days[-1] + 20)
    obs = _truth_obs(lib, list(days), ('in_ward', 'all_detected'), n_agents, severe=1.5)
    return kw, obs


def test_oracle_filter_without_severity_prior_makes_no_severity_call(ss_oracle):
    """severity_prior None: the filter runs over the transmission-scale reference, which has no severity entry points
    (a call would fail there), and its outputs equal those over the severity reference, whose scales stay 1."""
    kw, obs = _filter_case(ss_oracle)
    outs = []
    for lib in (ss_oracle, ts_oracle_library()):
        ctx = helpers.make_context(lib, seed=500, n_replicas=8, **kw)
        outs.append(ensemble.particle_filter(ctx, obs, seed=3, ess_threshold=0.9, transmission_prior=(1.0, 0.4),
                                             transmission_volatility=0.05))
        ctx.run(40 - ctx.day)
        outs.append(ctx.series(0, 40))
        if lib is ss_oracle:
            assert ctx.severity_scale().tolist() == [[1.0] * 3] * 8
    (a, ra, b, rb) = outs
    assert a['severity_scale'] is None and b['severity_scale'] is None and np.array_equal(ra, rb)
    for k in a:
        if k != 'severity_scale':
            assert np.array_equal(a[k], b[k]), k
    with pytest.raises(ValueError):
        ensemble.particle_filter(ctx, obs, severity_prior={'hospital': (1.0, 0.5)})
    with pytest.raises(ValueError):
        ensemble.particle_filter(ctx, obs, severity_prior={'severe': (0.0, 0.5)})


def test_oracle_filter_with_severity_prior_is_deterministic_and_equals_replay(ss_oracle):
    """Twice the same; the transmission draws are those of a run without severity_prior; unnamed scales stay 1; and the
    filter over two Contexts equals a replay of its scales, ancestors and seeds on one Context holding all replicas."""
    kw, obs = _filter_case(ss_oracle)
    res = []
    for sev in (SEV_PRIOR, SEV_PRIOR, None):
        parts = [helpers.make_context(ss_oracle, seed=500 + k * 6, n_replicas=6, **kw) for k in range(2)]
        out = ensemble.particle_filter(parts, obs, seed=3, ess_threshold=0.9, transmission_prior=(1.0, 0.5),
                                       transmission_volatility=0.05, severity_prior=sev, severity_volatility=0.05)
        for p in parts:
            p.run(40 - p.day)
        res.append((out, parts))
    (a, pa), (b, _), (c, _) = res
    for k in a:
        if k == 'severity_scale':
            assert sorted(a[k]) == ['fatal', 'severe']
            assert all(np.array_equal(a[k][n], b[k][n]) for n in a[k])
        else:
            assert np.array_equal(a[k], b[k]), k
    ts = a['transmission_scale']
    assert np.array_equal(ts[0], c['transmission_scale'][0])    # the prior draws come first, before severity's
    ss = a['severity_scale']['severe']
    assert ss.shape == (5, 12) and len(np.unique(ss[0])) == 12 and (ss[1:] != ss[:-1]).any()
    for p in pa:
        assert (p.severity_scale()[:, 1] == 1.0).all()          # critical was not named
    one = _replay(ss_oracle, a, 12, 500, kw, 40)
    for g in range(12):
        x, y = full_state(pa[g // 6], g % 6), full_state(one, g)
        for k in x:
            assert np.array_equal(x[k], y[k]), (g, k)
    assert np.array_equal(np.concatenate([p.severity_scale() for p in pa]), one.severity_scale())
    assert np.array_equal(np.concatenate([p.transmission_scale() for p in pa]), one.transmission_scale())


def test_oracle_filter_recovers_a_severity_scale(ss_oracle):
    """Truth at severe = 0.6 (transmission 1) on 60000 agents, observed weekly to day 70 as in_ward and all_detected; 64
    replicas with prior severe: (1, 0.5), volatility 0.02, dispersion 100, filter seed 1: the final 90 % weighted band of
    the severe scale holds 0.6 and lies below 1."""
    days, n = list(range(7, 71, 7)), 60000
    obs = _truth_obs(ss_oracle, days, ('in_ward', 'all_detected'), n, severe=0.6, max_days=80)
    ctx = helpers.make_context(ss_oracle, seed=900, n_replicas=64, max_days=80, age_count_override=helpers.small_population(n))
    out = ensemble.particle_filter(ctx, obs, seed=1, dispersion=100.0, severity_prior={'severe': (1.0, 0.5)},
                                   severity_volatility=0.02)
    assert out['transmission_scale'] is None and list(out['severity_scale']) == ['severe']
    lo, hi = _band(out, 'severe')
    assert lo <= 0.6 <= hi < 1.0, (lo, hi)


def test_oracle_filter_recovers_transmission_and_severity_jointly(ss_oracle):
    """Truth at transmission 1.4 and severe 0.6 on 100000 agents, weekly in_ward, in_icu, dead and all_detected to day
    70; 64 replicas (seed 901) with priors (1, 0.5) on both, volatility 0.02, dispersion 100, filter seed 2: both final
    90 % bands hold the truth.  The two scales trade off against each other at this size: over six (filter, ensemble)
    seed pairs (2..7, 901..906) both bands held the truth in three, and the severe band missed 0.6 upwards in the others."""
    days, n = list(range(7, 71, 7)), 100000
    obs = _truth_obs(ss_oracle, days, ('in_ward', 'in_icu', 'dead', 'all_detected'), n, severe=0.6, f=1.4, max_days=80)
    ctx = helpers.make_context(ss_oracle, seed=901, n_replicas=64, max_days=80, age_count_override=helpers.small_population(n))
    out = ensemble.particle_filter(ctx, obs, seed=2, dispersion=100.0, transmission_prior=(1.0, 0.5),
                                   transmission_volatility=0.02, severity_prior={'severe': (1.0, 0.5)},
                                   severity_volatility=0.02)
    (tlo, thi), (slo, shi) = _band(out, 'transmission'), _band(out, 'severe')
    assert tlo <= 1.4 <= thi and slo <= 0.6 <= shi, (tlo, thi, slo, shi)


# ---------------------------------------------------------------- GPU
# severe, critical, fatal per replica: 0.25 .. 16; the last clamps sc and dohc (ages 80+) once the stress schedule has
# vaccinated the old
SEV5 = [(0.25, 0.5, 0.25), (0.5, 2.0, 1.0), (1.0, 1.0, 1.0), (2.0, 0.25, 4.0), (16.0, 16.0, 16.0)]
TS5 = [0.5, 1.0, 1.7, 1.0, 0.8]


@pytest.mark.gpu
def test_gpu_heterogeneous_scales_equal_oracle(cuda_lib, ss_oracle):
    """Five replicas of the every-intervention schedule (tracing, vaccination, imports, saturated beds and ICU) with
    severity triples from 0.25 to 16 and transmission scales on top, both changed at day 60: every series, agent field,
    queue, capacity counter, seed, transmission and settings table equals the reference."""
    kw = dict(stress_kw(), max_days=130, contact_capacity=2.0)
    gpu = helpers.make_context(cuda_lib, seed=11, n_replicas=5, **kw)
    cpu = helpers.make_context(ss_oracle, seed=11, n_replicas=5, **kw)
    for c in (gpu, cpu):
        _set(c, SEV5)
        c.set_transmission_scale(TS5)
        c.run(60)
        _set(c, SEV5[::-1])
        c.set_transmission_scale(TS5[::-1])
        c.run(60)
    assert np.array_equal(gpu.severity_scale(), cpu.severity_scale())
    assert (cpu._engine.read_agents(0)['day_of_vaccination'] >= 0).any()
    assert_same_ensemble(gpu, cpu, 'heterogeneous severity scales')


def _oracle_full_hus(args):
    seed, s = args
    ctx = helpers.make_context(ss_oracle_library(), area='HUS', seed=seed, max_days=181)
    ctx.set_severity_scale(*s)
    ctx.run(180)
    return ctx.series(0, 180)[0], ctx._engine.read_agents(0), np.sort(ctx._engine.read_queue(0)), ctx._engine.read_available(0)


@pytest.mark.gpu
def test_gpu_bench_geometry_with_severity_scales_equals_oracle(cuda_lib):
    """256 HUS replicas, 180 days, every third replica at (1.5, 0.7, 2.0) and replica 100 at (0.5, 3.0, 0.6): replicas 0,
    100 and 255 against the reference with the same seeds and scales."""
    seed = 616161
    s = np.ones((256, 3))
    s[::3] = (1.5, 0.7, 2.0)
    s[100] = (0.5, 3.0, 0.6)
    gpu = helpers.make_context(cuda_lib, area='HUS', seed=seed, n_replicas=256, max_days=181)
    _set(gpu, s)
    gpu.run(180)
    rows = gpu.series(0, 180)
    mine = {r: (rows[r], gpu._engine.read_agents(r), np.sort(gpu._engine.read_queue(r)), gpu._engine.read_available(r))
            for r in (0, 100, 255)}
    gpu.close()
    with ProcessPoolExecutor(3, mp_context=multiprocessing.get_context('spawn')) as ex:
        ref = dict(zip((0, 100, 255), ex.map(_oracle_full_hus, [(seed + r, tuple(s[r])) for r in (0, 100, 255)])))
    for r in (0, 100, 255):
        for a, b in zip(mine[r], ref[r]):
            assert np.array_equal(a, b), r
    assert not np.array_equal(rows[0], rows[1])


@pytest.mark.gpu
def test_gpu_severity_scales_survive_every_move(cuda_lib, ss_oracle):
    """branch, export / import, copy_replicas_from and save_state / load_state into a fresh Context: 30 days later the
    CUDA engines equal the reference that made the same moves; reset() gives 1."""
    kw = dict(stress_kw(), max_days=100, contact_capacity=2.0)
    sa = [(0.5, 2.0, 1.0), (3.0, 1.0, 0.5), (16.0, 16.0, 16.0), (1.0, 1.0, 1.0)]
    side = {}
    for name, lib in (('gpu', cuda_lib), ('cpu', ss_oracle)):
        a = helpers.make_context(lib, seed=21, n_replicas=4, **kw)
        b = helpers.make_context(lib, seed=61, n_replicas=4, **kw)
        _set(a, sa)
        a.set_transmission_scale([0.7, 1.3, 1.0, 1.0])
        for x in (a, b):
            x.run(40)
        a.branch([0, 1, 1, 3], [501, 502, 503, 504])
        b.import_replicas([0], a.export_replicas([2]), [601])
        b.copy_replicas_from(a, [1], [3], [602])
        side[name] = (a, b)
    (ga, gb), (ca, cb) = side['gpu'], side['cpu']
    c = helpers.make_context(cuda_lib, seed=0, n_replicas=4, **kw)
    assert c.severity_scale().tolist() == [[1.0] * 3] * 4
    c.load_state(ga.save_state())
    for x in (ga, gb, c, ca, cb):
        x.run(30)
    np.testing.assert_array_equal(ga.severity_scale(), np.float32([sa[0], sa[1], sa[1], sa[3]]))
    np.testing.assert_array_equal(gb.severity_scale(), np.float32([sa[1], (1, 1, 1), (1, 1, 1), sa[1]]))
    assert np.array_equal(c.severity_scale(), ga.severity_scale())
    assert_same_ensemble(ga, ca, 'branched')
    assert_same_ensemble(gb, cb, 'imported and copied')
    assert_same_ensemble(c, ca, 'loaded')
    ga.reset(21)
    assert ga.severity_scale().tolist() == [[1.0] * 3] * 4


@pytest.mark.gpu
def test_gpu_reset_and_initial_state(cuda_lib, ss_oracle):
    """reset() returns the scales to 1 and draws the initial state with 1; an initial state set after
    set_severity_scale draws with the scales, on both sides."""
    kw = dict(stress_kw(40000), seed=8, n_replicas=2, max_days=60)
    gpu = helpers.make_context(cuda_lib, **kw)
    _set(gpu, [(3.0, 2.0, 4.0), (0.4, 0.5, 0.3)])
    gpu.run(20)
    gpu.reset(8)
    assert gpu.severity_scale().tolist() == [[1.0] * 3] * 2
    gpu.run(40)
    cpu = helpers.make_context(ss_oracle, **kw)
    cpu.run(40)
    assert_same_ensemble(gpu, cpu, 'after reset')
    ipc = [0, 0, 0, 0, 400, 300, 900]      # dead, in_icu, in_ward, confirmed, incubating, ill, recovered
    side = []
    for lib in (cuda_lib, ss_oracle):
        x = helpers.make_context(lib, seed=9, n_replicas=2, max_days=40, age_count_override=helpers.small_population(50000))
        _set(x, [(16.0, 1.0, 1.0), (1.0, 1.0, 1.0)])
        x._engine.set_initial_state(ipc)
        x.run(30)
        side.append(x)
    assert_same_ensemble(side[0], side[1], 'initial state with scales')
    ag = [side[1]._engine.read_agents(r) for r in range(2)]
    assert (ag[0]['severity'] == 2).sum() > (ag[1]['severity'] == 2).sum()


def _local_worker(world, q):
    try:
        from reina_b200 import sharded
        kw = dict(stress_kw(), seed=11, max_days=130)
        ctxs = [helpers.make_context(helpers.cuda_library(), device=0, **kw) for _ in range(world)]
        sharded.join_local(ctxs)
        for c in ctxs:
            c.set_severity_scale(2.5, 0.6, 3.0)
            c.set_transmission_scale(1.3)
        sharded.run_local(ctxs, 50)
        for c in ctxs:
            c.set_severity_scale(severe=0.5, fatal=16.0)
        sharded.run_local(ctxs, 50)
        q.put([(c.series(0, 100), c.severity_scale()) for c in ctxs])
    except Exception:
        q.put(traceback.format_exc())


@pytest.mark.gpu
@pytest.mark.parametrize('world', [2, 4])
def test_gpu_local_ranks_with_severity_scales_equal_the_single_engine(cuda_lib, ss_oracle, monkeypatch, world):
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
    single = []
    for lib in (cuda_lib, ss_oracle):
        ref = helpers.make_context(lib, **dict(stress_kw(), seed=11, max_days=130))
        ref.set_severity_scale(2.5, 0.6, 3.0)
        ref.set_transmission_scale(1.3)
        ref.run(50)
        ref.set_severity_scale(severe=0.5, fatal=16.0)
        ref.run(50)
        single.append(ref)
    assert np.array_equal(single[0].series(0, 100), single[1].series(0, 100))
    for rank, (rows, s) in enumerate(out):
        assert np.array_equal(rows, single[0].series(0, 100)), rank
        assert np.array_equal(s, single[0].severity_scale()), rank


def _gpu_filter_case(lib, days=(14, 21, 28, 35, 42, 49), **extra):
    kw = dict(age_count_override=helpers.small_population(80000), max_days=days[-1] + 20,
              variables=stress_kw()['variables'], interventions=helpers.stress_interventions(), **extra)
    obs = _truth_obs(lib, list(days), ('in_ward', 'in_icu', 'dead', 'all_detected'), 80000, severe=0.7, f=1.3,
                     seed=8888, max_days=kw['max_days'])
    return kw, obs


FILTER_KW = dict(seed=2, ess_threshold=0.9, transmission_prior=(1.0, 0.5), transmission_volatility=0.05,
                 severity_prior={'severe': (1.0, 0.5), 'critical': (1.0, 0.3), 'fatal': (1.0, 0.3)}, severity_volatility=0.05)


@pytest.mark.gpu
def test_gpu_filter_with_severity_prior_equals_oracle_and_replay(cuda_lib, ss_oracle):
    """Two engines x 8 replicas with severity and transmission priors: ancestors, seeds, scales, weights and evidence
    equal the reference's filter, every replica equals it afterwards, and the split run equals its replay on one
    16-replica engine."""
    R, seed0 = 8, 11
    outs = []
    for lib in (cuda_lib, ss_oracle):
        kw, obs = _gpu_filter_case(lib)
        parts = [helpers.make_context(lib, seed=seed0 + k * R, n_replicas=R, **kw) for k in range(2)]
        out = ensemble.particle_filter(parts, obs, **FILTER_KW)
        for p in parts:
            p.run(kw['max_days'] - p.day)
        outs.append((out, parts))
    (a, pa), (b, pb) = outs
    for k in a:
        if k == 'severity_scale':
            assert sorted(a[k]) == sorted(b[k]) and all(np.array_equal(a[k][n], b[k][n]) for n in a[k])
        else:
            assert np.array_equal(a[k], b[k]), k
    for g, c in zip(pa, pb):
        assert_same_ensemble(g, c, 'gpu vs oracle')
    one = _replay(cuda_lib, a, 2 * R, seed0, kw, kw['max_days'])
    for g in range(2 * R):
        x, y = full_state(pa[g // R], g % R), full_state(one, g)
        for k in x:
            assert np.array_equal(x[k], y[k]), (g, k)


def _nccl_worker(rank, world, uid, q):
    try:
        from reina_b200 import comm as _comm
        R, seed0 = 8, 11
        kw, obs = _gpu_filter_case(helpers.cuda_library(), device=rank)
        ctx = helpers.make_context(helpers.cuda_library(), seed=seed0 + rank * R, n_replicas=R, **kw)
        c = _comm.connect(ctx._engine, rank=rank, size=world, unique_id=uid)
        out = ensemble.particle_filter(ctx, obs, comm=c, **FILTER_KW)
        ctx.run(kw['max_days'] - ctx.day)
        q.put((rank, dict(out=out, rows=ctx.series(0, kw['max_days']), scale=ctx.severity_scale())))
    except Exception:
        q.put((rank, traceback.format_exc()))


@pytest.mark.gpu
def test_gpu_nccl_filter_with_severity_prior_equals_replay(cuda_lib):
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
    for n in out['severity_scale']:
        assert np.array_equal(out['severity_scale'][n], res[1]['out']['severity_scale'][n]), n
    kw, _ = _gpu_filter_case(cuda_lib)
    one = _replay(cuda_lib, out, 2 * R, seed0, kw, kw['max_days'])
    rows, s = one.series(0, kw['max_days']), one.severity_scale()
    for k in range(2):
        assert np.array_equal(res[k]['rows'], rows[k * R:(k + 1) * R]), k
        assert np.array_equal(res[k]['scale'], s[k * R:(k + 1) * R]), k
