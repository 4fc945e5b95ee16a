"""Host-side logic: contact tables, intervention schedule, the Context surface (run on the CPU oracle library),
and that both shared libraries export every symbol of include/reina_b200.h."""
import re
import os

import numpy as np
import pytest

import helpers
from reina_b200 import _abi, inputs, model


def test_libraries_export_every_declared_symbol():
    hdr = open(os.path.join(helpers.ROOT, 'include', 'reina_b200.h')).read()
    declared = sorted(set(re.findall(r'\brb_([a-z_]+)\s*\(', hdr)))
    assert set(declared) == set(_abi.SYMBOLS) | set(_abi.SHARD_SYMBOLS), set(declared) ^ (set(_abi.SYMBOLS) | set(_abi.SHARD_SYMBOLS))
    cuda = _abi.Library(_abi.CUDA_LIB_PATH, 'rb_')          # loads without a GPU; no compute call is made
    orac = helpers.oracle_library()
    for name in declared:
        assert hasattr(cuda.dll, 'rb_' + name), name
        # the multi-GPU entry points have no counterpart in the sequential CPU oracle
        assert name in _abi.SHARD_SYMBOLS or hasattr(orac.dll, 'ro_' + name), name


def test_shard_ownership_is_a_balanced_partition():
    """Stripes of 4096 age-sorted agents dealt round-robin: every agent has exactly one owner and every rank
    holds close to 1/nranks of every age decade (what keeps the per-rank sweep work balanced)."""
    counts = inputs.synthetic_age_counts(1685983)
    age_of = np.repeat(np.arange(len(counts)), counts)
    for nranks in (1, 2, 4, 8):
        owner = _abi.owner_of(np.arange(age_of.size), nranks)
        assert owner.min() == 0 and owner.max() == nranks - 1
        for decade in range(9):
            sel = (age_of // 10 == decade) if decade < 8 else (age_of >= 80)
            share = np.bincount(owner[sel], minlength=nranks) / sel.sum()
            assert np.abs(share - 1.0 / nranks).max() < 0.05, (nranks, decade, share)


def test_no_cpu_fallback(tmp_path):
    """The product must fail loudly when its CUDA library is missing, and creating a Context without a GPU fails."""
    with pytest.raises(_abi.EngineError):
        _abi.Library(str(tmp_path / 'libreina_b200.so'), 'rb_')
    import ctypes
    ndev = ctypes.c_int(0)
    try:
        rc = ctypes.CDLL('libcudart.so').cudaGetDeviceCount(ctypes.byref(ndev))
    except OSError:
        rc = 1
    if rc != 0 or ndev.value == 0:
        with pytest.raises(_abi.EngineError, match='no CUDA device|CUDA'):
            helpers.make_context(_abi.cuda_library(), age_count_override=helpers.small_population(2000))


def _pandas_tables(cm):
    """ContactMatrix.generate_contact_probabilities restated with the pandas operations of main.pyx:1195-1235."""
    import pandas as pd
    recs = []
    for (place, band), col in zip(cm.keys, range(len(cm.keys))):
        for age in range(cm.n_ages):
            recs.append((place, age, band, cm.base[age, col]))
    df = pd.DataFrame(recs, columns=['place_type', 'participant_age', 'contact_age', 'contacts'])
    for place, min_age, max_age, factor in cm.mobility_factors:
        if factor == 1.0:
            continue
        flt = (df.participant_age >= min_age) & (df.participant_age <= max_age)
        if place != model.PLACE_ALL:
            flt &= df.place_type == model.CONTACT_PLACE_TO_STR[place]
        df.loc[flt, 'contacts'] *= float(factor)
    total = df.groupby('participant_age')['contacts'].sum()
    df = df.set_index(['place_type', 'participant_age', 'contact_age']).sort_index()
    df = df.unstack('participant_age')
    df.columns = df.columns.droplevel(0)
    cum = df.divide(total, axis=1).cumsum()
    return total.values, cum.values.T, list(cum.index)


def test_contact_tables_match_pandas_restatement():
    cm = model.ContactMatrix(inputs.contacts_long(), 101)
    cm.set_mobility_factor(0.2, place=5, min_age=0, max_age=70)
    cm.set_mobility_factor(0.95)
    cm.set_mobility_factor(0.0, place=2, min_age=19, max_age=None)
    cm.set_mask_probability(0.8, min_age=65)
    t = cm.generate()
    total, cum, index = _pandas_tables(cm)
    nk = len(cm.keys)
    assert [(p, b) for p, b in index] == cm.keys                     # row order: place name, then band
    np.testing.assert_allclose(t['nr_contacts'], total, rtol=1e-12)
    np.testing.assert_allclose(t['cum_p'][:, :nk], cum, rtol=0, atol=1e-12)
    assert (np.diff(t['cum_p'][:, :nk], axis=1) >= 0).all()
    assert t['mask_p'][70, 0] == np.float32(0.8) and t['mask_p'][30, 0] == 0
    assert cm.mobility_factor == np.float32(0.0)                      # last factor set, any key (main.pyx:1251)
    # tabulated number-of-contacts distribution: monotone, and equal to the sampled lognormal rule
    cdf = t['ncontact_cdf']
    assert (np.diff(cdf[:, 0, :], axis=1) >= 0).all() and (cdf <= 1).all()
    rng = np.random.default_rng(5)
    c = total[30]
    f = np.maximum(rng.lognormal(0, 0.5, 400000) * c, 1.0).astype(np.int64) - 1
    emp = (np.minimum(f, 100)[:, None] <= np.arange(6)[None, :]).mean(0)
    np.testing.assert_allclose(emp, cdf[30, 0, :6], atol=4e-3)


@pytest.mark.parametrize('seed', range(8))
def test_contact_tables_random_mobility_sequences(seed):
    """Random sequences of limit-mobility settings (keys stack multiplicatively, a repeated key is overwritten,
    main.pyx:1250-1266) against the pandas restatement of generate_contact_probabilities."""
    rng = np.random.default_rng(100 + seed)
    cm = model.ContactMatrix(inputs.contacts_long(), 101)
    for _ in range(int(rng.integers(1, 9))):
        place = None if rng.random() < 0.3 else int(rng.integers(0, 6))
        lo = None if rng.random() < 0.4 else int(rng.integers(0, 80))
        hi = None if rng.random() < 0.4 else int(rng.integers(lo or 0, 101))
        cm.set_mobility_factor(float(rng.choice([0.0, 0.05, 0.2, 0.5, 0.8, 1.0])), place=place, min_age=lo, max_age=hi)
    if all(f[3] == 0.0 for f in cm.mobility_factors if f[0] == model.PLACE_ALL and f[1] == 0 and f[2] == 100) and \
            any(f[0] == model.PLACE_ALL and f[1] == 0 and f[2] == 100 for f in cm.mobility_factors):
        pytest.skip('all contacts switched off for everybody: the reference divides by zero there too')
    t = cm.generate()
    total, cum, index = _pandas_tables(cm)
    nk = len(cm.keys)
    ok = total > 0                      # an age whose every contact is switched off has no distribution (0 / 0) on both sides
    np.testing.assert_allclose(t['nr_contacts'], total, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(t['cum_p'][ok, :nk], cum[ok], rtol=0, atol=1e-12)
    assert (np.diff(t['cum_p'][ok, :nk], axis=1) >= -1e-15).all()
    assert np.all(np.abs(t['cum_p'][ok, nk - 1] - 1.0) < 1e-12)
    cdf = t['ncontact_cdf']
    assert (np.diff(cdf, axis=2) >= 0).all() and (cdf <= 1).all() and (cdf >= 0).all()


def test_intervention_tuples_and_schedule(oracle_lib):
    ivs = inputs.active_interventions()
    assert len(ivs) == 40 and ivs[6].get_param_values() == dict(reduction=80, min_age=0, max_age=70, place='other')
    assert inputs.iv_tuple_to_obj(['wear-masks', '2020-07-01', 80, 65, None, None]).get_param_values() == \
        dict(share_of_contacts=80, min_age=65)
    assert len(inputs.scenario_interventions('mitigation')) == 58
    halved = inputs.scenario_interventions('looser-restrictions-to-start-with')
    assert halved[6][2] == 40 and halved[8][2] == 2
    ctx = helpers.make_context(oracle_lib, age_count_override=helpers.small_population(5000), max_days=300)
    ctx.run(260)
    plan = ctx._plan
    assert [plan[d].testing_mode for d in (0, 2, 26, 118)] == [0, 2, 3, 1]          # NO_TESTING, ALL, ONLY_SEVERE, CT
    assert abs(plan[41].p_detected_anyway - 0.5) < 1e-6 and abs(plan[118].p_successful_tracing - 0.3) < 1e-6
    assert plan[4].n_imports == 1 and plan[4].import_amount[0] == 20                 # 2020-02-22
    # 50 / week from 2020-07-01 through a C-float accumulator (main.pyx:1671-1685): 7 x 7.142857 truncates to 49
    assert sum(p.trickle[0] for p in plan[134:141]) in (49, 50) and 498 <= sum(p.trickle[0] for p in plan[134:204]) <= 500
    assert sum(p.trickle[0] for p in plan[:134]) == 0
    epochs = [p.table_epoch for p in plan]
    assert epochs[0] == 0 and epochs[23] == 1 and max(epochs) == 11 and sorted(set(epochs)) == list(range(12))
    s = ctx.generate_state()
    assert abs(s['mobility_limitation'] - (1 - np.float32(1.0))) < 1e-6
    assert ctx.get_date_for_today() == '2020-11-04'


def test_context_surface(oracle_lib):
    ctx = helpers.make_context(oracle_lib, age_count_override=helpers.small_population(8000), seed=3)
    s0 = ctx.generate_state()
    assert set(s0) >= {'available_icu_units', 'available_hospital_beds', 'total_icu_units', 'r', 'exposed_per_day',
                       'ct_cases_per_day', 'mobility_limitation', 'infected_by_variant', 'daily_contacts', *_abi.ATTRS}
    assert s0['susceptible'].dtype == np.int32 and s0['susceptible'].sum() == 8000 and s0['infected'].sum() == 0
    assert list(s0['infected_by_variant']) == ['wild-type', 'b1.1.7']
    assert list(s0['daily_contacts']) == ['home', 'work', 'school', 'transport', 'leisure', 'other']
    for _ in range(30):
        ctx.iterate()
    s = ctx.generate_state()
    tot = sum(s[k].sum() for k in ('susceptible', 'infected', 'recovered', 'dead'))
    assert tot == 8000 and s['all_infected'].sum() > 0
    assert (ctx.get_population_stats('all_infected') >= 0).all() and len(ctx.get_population_stats('dead')) == 101
    with pytest.raises(Exception):
        ctx.get_population_stats('nonsense')
    with pytest.raises(Exception):
        ctx.apply_intervention(inputs.Intervention('no-such-intervention', '2020-01-01'))
    assert model.PROBLEM_TO_STR[7] == 'Wrong state' and model.SEVERITY_TO_STR[4] == 'FATAL'
    assert model.DISEASE_PARAMS[0] == 'p_susceptibility' and len(model.DISEASE_PARAMS) == 18
    # reset(): a fresh run with another seed, same plan
    ctx.reset(77)
    assert ctx.day == 0 and ctx.generate_state()['infected'].sum() == 0


def test_ensemble_replicas_and_reset(oracle_lib):
    counts = helpers.small_population(6000)
    a = helpers.make_context(oracle_lib, age_count_override=counts, seed=10, n_replicas=2)
    a.run(60)
    rows = a.series(0, 60)
    b = helpers.make_context(oracle_lib, age_count_override=counts, seed=11)
    b.run(60)
    assert np.array_equal(rows[1], b.series(0, 60)[0])
    a.reset(11)
    a.run(60)
    assert np.array_equal(a.series(0, 60)[0], rows[1])


def test_simulate_individuals_shapes(oracle_lib):
    from reina_b200 import simulation
    v = inputs.default_variables(simulation_days=25)
    ctx = helpers.make_context(oracle_lib, variables=v, age_count_override=helpers.small_population(4000), max_days=30)
    seen = []
    df, adf = simulation.simulate_individuals(v, context=ctx, step_callback=lambda d: seen.append(len(d.dropna())) or True,
                                              callback_day_interval=10)
    assert seen == [10, 20, 25]
    assert list(df.columns) == simulation.POP_ATTRS + simulation.STATE_ATTRS + simulation.EXPOSURES_ATTRS + ['us_per_infected']
    assert df.shape == (25, 26) and adf.shape == (25, 12 * 9)
    assert adf.columns.names == ['attr', 'age_group'] and ('dead', '80+') in adf.columns
    assert df['susceptible'].iloc[0] == 4000
    with pytest.raises(simulation.ExecutionInterrupted):
        simulation.simulate_individuals(v, context=helpers.make_context(
            oracle_lib, variables=v, age_count_override=helpers.small_population(4000), max_days=30),
            step_callback=lambda d: False)


def test_monte_carlo_driver_and_percentile_bands(oracle_lib, tmp_path):
    """run_monte_carlo (calc/simulation.py:365-385 made to work): long frame with run / scenario columns, the csv the
    reference writes, and percentile bands per day."""
    from reina_b200 import ensemble, simulation
    v = inputs.default_variables(simulation_days=30)
    ctx = helpers.make_context(oracle_lib, variables=v, age_count_override=helpers.small_population(6000), n_replicas=4, max_days=31)
    csv = tmp_path / 'reina_default.csv'
    df, bands = simulation.run_monte_carlo('default', n_seeds=10, seed0=100, variables=v, context=ctx, csv_path=str(csv),
                                           bands=(5, 50, 95))
    assert sorted(df['run'].unique()) == list(range(100, 110))           # the last launch is only partly used
    assert len(df) == 10 * 30 and set(df['scenario']) == {'default'} and csv.exists()
    assert set(bands) == {5, 50, 95} and bands[50].shape == (30, 25)
    assert (bands[5].to_numpy() <= bands[50].to_numpy()).all() and (bands[50].to_numpy() <= bands[95].to_numpy()).all()
    per_run = df.pivot(index='date', columns='run', values='all_infected').to_numpy()
    assert np.allclose(bands[50]['all_infected'].to_numpy(), np.percentile(per_run, 50, axis=1))
    # replica r of a launch == the single run with that seed
    single = helpers.make_context(oracle_lib, variables=v, age_count_override=helpers.small_population(6000), seed=105, max_days=31)
    one, _ = simulation.simulate_individuals(v, context=single)
    assert np.array_equal(one['all_infected'].to_numpy(), df[df['run'] == 105]['all_infected'].to_numpy())
    cube = np.arange(24, dtype=float).reshape(4, 3, 2)
    assert np.allclose(ensemble.percentile_bands(cube, (0, 100))[100], cube[3]) and np.allclose(ensemble.gather_rows(cube), cube)


def test_serving_worker_reuses_contexts(oracle_lib):
    """The long-lived worker of reina_b200.serving (replaces a process per request, simulation_thread.py:14-61):
    results / finished / error entries, context reuse across seeds, a new context for other inputs, cancellation."""
    from reina_b200 import serving, simulation
    built = []

    def factory(v, scenario):
        built.append(v['simulation_days'])
        return helpers.make_context(oracle_lib, variables=v, scenario=scenario, seed=v['random_seed'],
                                    age_count_override=helpers.small_population(5000), max_days=v['simulation_days'] + 1)

    w = serving.SimulationWorker(context_factory=factory, callback_day_interval=10, max_contexts=2)
    v = inputs.default_variables(simulation_days=25)
    jobs = []
    for seed in (7, 8):
        vv = dict(v); vv['random_seed'] = seed
        jobs.append(w.submit(vv))
    res = [w.wait(j, timeout=120) for j in jobs]
    assert all(r['finished'] and r['error'] is None for r in res)
    assert [r['reused_context'] for r in res] == [False, True] and built == [25]
    assert res[0]['total'].shape == (25, 26) and res[0]['age_groups'].shape == (25, 12 * 9)
    assert not res[0]['total']['all_infected'].equals(res[1]['total']['all_infected'])      # different seeds
    vv = dict(v); vv['random_seed'] = 8
    direct, _ = simulation.simulate_individuals(vv, context=factory(vv, None))
    assert np.array_equal(direct['all_infected'].to_numpy(), res[1]['total']['all_infected'].to_numpy())
    v2 = inputs.default_variables(simulation_days=12)
    r2 = w.wait(w.submit(v2), timeout=120)
    assert r2['finished'] and not r2['reused_context'] and r2['total'].shape[0] == 12
    # a failing request reports its error like the reference's <key>-error entry
    bad = dict(v); bad['interventions'] = [['no-such-intervention', '2020-02-20']]
    r3 = w.wait(w.submit(bad), timeout=120)
    assert r3['finished'] and r3['error']
    w.close()


def test_surface_equals_the_reference_module(oracle_lib):
    """Side by side with the UNMODIFIED reference module (oracle/_ref): module constants, the keys / dtypes / shapes of
    generate_state(), get_population_stats(), get_date_for_today() and the exception behaviour (SURVEY.md section 8b)."""
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip('oracle/_ref not built')
    ref_model = ref_harness.load_model()
    assert tuple(ref_model.DISEASE_PARAMS) == tuple(model.DISEASE_PARAMS)
    assert dict(ref_model.SEVERITY_TO_STR) == model.SEVERITY_TO_STR and dict(ref_model.STATE_TO_STR) == model.STATE_TO_STR
    assert dict(ref_model.PROBLEM_TO_STR) == model.PROBLEM_TO_STR
    assert issubclass(ref_model.SimulationFailed, Exception) and issubclass(model.SimulationFailed, Exception)
    counts = helpers.small_population(8000)
    ref = ref_harness.make_context(age_count_override=counts, seed=3)
    mine = helpers.make_context(oracle_lib, age_count_override=counts, seed=3)
    for day in range(3):
        a, b = ref.generate_state(), mine.generate_state()
        assert set(a) == set(b), set(a) ^ set(b)
        for k in a:
            if isinstance(a[k], np.ndarray):
                assert a[k].dtype == b[k].dtype == np.int32 and a[k].shape == b[k].shape, k
            elif isinstance(a[k], dict):
                assert list(a[k]) == list(b[k]), k
            else:
                assert isinstance(b[k], (int, float)), k
        if day == 0:        # before the first iterate() nothing is random: the rows are equal
            for k in a:
                if isinstance(a[k], np.ndarray):
                    assert np.array_equal(a[k], b[k]), k
                elif isinstance(a[k], dict):
                    assert a[k] == b[k], k
                else:
                    assert abs(a[k] - b[k]) < 1e-6, k
        assert ref.get_date_for_today() == mine.get_date_for_today()
        ref.iterate(); mine.iterate()
    for what in ('dead', 'all_infected', 'all_detected'):
        ra, rb = np.asarray(ref.get_population_stats(what)), np.asarray(mine.get_population_stats(what))
        assert ra.shape == rb.shape and ra.dtype.kind == rb.dtype.kind == 'i', what
    for ctx in (ref, mine):
        with pytest.raises(Exception):
            ctx.get_population_stats('nonsense')
        with pytest.raises(Exception):
            ctx.apply_intervention(inputs.Intervention('no-such-intervention', '2020-01-01'))


@pytest.mark.parametrize('gold_name,area', [('varsinais_suomi_default_n256', 'Varsinais-Suomi'), ('hus_default_n256', 'HUS')])
def test_day0_state_equals_the_stored_reference_rows(oracle_lib, gold_name, area):
    """The day-0 half of the comparison above without the reference module: before the first iterate() nothing is
    random, so generate_state() must give, in every series, the value the unmodified reference engine gave in all 256
    seeds of its stored ensemble (tests/golden/make_golden.py)."""
    from oracle import ref_harness
    gold = np.load(os.path.join(helpers.ROOT, 'tests', 'golden', 'ref_ensemble_%s.npz' % gold_name))
    assert list(gold['names']) == ref_harness.series_names() and (gold['std'][0] == 0).all()
    ctx = helpers.make_context(oracle_lib, area=area, seed=3)
    row = np.array(ref_harness.state_row(ctx.generate_state()))
    bad = np.flatnonzero(row != gold['mean'][0])
    assert not len(bad), [(gold['names'][k], row[k], gold['mean'][0, k]) for k in bad]


# ---------------------------------------------------------------------------------------------------
# round-2 host logic: intervention ordering, direct apply_intervention, input validation, job pruning
# ---------------------------------------------------------------------------------------------------
def test_import_sees_the_testing_mode_of_its_turn(oracle_lib):
    """Interventions of one date are applied in list order (main.pyx:2012-2015) and import-infections infects at once
    (:1897-1899): the imported cases get an infectee list iff contact tracing was the mode when the import's turn came
    (person_infect, :227-233), not the mode the day ends with."""
    counts = helpers.small_population(6000)
    day = '2020-02-20'

    def run(order):
        ivs = [inputs.iv_tuple_to_obj(t) for t in order]
        ctx = helpers.make_context(oracle_lib, age_count_override=counts, seed=4, interventions=ivs, max_days=8)
        ctx.run(3)
        return ctx._plan[2], ctx._engine.read_agents(0)

    imp, ct, plain = ['import-infections', day, 30], ['test-with-contact-tracing', day, 50], ['test-all-with-symptoms', day]
    dp, ag = run([imp, ct])                      # imported BEFORE tracing starts: no lists, although the day ends in CT mode
    assert dp.import_traced == 0 and dp.testing_mode == model.ALL_WITH_SYMPTOMS_CT
    assert ((ag['state'] > 0).sum() >= 25) and not (ag['flags'][ag['state'] > 0] & 8).any()
    dp, ag = run([ct, imp])                      # tracing first: every imported case owns a list
    assert dp.import_traced == 1
    assert (ag['flags'][ag['state'] > 0] & 8).all()
    dp, ag = run([ct, imp, plain, ['import-infections', day, 10]])      # CT only for the first of two imports
    assert dp.import_traced == 0b01 and dp.n_imports == 2 and dp.testing_mode == model.ALL_WITH_SYMPTOMS
    n_list = int((ag['flags'][ag['state'] > 0] & 8).astype(bool).sum())
    assert 25 <= n_list <= 30 and (ag['state'] > 0).sum() >= n_list + 8


def test_direct_apply_intervention_takes_effect_from_today(oracle_lib):
    """apply_intervention is reference surface (calc/simulation.py:321) and acts immediately.  After reset() the plan
    already extends past today: a direct call must re-plan from today instead of being ignored, and a later
    add_intervention must not lose it."""
    counts = helpers.small_population(8000)
    imp = inputs.iv_tuple_to_obj(['import-infections', '2020-01-01', 40])        # its date is irrelevant for a direct call

    def infected_after(ctx, days):
        ctx.run(days)
        G = len(ctx.age_group_labels)
        return int(ctx.series(0, ctx.day)[0, -1, 3 * G:4 * G].sum())

    base = helpers.make_context(oracle_lib, age_count_override=counts, seed=6, interventions=[], max_days=40)
    assert infected_after(base, 12) == 0
    base.reset(6)                                    # plan of 12 days kept
    assert len(base._plan) == 12 and base.day == 0
    base.run(5)
    base.apply_intervention(imp)                     # day 5: must not be swallowed by the 7 days planned ahead
    assert len(base._plan) == 5
    got = infected_after(base, 6)
    assert got >= 35, got
    assert base._plan[5].n_imports == 1 and base._plan[5].import_amount[0] == 40
    base.add_intervention(inputs.iv_tuple_to_obj(['limit-mobility', '2020-03-01', 30]))     # re-plans; the direct call survives
    base.run(1)
    assert base._plan[5].n_imports == 1 and len(base._plan) == 12
    base.reset(9)                                    # a fresh run: the direct call belonged to the old one
    assert infected_after(base, 12) == 0
    with pytest.raises(Exception):
        base.apply_intervention(inputs.Intervention('no-such-intervention', '2020-01-01'))


def test_empty_contact_band_and_import_class_are_refused(oracle_lib):
    """A contact row / import class that can be drawn but holds nobody would take `x % 0` for the person index: both
    libraries refuse the input with an error instead (the reference would die with SIGFPE)."""
    counts = helpers.small_population(4000)
    counts[70:] = 0                                   # the whole 70+ band empty (every age has a row into it)
    counts[30] += 4000 - counts.sum()
    with pytest.raises(_abi.EngineError, match='empty'):
        helpers.make_context(oracle_lib, age_count_override=counts)
    counts = helpers.small_population(4000)
    counts[:20] = 0                                   # import class 0-19 (weight 15 %) empty; contact bands 0-4 ... 15-19 too
    counts[40] += 4000 - counts.sum()
    with pytest.raises(_abi.EngineError, match='empty'):
        helpers.make_context(oracle_lib, age_count_override=counts)


def test_serving_worker_forgets_old_jobs(oracle_lib):
    from reina_b200 import serving

    def factory(v, scenario):
        return helpers.make_context(oracle_lib, variables=v, scenario=scenario, seed=v['random_seed'],
                                    age_count_override=helpers.small_population(3000), max_days=v['simulation_days'] + 1)
    w = serving.SimulationWorker(context_factory=factory, callback_day_interval=5, max_finished_jobs=2)
    v = inputs.default_variables(simulation_days=6)
    jobs = [w.submit(dict(v, random_seed=s)) for s in range(4)]
    for j in jobs[2:]:
        assert w.wait(j, timeout=120)['finished']
    assert set(w._jobs) == set(jobs[2:])              # the two oldest finished jobs were dropped
    w.release(jobs[3])
    assert set(w._jobs) == {jobs[2]}
    with pytest.raises(KeyError):
        w.results(jobs[0])
    w.close()


# ---------------------------------------------------------------- the random blocks against Random123's known answers
def _py_philox4(k0, k1, c):
    M = 0xffffffff
    c0, c1, c2, c3 = c
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & M, p1 & M, ((p0 >> 32) ^ c3 ^ k1) & M, p0 & M
        k0, k1 = (k0 + 0x9E3779B9) & M, (k1 + 0xBB67AE85) & M
    return [c0, c1, c2, c3]


def test_random_blocks_match_random123_known_answers():
    """(e) of north_star: simrandom replaced by counter-based Philox.  The algorithm lives in no dependency of the
    reference (Random123, Salmon et al. 2011, is restated in rng.cuh / reina_oracle.c), so it is pinned here: the plain
    Python restatement below reproduces the published kat_vectors of philox4x32-10, and both libraries (host build of
    the very function the kernels inline) reproduce the restatement on the key layout the engine uses."""
    M = 0xffffffff
    assert _py_philox4(0, 0, (0, 0, 0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert _py_philox4(M, M, (M, M, M, M)) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert _py_philox4(0xa4093822, 0x299f31d0, (0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344)) == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    import ctypes as C
    rng = np.random.RandomState(5)
    for lib in (helpers.oracle_library(), _abi.Library(_abi.CUDA_LIB_PATH, 'rb_')):
        for _ in range(50):
            key = int(rng.randint(0, 2 ** 32, dtype=np.uint64))
            ctr = [int(v) for v in rng.randint(0, 2 ** 32, size=4, dtype=np.uint64)]
            cbuf, out = (C.c_uint32 * 4)(*ctr), (C.c_uint32 * 4)()
            assert lib.f['rng_block'](4, key, cbuf, out) == 0
            assert list(out) == _py_philox4(key, 0x5EEDB200, ctr)
        assert lib.f['rng_block'](2, 0, cbuf, out) != 0


def test_half_joined_engine_refuses_to_step():
    """A population-sharded join that fails half-way may already have changed an engine's ownership split (it would
    sweep only its stripes and still look like a whole population): such an engine must not step."""
    class FailingLib:
        f = {'shard_init': lambda *a: 1, 'shard_init_local': lambda *a: 1, 'step': lambda *a: 0}

        def check(self, rc, what):
            if rc:
                raise _abi.EngineError(what + ' failed')

    def fake_engine():
        e = object.__new__(_abi.Engine)
        e.lib, e.h, e.half_joined, e.rank, e.nranks = FailingLib(), None, False, 0, 1
        return e
    a = fake_engine()
    with pytest.raises(_abi.EngineError):
        a.shard_init(0, 2, b'x' * 128)
    with pytest.raises(_abi.EngineError, match='half-joined'):
        a.step(1)
    b, c = fake_engine(), fake_engine()
    b.step(1)                                   # a healthy engine steps
    with pytest.raises(_abi.EngineError):
        _abi.shard_init_local([b, c])
    for e in (b, c):
        with pytest.raises(_abi.EngineError, match='half-joined'):
            e.step(1)


def test_run_local_prepares_every_rank_before_any_launch():
    """sharded.run_local: planning, uploads and the schedule of ALL ranks first (they may synchronise with the device, and
    a rank that is already waiting for a peer occupies it), only then the launches, each on a thread of its own; an error
    on one rank's thread surfaces in the caller."""
    import threading
    from reina_b200 import sharded
    log, lock = [], threading.Lock()

    class FakeEngine:
        def sync(self):
            with lock:
                log.append('sync')

    class FakeCtx:
        def __init__(self, k, fail=False):
            self.k, self.fail, self._engine = k, fail, FakeEngine()

        def _prepare_run(self, days):
            with lock:
                log.append('prepare')

        def _launch_run(self, days):
            with lock:
                log.append('launch')
            if self.fail:
                raise model.SimulationFailed('Other failure')

        def _finish_run(self):
            with lock:
                log.append('finish')
    ctxs = [FakeCtx(k) for k in range(4)]
    sharded.run_local(ctxs, 7)
    assert log[:8] == ['prepare'] * 4 + ['sync'] * 4            # every rank prepared and idle ...
    assert sorted(log[8:]) == ['finish'] * 4 + ['launch'] * 4   # ... before the first launch
    del log[:]
    with pytest.raises(model.SimulationFailed):
        sharded.run_local([FakeCtx(0), FakeCtx(1, fail=True)], 3)
