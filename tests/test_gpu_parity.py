"""CUDA engine vs CPU oracle, bit-exact, through the C-ABI (the parity tests proper).

The oracle is the sequential restatement of the reference algorithm (oracle/reina_oracle.c); both sides get the
same seeded inputs, and every daily series, every agent field, the test queue and the free-capacity counters
must be IDENTICAL -- integer and index work, so the bar is bit-exact.
"""
import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu


def _pair(cuda_lib, oracle_lib, **kw):
    return helpers.make_context(cuda_lib, **kw), helpers.make_context(oracle_lib, **kw)


def _run_and_compare(gpu, cpu, days, chunk=None):
    chunk = chunk or days
    done = 0
    while done < days:
        n = min(chunk, days - done)
        gpu.run(n)
        cpu.run(n)
        done += n
    rep = helpers.diff_report(gpu, cpu, days)
    assert not rep, '\n'.join(rep)


@pytest.mark.parametrize('n_agents,seed', [(20000, 1), (120000, 2)])
def test_default_interventions_180_days(cuda_lib, oracle_lib, n_agents, seed):
    """HUS-shaped population, the reference's default intervention list (variables.py:366-412), hospital
    capacity scaled with the population so that ward and ICU saturate as they do at full size."""
    counts = helpers.small_population(n_agents)
    v = helpers.inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = helpers.scaled_capacity(n_agents)
    gpu, cpu = _pair(cuda_lib, oracle_lib, variables=v, age_count_override=counts, seed=seed)
    _run_and_compare(gpu, cpu, 180)
    last = gpu.series(0, 180)[0, -1]
    G = len(gpu.age_group_labels)
    assert last[3 * G:4 * G].sum() > n_agents * 0.05        # the epidemic actually happened


def test_every_intervention_type(cuda_lib, oracle_lib):
    """Imports of both variants, weekly trickle, all testing modes, contact tracing at 60/100/35 %, masks,
    mobility limits, three vaccination programme updates, capacity building, saturated tiny hospital."""
    counts = helpers.small_population(80000)
    v = helpers.inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = 25, 3
    ivs = helpers.stress_interventions()
    gpu, cpu = _pair(cuda_lib, oracle_lib, variables=v, age_count_override=counts, seed=11, interventions=ivs)
    _run_and_compare(gpu, cpu, 120, chunk=7)          # also exercises multi-call stepping
    G = len(gpu.age_group_labels)
    s = gpu.series(0, 120)[0]
    assert s[-1, 1 * G:2 * G].sum() > 0                # vaccinated
    assert s[:, 13 * G + 7].max() > 50                 # ct_cases_per_day
    assert s[:, 13 * G + 1].min() == 0                 # ward saturated (available beds hit 0)


def test_contact_tracing_scenario(cuda_lib, oracle_lib):
    """scenarios.py 'hammer-and-dance': contact tracing from day 73, efficiency 30 -> 60 %."""
    counts = helpers.small_population(150000)
    v = helpers.inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = helpers.scaled_capacity(150000)
    gpu, cpu = _pair(cuda_lib, oracle_lib, variables=v, age_count_override=counts, seed=5,
                     scenario='hammer-and-dance')
    _run_and_compare(gpu, cpu, 180)


@pytest.fixture
def wide_boundary(monkeypatch):
    """Every day boundary runs as a TEAM of CTAs joined by a grid barrier (boundary.cuh), whatever the day's load:
    the engine reads RB_WIDE_MIN / RB_WIDE_CTAS when it is created."""
    monkeypatch.setenv('RB_WIDE_MIN', '0')
    monkeypatch.setenv('RB_WIDE_CTAS', '8')


@pytest.mark.parametrize('case', ['stress', 'tracing', 'default', 'replicas'])
def test_wide_day_boundary(cuda_lib, oracle_lib, wide_boundary, case):
    """The multi-CTA day boundary (team sort, chained capacity scan, tracing over the whole team) against the oracle:
    every intervention type with a saturated tiny hospital, the contact-tracing scenario, the default run, and
    three replicas side by side."""
    v = helpers.inputs.default_variables()
    if case == 'stress':
        counts = helpers.small_population(80000)
        v['hospital_beds'], v['icu_units'] = 25, 3
        gpu, cpu = _pair(cuda_lib, oracle_lib, variables=v, age_count_override=counts, seed=11, interventions=helpers.stress_interventions())
        _run_and_compare(gpu, cpu, 120, chunk=7)
    elif case == 'tracing':
        counts = helpers.small_population(150000)
        v['hospital_beds'], v['icu_units'] = helpers.scaled_capacity(150000)
        gpu, cpu = _pair(cuda_lib, oracle_lib, variables=v, age_count_override=counts, seed=5, scenario='hammer-and-dance')
        _run_and_compare(gpu, cpu, 180)
    elif case == 'default':
        counts = helpers.small_population(120000)
        v['hospital_beds'], v['icu_units'] = helpers.scaled_capacity(120000)
        gpu, cpu = _pair(cuda_lib, oracle_lib, variables=v, age_count_override=counts, seed=2)
        _run_and_compare(gpu, cpu, 180)
    else:
        counts = helpers.small_population(30000)
        v['hospital_beds'], v['icu_units'] = helpers.scaled_capacity(30000)
        kw = dict(variables=v, age_count_override=counts, interventions=helpers.stress_interventions())
        gpu = helpers.make_context(cuda_lib, seed=40, n_replicas=3, **kw)
        gpu.run(100)
        rows = gpu.series(0, 100)
        for r in range(3):
            cpu = helpers.make_context(oracle_lib, seed=40 + r, **kw)
            cpu.run(100)
            assert np.array_equal(rows[r], cpu.series(0, 100)[0]), 'replica %d differs' % r
            assert np.array_equal(gpu._engine.read_agents(r), cpu._engine.read_agents(0))


def test_replicas_match_single_runs(cuda_lib, oracle_lib):
    """An R-replica context equals R single-seed runs (replica r uses seed + r)."""
    counts = helpers.small_population(30000)
    v = helpers.inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = helpers.scaled_capacity(30000)
    kw = dict(variables=v, age_count_override=counts)
    gpu = helpers.make_context(cuda_lib, seed=40, n_replicas=3, **kw)
    gpu.run(100)
    rows = gpu.series(0, 100)
    for r in range(3):
        cpu = helpers.make_context(oracle_lib, seed=40 + r, **kw)
        cpu.run(100)
        ref = cpu.series(0, 100)[0]
        mism = np.argwhere(rows[r] != ref)
        assert len(mism) == 0, 'replica %d differs first at (day, col) %s' % (r, mism[0])
        assert np.array_equal(gpu._engine.read_agents(r), cpu._engine.read_agents(0))


def test_edge_cases(cuda_lib, oracle_lib):
    """Tiny population, zero hospital capacity, empty age bands."""
    counts = helpers.small_population(3000)
    counts[90:] = 0
    counts[0] += 3000 - counts.sum()
    v = helpers.inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = 0, 0
    ivs = helpers.stress_interventions()
    gpu, cpu = _pair(cuda_lib, oracle_lib, variables=v, age_count_override=counts, seed=3, interventions=ivs)
    _run_and_compare(gpu, cpu, 90)


def test_per_day_api_matches_batched_run(cuda_lib):
    """iterate()/generate_state() one day at a time == run(n) (the reference's calling pattern,
    calc/simulation.py:194-270)."""
    counts = helpers.small_population(20000)
    a = helpers.make_context(cuda_lib, age_count_override=counts, seed=9)
    b = helpers.make_context(cuda_lib, age_count_override=counts, seed=9)
    states = []
    for _ in range(40):
        states.append(a.generate_state())
        a.iterate()
    b.run(40)
    rows = b.series(0, 40)[0]
    G = len(b.age_group_labels)
    for d, s in enumerate(states):
        for i, attr in enumerate(helpers._abi.ATTRS):
            assert np.array_equal(s[attr], rows[d, i * G:(i + 1) * G]), (d, attr)
    assert a.get_date_for_today() == '2020-03-29'


def test_sampler_parity(cuda_lib, oracle_lib):
    """Context.sample kinds (main.pyx:2047-2101): CUDA == oracle draw for draw."""
    counts = helpers.small_population(5000)
    gpu = helpers.make_context(cuda_lib, age_count_override=counts)
    cpu = helpers.make_context(oracle_lib, age_count_override=counts)
    for what in ('contacts_per_day', 'symptom_severity', 'incubation_period', 'illness_period',
                 'hospitalization_period', 'icu_period', 'onset_to_removed_period'):
        for age, sev in ((5, 'MILD'), (45, 'SEVERE'), (85, 'CRITICAL'), (70, 'FATAL')):
            assert np.array_equal(gpu.sample(what, age, sev), cpu.sample(what, age, sev)), (what, age, sev)


def test_checkpoint_resume(cuda_lib, oracle_lib):
    """save_state() in the middle of a run, load_state() into a fresh Context: the resumed run is bit-identical to
    the uninterrupted one (and to the oracle), stats rows of the days before the checkpoint included."""
    counts = helpers.small_population(60000)
    v = helpers.inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = 20, 2
    kw = dict(variables=v, age_count_override=counts, seed=21, interventions=helpers.stress_interventions(), n_replicas=2)
    a = helpers.make_context(cuda_lib, **kw)
    a.run(47)
    blob = a.save_state()
    a.run(43)
    b = helpers.make_context(cuda_lib, **kw)
    b.load_state(blob)
    assert b.day == 47 and b.get_date_for_today() == '2020-04-05'
    b.run(43)
    assert np.array_equal(a.series(0, 90), b.series(0, 90))
    for r in range(2):
        assert np.array_equal(a._engine.read_agents(r), b._engine.read_agents(r))
        # the queue is a set until contact tracing sorts it: entries are appended in scheduling order
        assert np.array_equal(np.sort(a._engine.read_queue(r)), np.sort(b._engine.read_queue(r)))
    cpu = helpers.make_context(oracle_lib, **dict(kw, n_replicas=1))
    cpu.run(90)
    assert np.array_equal(cpu.series(0, 90)[0], b.series(0, 90)[0])
    other = helpers.make_context(cuda_lib, **dict(kw, n_replicas=1))
    with pytest.raises(helpers._abi.EngineError):
        other.load_state(blob)                      # a blob of two replicas does not fit an engine of one


def test_initial_population_condition(cuda_lib, oracle_lib):
    """Population.set_initial_state (main.pyx:1452-1516): a run that starts from hospital figures of the case file and
    incubating / ill / recovered people -- drawn with replacement, quirks included -- CUDA == oracle bit for bit,
    replicas and reset() included; a tiny hospital makes the initial hospitalisations overflow."""
    counts = helpers.small_population(50000)
    v = helpers.inputs.default_variables()
    v.update(start_date='2020-04-01', incubating_at_simulation_start=400, ill_at_simulation_start=300,
             recovered_at_simulation_start=900)
    v['hospital_beds'], v['icu_units'] = 40, 20          # the case file has 52 in ward, 32 in ICU on that day
    kw = dict(variables=v, age_count_override=counts)
    one, ref = _pair(cuda_lib, oracle_lib, seed=77, **kw)
    _run_and_compare(one, ref, 45)                        # reports the first differing series / agent field
    gpu = helpers.make_context(cuda_lib, seed=77, n_replicas=2, **kw)
    s0 = gpu.generate_state()
    assert s0['all_infected'].sum() == 9 + 32 + 52 + 400 + 300 + 900 and s0['available_hospital_beds'] < 40
    gpu.run(60)
    rows = gpu.series(0, 60)
    for r in range(2):
        cpu = helpers.make_context(oracle_lib, seed=77 + r, **kw)
        cpu.run(60)
        assert np.array_equal(rows[r], cpu.series(0, 60)[0]), 'replica %d' % r
        assert np.array_equal(gpu._engine.read_agents(r), cpu._engine.read_agents(0))
    gpu.reset(500)                                        # a fresh ensemble starts from the same condition
    gpu.run(30)
    cpu = helpers.make_context(oracle_lib, seed=500, **kw)
    cpu.run(30)
    assert np.array_equal(gpu.series(0, 30)[0], cpu.series(0, 30)[0])
