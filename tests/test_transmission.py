"""Transmission statistics (rb_transmission_stats / rb_read_infection_days, Context.transmission_stats / transmission_tree,
ensemble.transmission_summary): who infected whom and when.

CPU: the oracle's tables equal a numpy restatement from the line list, cell for cell; the tables' invariants; the summary
formulas; two gloo ranks summarise like one process.  GPU: the CUDA tables equal the oracle's at the bench geometry (full
HUS, 256 replicas, 180 days) and on the every-intervention schedule, survive save / load and reset, and are the same on
every rank of a population-sharded run.

The CPU reference is tests/oracle_transmission.c: the sequential oracle, unchanged, plus the three entry points as plain
loops, compiled here into a library of its own (in the temporary directory, keyed by the hash of its sources)."""
import hashlib
import multiprocessing
import os
import socket
import subprocess
import sys
import tempfile
import traceback
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

import helpers
from reina_b200 import _abi, ensemble

TABLES = ('cohort_infected', 'cohort_offspring', 'cohort_open', 'offspring_hist', 'generation_interval_hist',
          'group_closed', 'group_offspring', 'variant_closed', 'variant_offspring')
INITIAL_STATE = dict(start_date='2020-04-01', incubating_at_simulation_start=400, ill_at_simulation_start=300,
                     recovered_at_simulation_start=900)


_tx_oracle = None


def tx_oracle_library():
    """The CPU oracle with the transmission entry points (tests/oracle_transmission.c), built once per source state."""
    global _tx_oracle
    if _tx_oracle is None:
        srcs = [os.path.join(helpers.ROOT, *p) for p in (('tests', 'oracle_transmission.c'), ('oracle', 'reina_oracle.c'),
                                                        ('include', 'reina_b200.h'))]
        key = hashlib.sha1(b''.join(open(f, 'rb').read() for f in srcs)).hexdigest()[:16]
        lib = os.path.join(tempfile.gettempdir(), 'reina_tx_oracle_%d_%s.so' % (os.getuid(), key))
        if not os.path.exists(lib):
            tmp = '%s.%d.tmp' % (lib, os.getpid())
            # the flags of oracle/Makefile: float ops must round like the CUDA engine's -fmad=false
            subprocess.run([os.environ.get('CC', 'gcc'), '-O2', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math',
                            '-shared', '-o', tmp, srcs[0], '-lm'], check=True)
            os.replace(tmp, lib)
        _tx_oracle = _abi.Library(lib, 'ro_')
        _tx_oracle.bind_transmission()
    return _tx_oracle


@pytest.fixture(scope='module')
def tx_oracle():
    return tx_oracle_library()


def restate(ctx, r):
    """The tables of replica r recomputed in numpy from the line list and the agent records."""
    tree = ctx.transmission_tree(r)
    ag = ctx._engine.read_agents(r)
    a, d, inf = tree['agent'], tree['day'], tree['infector']
    o, st, var = ag['n_infected'][a].astype(np.int64), ag['state'][a], ag['variant'][a]
    M, B, G, V = ctx.day + 1, _abi.RB_TX_BINS, len(ctx.age_group_labels), len(ctx.variant_names)
    opn = (st == 1) | (st == 2)                     # INCUBATION, ILLNESS
    closed = ~opn
    day_of = np.full(ctx.n_agents, -1, dtype=np.int64)
    day_of[a] = d
    child = inf >= 0
    g = ctx._group_of_age[tree['age'][closed]]
    cnt = lambda x, n, w=None: np.bincount(x, weights=w, minlength=n).astype(np.int64)
    return dict(cohort_infected=cnt(d, M), cohort_offspring=cnt(d, M, o), cohort_open=cnt(d[opn], M),
                offspring_hist=cnt(np.minimum(o[closed], B - 1), B),
                generation_interval_hist=cnt(np.clip(d[child] - day_of[inf[child]], 0, B - 1), B),
                group_closed=cnt(g, G), group_offspring=cnt(g, G, o[closed]),
                variant_closed=cnt(var[closed], V), variant_offspring=cnt(var[closed], V, o[closed]))


def check_invariants(t, r, n_children=None, initial_state=False):
    row = {k: t[k][r] for k in TABLES}
    closed = (row['cohort_infected'] - row['cohort_open']).sum()
    assert row['cohort_offspring'].sum() == row['generation_interval_hist'].sum(), r
    assert row['offspring_hist'].sum() == row['group_closed'].sum() == row['variant_closed'].sum() == closed, r
    assert row['group_offspring'].sum() == row['variant_offspring'].sum(), r
    if not initial_state:      # only the initial state's ill agents, infected on day 0, infect others on day 0
        assert row['generation_interval_hist'][0] == 0, r
    if n_children is not None:
        assert row['cohort_offspring'].sum() == n_children, r


def all_infected_today(ctx):
    ctx.generate_state()
    G = len(ctx.age_group_labels)
    return ctx._engine.read_stats(ctx.day, 1)[:, 0, 3 * G:4 * G].sum(axis=1)


def stress_kw(n_agents=80000):
    v = helpers.inputs.default_variables()
    v['hospital_beds'], v['icu_units'] = 25, 3
    return dict(variables=v, age_count_override=helpers.small_population(n_agents), interventions=helpers.stress_interventions())


def initial_state_kw(n_agents=50000):
    v = helpers.inputs.default_variables()
    v.update(INITIAL_STATE)
    v['hospital_beds'], v['icu_units'] = 40, 20
    return dict(variables=v, age_count_override=helpers.small_population(n_agents))


# ---------------------------------------------------------------- CPU (oracle)
@pytest.mark.parametrize('case', ['stress', 'initial_state'])
def test_oracle_tables_equal_restatement(tx_oracle, case):
    kw = stress_kw() if case == 'stress' else initial_state_kw()
    ctx = helpers.make_context(tx_oracle, seed=11, n_replicas=4, max_days=130, **kw)
    ctx.run(120)
    t = ctx.transmission_stats()
    assert set(t) == set(TABLES)
    assert t['cohort_infected'].shape == (4, 121) and t['variant_closed'].shape == (4, len(ctx.variant_names))
    assert t['offspring_hist'].shape == (4, _abi.RB_TX_BINS) and t['group_closed'].shape == (4, len(ctx.age_group_labels))
    totals = all_infected_today(ctx)
    for r in range(4):
        ref = restate(ctx, r)
        for k in TABLES:
            assert np.array_equal(t[k][r], ref[k]), (case, r, k)
        check_invariants(t, r, int((ctx._engine.read_agents(r)['infector'] >= 0).sum()), case == 'initial_state')
        if case == 'stress':       # an initial state counts a person drawn twice twice in all_infected
            assert t['cohort_infected'][r].sum() == totals[r], r
        else:
            assert t['cohort_infected'][r, 0] > 1000     # the initial state is infected on day 0
    if case == 'stress':
        assert t['variant_closed'][:, 1].sum() > 0       # the second variant spread
    # recent cohorts can still infect, early ones are complete; today's cohort is empty until today is simulated
    assert t['cohort_open'][:, -10:].sum() > 0 and t['cohort_open'][:, :20].sum() == 0
    assert t['cohort_infected'][:, -1].sum() == 0


def test_infection_days_of_roots(tx_oracle):
    """Imports and initial-state draws carry the day they happened, children the day of their transmission."""
    ctx = helpers.make_context(tx_oracle, seed=3, max_days=70, **initial_state_kw(20000))
    ctx.run(60)
    tree = ctx.transmission_tree(0)
    roots = tree['infector'] < 0
    assert roots.sum() > 1000 and (tree['day'][roots] == 0).all()      # no imports after 2020-04-01 in the defaults
    assert np.array_equal(np.flatnonzero(ctx._engine.read_infection_days(0) >= 0), tree['agent'])
    assert np.array_equal(tree['age'], np.searchsorted(ctx._age_start, tree['agent'], side='right') - 1)
    kw = stress_kw(20000)
    ctx = helpers.make_context(tx_oracle, seed=3, max_days=70, **kw)
    ctx.run(60)
    tree = ctx.transmission_tree(0)
    roots = np.unique(tree['day'][tree['infector'] < 0])
    # 'import-infections' on 2020-02-18 (day 0) and 2020-03-10 (day 21), the weekly trickle from 2020-02-21 (day 3) on
    assert {0, 3, 21} <= set(roots.tolist()) and roots.max() > 50
    child = tree['infector'] >= 0
    days = ctx._engine.read_infection_days(0)
    assert (tree['day'][child] > days[tree['infector'][child]]).all()


def _hand_built():
    n = np.array([[10, 0, 4], [20, 0, 6], [30, 0, 0]])
    off = np.array([[15, 0, 2], [22, 0, 9], [51, 0, 0]])
    return dict(cohort_infected=n, cohort_offspring=off, cohort_open=np.array([[0, 0, 1], [0, 0, 0], [0, 0, 0]]),
                offspring_hist=np.array([[3, 1, 0, 2], [1, 0, 0, 0], [0, 1, 1, 0]]),
                generation_interval_hist=np.array([[0, 2, 3, 0], [0, 0, 1, 0], [0, 1, 1, 1]]),
                group_closed=np.array([[2, 4], [1, 0], [0, 2]]), group_offspring=np.array([[1, 6], [0, 0], [0, 3]]),
                variant_closed=np.array([[6], [1], [2]]), variant_offspring=np.array([[7], [0], [3]]))


def test_summary_formulas():
    s = ensemble.transmission_summary(_hand_built())
    K = 3
    n = np.array([10, 20, 30.])
    off = np.array([15, 22, 51.])
    R = off.sum() / n.sum()
    se = np.sqrt(((off - R * n) ** 2).sum() / ((n.sum() / K) ** 2 * K * (K - 1)))
    assert s['n_replicas'] == 3
    np.testing.assert_allclose(s['cohort_R'][0], R, rtol=1e-14)
    np.testing.assert_allclose(s['cohort_R_se'][0], se, rtol=1e-12)
    assert np.isnan(s['cohort_R'][1]) and np.isnan(s['cohort_R_se'][1])
    np.testing.assert_allclose(s['cohort_R'][2], 11 / 10)
    assert s['complete'].tolist() == [True, True, False]
    x = np.repeat(np.arange(4), [4, 2, 1, 2])              # closed cases' offspring counts
    assert s['offspring_mean'] == pytest.approx(x.mean()) and s['offspring_var'] == pytest.approx(x.var(ddof=1))
    m, v = x.mean(), x.var(ddof=1)
    assert s['dispersion_k'] == pytest.approx(m * m / (v - m))
    np.testing.assert_allclose(s['gi_pmf'], np.array([0, 3, 5, 1]) / 9)
    assert s['gi_mean'] == pytest.approx((3 + 10 + 3) / 9)
    np.testing.assert_allclose(s['R_by_group'], [1 / 3, 9 / 6])
    np.testing.assert_allclose(s['R_by_variant'], [10 / 9])
    # no overdispersion: k is infinite
    eq = dict(_hand_built(), offspring_hist=np.array([[0, 5, 0, 0], [0, 5, 0, 0], [0, 5, 0, 0]]))
    assert ensemble.transmission_summary(eq)['dispersion_k'] == np.inf


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_make(n_replicas, seed):
    return helpers.make_context(tx_oracle_library(), age_count_override=helpers.small_population(4000),
                                seed=seed, n_replicas=n_replicas, max_days=64)


def _gloo_worker(rank, world, port, out_dir):
    sys.path.insert(0, os.path.join(helpers.ROOT, 'tests'))
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    ctx = _gloo_make(2, ensemble.seeds_for_rank(300, 2, rank))
    ctx.run(50)
    s = ensemble.transmission_summary(ctx.transmission_stats(), helpers.TorchComm(dist))
    np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), **{k: np.asarray(v) for k, v in s.items()})
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_summary_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_gloo_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / 'rank0.npz'), np.load(tmp_path / 'rank1.npz')
    ctx = _gloo_make(4, 300)                  # seeds 300..303 = rank 0 (300, 301) + rank 1 (302, 303)
    ctx.run(50)
    one = ensemble.transmission_summary(ctx.transmission_stats())
    assert int(r0['n_replicas']) == 4 and np.nansum(one['cohort_infected']) > 0
    for k, v in one.items():
        np.testing.assert_allclose(r0[k], v, rtol=1e-12, equal_nan=True, err_msg=k)
        np.testing.assert_array_equal(r0[k], r1[k], err_msg=k)


# ---------------------------------------------------------------- GPU
def _oracle_full_hus(args):
    scenario, variables, seed = args
    ctx = helpers.make_context(tx_oracle_library(), area='HUS', scenario=scenario, seed=seed, max_days=181, variables=variables)
    ctx.run(180)
    return ctx.transmission_stats(), ctx._engine.read_infection_days(0)


@pytest.mark.gpu
@pytest.mark.parametrize('scenario,initial', [(None, False), ('hammer-and-dance', False), (None, True)])
def test_full_hus_256_replicas_equal_oracle(cuda_lib, scenario, initial):
    """The bench geometry: full HUS, 256 replicas, 180 days.  Replicas 0 and 255 against the oracle with the same seeds,
    every replica against the invariants."""
    variables = None
    if initial:
        from test_oracle_pinned import INITIAL_STATE_VARIABLES
        variables = helpers.inputs.default_variables()
        variables.update(INITIAL_STATE_VARIABLES)
    seed = 515151
    gpu = helpers.make_context(cuda_lib, area='HUS', scenario=scenario, seed=seed, n_replicas=256, max_days=181, variables=variables)
    gpu.run(180)
    t = gpu.transmission_stats()
    days = {r: gpu._engine.read_infection_days(r) for r in (0, 255)}
    totals = all_infected_today(gpu)
    gpu.close()
    with ProcessPoolExecutor(2, mp_context=multiprocessing.get_context('spawn')) as ex:
        ref = dict(zip((0, 255), ex.map(_oracle_full_hus, [(scenario, variables, seed + r) for r in (0, 255)])))
    for r in (0, 255):
        for k in TABLES:
            assert np.array_equal(t[k][r], ref[r][0][k][0]), (scenario, initial, r, k)
        assert np.array_equal(days[r], ref[r][1]), (scenario, initial, r)
    for r in range(256):
        check_invariants(t, r, initial_state=initial)
        if not initial:
            assert t['cohort_infected'][r].sum() == totals[r], r
    assert t['cohort_infected'].sum() > 256 * 100000          # the epidemic happened


@pytest.mark.gpu
def test_every_intervention_type_equal_oracle(cuda_lib, tx_oracle):
    """Both variants, vaccination, contact tracing and a saturated hospital, three replicas side by side."""
    kw = stress_kw()
    gpu = helpers.make_context(cuda_lib, seed=11, n_replicas=3, max_days=130, **kw)
    for _ in range(4):
        gpu.run(30)
    t = gpu.transmission_stats()
    for r in range(3):
        cpu = helpers.make_context(tx_oracle, seed=11 + r, max_days=130, **kw)
        cpu.run(120)
        c = cpu.transmission_stats()
        for k in TABLES:
            assert np.array_equal(t[k][r], c[k][0]), (r, k)
        assert np.array_equal(gpu._engine.read_infection_days(r), cpu._engine.read_infection_days(0)), r
        tree, ctree = gpu.transmission_tree(r), cpu.transmission_tree(0)
        assert all(np.array_equal(tree[k], ctree[k]) for k in tree), r
        check_invariants(t, r, int((gpu._engine.read_agents(r)['infector'] >= 0).sum()))
    assert t['variant_closed'][:, 1].sum() > 0


@pytest.mark.gpu
def test_tables_survive_save_load_and_reset(cuda_lib):
    kw = dict(stress_kw(60000), seed=21, n_replicas=2, max_days=100)
    a = helpers.make_context(cuda_lib, **kw)
    a.run(47)
    blob, t47 = a.save_state(), a.transmission_stats()
    b = helpers.make_context(cuda_lib, **kw)
    b.load_state(blob)
    tb = b.transmission_stats()
    assert all(np.array_equal(t47[k], tb[k]) for k in TABLES)
    a.run(43)
    b.run(43)
    t90 = a.transmission_stats()
    tb = b.transmission_stats()
    assert all(np.array_equal(t90[k], tb[k]) for k in TABLES)
    a.reset(21)                                 # the sparse reset, then the same run again
    assert a.transmission_stats()['cohort_infected'].sum() == 0
    a.run(90)
    ta = a.transmission_stats()
    assert all(np.array_equal(t90[k], ta[k]) for k in TABLES)
    assert np.array_equal(a._engine.read_infection_days(1), b._engine.read_infection_days(1))


def _local_worker(world, chunk, q):
    try:
        from reina_b200 import sharded
        kw = dict(stress_kw(), seed=11, max_days=130)
        ctxs = [helpers.make_context(helpers.cuda_library(), device=0, **kw) for _ in range(world)]
        sharded.join_local(ctxs)
        done = 0
        while done < 120:
            n = min(chunk, 120 - done)
            sharded.run_local(ctxs, n)
            done += n
        q.put([(c.transmission_stats(), c._engine.read_infection_days(0)) for c in ctxs])
    except Exception:
        q.put(traceback.format_exc())


@pytest.mark.gpu
@pytest.mark.parametrize('world', [2, 4])
def test_local_ranks_on_one_gpu(cuda_lib, tx_oracle, monkeypatch, world):
    """Population-sharded mode (several ranks on one GPU, as tests/test_gpu_sharded.py runs them): every rank returns the
    tables and infection days of the single-engine run."""
    monkeypatch.setenv('CUDA_DEVICE_MAX_CONNECTIONS', '32')
    monkeypatch.setenv('CUDA_MODULE_LOADING', 'EAGER')
    mpc = multiprocessing.get_context('spawn')
    q = mpc.Queue()
    p = mpc.Process(target=_local_worker, args=(world, 31, q))
    p.start()
    try:
        out = q.get(timeout=300)
    finally:
        p.join(timeout=30)
        if p.is_alive():
            p.kill()
    assert not isinstance(out, str), 'local ranks failed:\n%s' % out
    ref = helpers.make_context(tx_oracle, **dict(stress_kw(), seed=11, max_days=130))
    ref.run(120)
    t, days = ref.transmission_stats(), ref._engine.read_infection_days(0)
    for rank, (tr, dr) in enumerate(out):
        for k in TABLES:
            assert np.array_equal(tr[k], t[k]), (rank, k)
        assert np.array_equal(dr, days), rank
