"""Transmission by setting and age (rb_transmission_settings / rb_read_infection_places, Context.transmission_settings /
infection_places, ensemble.setting_summary): where infections happened and who infected whom.

CPU: the oracle's tables equal a numpy restatement from the line list, cell for cell, and agree with the transmission
statistics of the same state; a school closure leaves no school infection; the summary formulas; two gloo ranks summarise
like one process.  GPU: the CUDA tables and per-agent places equal the oracle's at the bench geometry (full HUS, 256
replicas, 180 days) and on the every-intervention schedule, survive save / load and reset, and are the same on every rank
of a population-sharded run.

The CPU reference is tests/oracle_settings.c over an instrumented copy of the sequential oracle: the copy made here adds
one write-only field to the oracle's Agent, set where the oracle infects (person_infect: a root; right after
person_expose_others' person_infect call: the place of the contact row its own scan picked).  oracle/ itself stays as it
is.  The copy, tests/oracle_transmission.c, tests/oracle_settings.c and the header are compiled into a library of its own
in the temporary directory, keyed by the hash of the sources."""
import hashlib
import multiprocessing
import os
import shutil
import subprocess
import sys
import tempfile
import traceback
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

import helpers
from reina_b200 import _abi, ensemble
from reina_b200.model import Context
from test_transmission import _free_port, initial_state_kw, stress_kw

SETTINGS = ('by_day_place', 'pair_all', 'pair_closed', 'closed_by_group')
P = _abi.RB_N_PLACES
SCHOOL = Context.PLACE_NAMES.index('school')

# (anchor in oracle/reina_oracle.c, line inserted after it): the place of every infection, observed where it happens
ORACLE_PROBES = [
    ('    uint8_t ward_days, icu_days;\n', '    uint8_t infection_place;   /* test build: RB_PLACE_ROOT or the contact row\'s place */\n'),
    ('    t->day_of_infection = (int16_t)e->day;\n', '    t->infection_place = RB_PLACE_ROOT;\n'),
    ('        person_infect(e, r, ti, ai, -1, slot);\n', '        t->infection_place = tb->place[p->age][row];\n'),
]

_sx_oracle = None


def sx_oracle_library():
    """The oracle with the probes above plus the transmission and settings entry points, built once per source state."""
    global _sx_oracle
    if _sx_oracle is None:
        files = [('oracle', 'reina_oracle.c'), ('tests', 'oracle_transmission.c'), ('tests', 'oracle_settings.c'),
                 ('include', 'reina_b200.h')]
        src = {f: open(os.path.join(helpers.ROOT, *f), 'rb').read().decode() for f in files}
        key = hashlib.sha1(''.join(src[f] for f in files).encode() + repr(ORACLE_PROBES).encode()).hexdigest()[:16]
        lib = os.path.join(tempfile.gettempdir(), 'reina_sx_oracle_%d_%s.so' % (os.getuid(), key))
        if not os.path.exists(lib):
            text = src[('oracle', 'reina_oracle.c')]
            for anchor, line in ORACLE_PROBES:
                assert text.count(anchor) == 1, 'oracle probe anchor not found exactly once: %r' % anchor
                text = text.replace(anchor, anchor + line)
            src[('oracle', 'reina_oracle.c')] = text
            tree = tempfile.mkdtemp(prefix='reina_sx_oracle_')
            try:
                for f in files:
                    os.makedirs(os.path.join(tree, f[0]), exist_ok=True)
                    with open(os.path.join(tree, *f), 'w') as fh:
                        fh.write(src[f])
                tmp = '%s.%d.tmp' % (lib, os.getpid())
                # the flags of oracle/Makefile: float ops must round like the CUDA engine's -fmad=false
                subprocess.run([os.environ.get('CC', 'gcc'), '-O2', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math',
                                '-shared', '-o', tmp, os.path.join(tree, 'tests', 'oracle_settings.c'), '-lm'], check=True)
                os.replace(tmp, lib)
            finally:
                shutil.rmtree(tree, ignore_errors=True)
        _sx_oracle = _abi.Library(lib, 'ro_')
        _sx_oracle.bind_transmission()
        _sx_oracle.bind_settings()
    return _sx_oracle


@pytest.fixture(scope='module')
def sx_oracle():
    return sx_oracle_library()


def restate(ctx, r):
    """The settings tables of replica r recomputed in numpy from the line list, the places and the agents' states."""
    tree, place = ctx.transmission_tree(r), ctx.infection_places(r)
    st = ctx._engine.read_agents(r)['state']
    a, inf, d = tree['agent'], tree['infector'], tree['day']
    G = len(ctx.age_group_labels)
    closed = lambda s: (s != 1) & (s != 2)          # neither INCUBATION nor ILLNESS
    cg = ctx._group_of_age[tree['age']]
    ch = inf >= 0
    ig = ctx._group_of_age[np.searchsorted(ctx._age_start, inf[ch], side='right') - 1]
    cell = (place[ch] * G + ig) * G + cg[ch]
    cnt = lambda x, n: np.bincount(x, minlength=n).astype(np.int64)
    return dict(by_day_place=cnt(d * (P + 1) + place, (ctx.day + 1) * (P + 1)).reshape(ctx.day + 1, P + 1),
                pair_all=cnt(cell, P * G * G).reshape(P, G, G),
                pair_closed=cnt(cell[closed(st[inf[ch]])], P * G * G).reshape(P, G, G),
                closed_by_group=cnt(cg[closed(st[a])], G))


def check_invariants(s, t, r, n_children=None):
    """Against the transmission statistics of the same state."""
    bdp = s['by_day_place'][r]
    assert bdp[:, :P].sum() == s['pair_all'][r].sum() >= s['pair_closed'][r].sum(), r
    if n_children is not None:
        assert bdp[:, :P].sum() == n_children, r
    assert np.array_equal(bdp.sum(axis=1), t['cohort_infected'][r]), r
    assert np.array_equal(s['pair_closed'][r].sum(axis=(0, 2)), t['group_offspring'][r]), r
    assert np.array_equal(s['closed_by_group'][r], t['group_closed'][r]), r


def school_kw(n_agents=80000):
    v = helpers.inputs.default_variables()
    ivs = [['import-infections', '2020-02-18', 300], ['limit-mobility', '2020-03-14', 100, None, None, 'school']]
    return dict(variables=v, age_count_override=helpers.small_population(n_agents),
                interventions=[helpers.inputs.iv_tuple_to_obj(t) for t in ivs])


def check_school_closure(ctx, s):
    """No school infection on a day whose contact table has no school contact left, some before."""
    def school_mass(t):
        rows = t['place'][:, :t['n_rows'][0]] == SCHOOL
        p = np.diff(np.concatenate([np.zeros((t['cum_p'].shape[0], 1)), t['cum_p'][:, :t['n_rows'][0]]], axis=1), axis=1)
        return p[rows].sum()
    epochs = ctx._epoch_of_day()
    shut = np.array([school_mass(ctx._tables[e]) == 0 for e in epochs])
    assert shut.any() and not shut[0] and shut[shut.argmax():].all()
    school = s['by_day_place'][:, :ctx.day, SCHOOL]
    assert school[:, shut].sum() == 0
    assert school[:, ~shut].sum() > 0


# ---------------------------------------------------------------- CPU (oracle)
@pytest.mark.parametrize('case', ['stress', 'initial_state'])
def test_oracle_tables_equal_restatement(sx_oracle, case):
    kw = stress_kw() if case == 'stress' else initial_state_kw()
    ctx = helpers.make_context(sx_oracle, seed=11, n_replicas=4, max_days=130, **kw)
    ctx.run(120)
    s, t = ctx.transmission_settings(), ctx.transmission_stats()
    G = len(ctx.age_group_labels)
    assert set(s) == set(SETTINGS)
    assert s['by_day_place'].shape == (4, 121, P + 1) and s['pair_all'].shape == (4, P, G, G)
    assert s['pair_closed'].shape == (4, P, G, G) and s['closed_by_group'].shape == (4, G)
    for r in range(4):
        ref = restate(ctx, r)
        for k in SETTINGS:
            assert np.array_equal(s[k][r], ref[k]), (case, r, k)
        tree = ctx.transmission_tree(r)
        assert ctx.infection_places(r).shape == tree['agent'].shape
        assert (ctx.infection_places(r)[tree['infector'] < 0] == _abi.RB_PLACE_ROOT).all()
        check_invariants(s, t, r, int((tree['infector'] >= 0).sum()))
    # infections happened in every place the stress schedule leaves open, and the roots are where they belong
    assert (s['pair_all'].sum(axis=(0, 2, 3)) > 0).all()
    if case == 'initial_state':
        assert s['by_day_place'][:, 0, _abi.RB_PLACE_ROOT].min() > 1000
    else:
        assert s['by_day_place'][:, 21, _abi.RB_PLACE_ROOT].min() >= 90      # the 100 imports of 2020-03-10


def test_oracle_checks_the_epochs(sx_oracle):
    """The epochs given must be those the run used, one per completed day."""
    ctx = helpers.make_context(sx_oracle, seed=5, max_days=40, **stress_kw(20000))
    ctx.run(30)
    ep = ctx._epoch_of_day()
    assert len(set(ep.tolist())) > 2
    ctx._engine.transmission_settings(ep)
    for bad in (ep[:-1], np.concatenate([ep, ep[-1:]]), np.where(np.arange(ep.size) == 20, ep + 1, ep)):
        with pytest.raises(_abi.EngineError):
            ctx._engine.transmission_settings(bad)
        with pytest.raises(_abi.EngineError):
            ctx._engine.read_infection_places(0, bad)


def test_school_closure_oracle(sx_oracle):
    ctx = helpers.make_context(sx_oracle, seed=8, n_replicas=2, max_days=70, **school_kw())
    ctx.run(60)
    check_school_closure(ctx, ctx.transmission_settings())


def _hand_built():
    """3 replicas, 2 days, 2 age groups."""
    bdp = np.zeros((3, 2, P + 1), dtype=np.int64)
    bdp[:, 0, P] = [5, 4, 6]
    bdp[0, 1, :P] = [4, 2, 1, 0, 3, 0]
    bdp[1, 1, :P] = [6, 1, 0, 0, 1, 2]
    bdp[2, 1, :P] = [2, 2, 2, 1, 1, 0]
    pc = np.zeros((3, P, 2, 2), dtype=np.int64)
    # ngm_by_place[0] = [[1, .5], [.5, 1]], ngm_by_place[1] = [[.2, .1], [.1, .2]] with 10 closed cases per group
    pc[0, 0] = [[6, 1], [2, 4]]
    pc[1, 0] = [[4, 4], [3, 6]]
    pc[0, 1] = [[2, 1], [1, 2]]
    closed = np.array([[4, 5], [6, 5], [0, 0]])
    return dict(by_day_place=bdp, pair_all=pc + 1, pair_closed=pc, closed_by_group=closed)


def test_summary_formulas():
    h = _hand_built()
    s = ensemble.setting_summary(h)
    K = 3
    x = h['by_day_place'][:, :, :P].sum(axis=1).astype(np.float64)
    c = x.sum(axis=1)
    share = x.sum(0) / c.sum()
    se = np.array([np.sqrt(((x[:, p] - share[p] * c) ** 2).sum() / ((c.sum() / K) ** 2 * K * (K - 1))) for p in range(P)])
    assert s['n_replicas'] == 3
    np.testing.assert_allclose(s['share'], share, rtol=1e-14)
    np.testing.assert_allclose(s['share_se'], se, rtol=1e-12)
    assert s['share'].sum() == pytest.approx(1.0)
    np.testing.assert_allclose(s['incidence_by_place_mean'], h['by_day_place'].mean(axis=0))
    np.testing.assert_allclose(s['incidence_by_place_std'], h['by_day_place'].std(axis=0, ddof=1))
    np.testing.assert_array_equal(s['waifw'], (h['pair_all']).sum(axis=(0, 1)))
    np.testing.assert_allclose(s['ngm_by_place'][0], [[1, .5], [.5, 1]])
    np.testing.assert_allclose(s['ngm_by_place'][1], [[.2, .1], [.1, .2]])
    np.testing.assert_allclose(s['ngm'], [[1.2, .6], [.6, 1.2]])
    np.testing.assert_allclose(s['R_by_place'], [1.5, .3, 0, 0, 0, 0])
    # eigenvalues of [[a, b], [b, a]] are a +- b
    assert s['rho'] == pytest.approx(1.8)
    np.testing.assert_allclose(s['rho_without'], [.3, 1.5, 1.8, 1.8, 1.8, 1.8])
    # orientation: infections by group 0 of group 1 are the column of group 0; a group without closed cases is NaN
    one = dict(by_day_place=h['by_day_place'][:1], pair_all=h['pair_all'][:1], closed_by_group=np.array([[8, 0]]),
               pair_closed=np.zeros((1, P, 2, 2), dtype=np.int64))
    one['pair_closed'][0, 2, 0, 1] = 4
    s1 = ensemble.setting_summary(one)
    assert s1['ngm'][1, 0] == 0.5 and s1['ngm'][0, 0] == 0 and np.isnan(s1['ngm'][:, 1]).all()
    assert s1['rho'] == 0.0 and np.isnan(s1['share_se']).all()
    np.testing.assert_allclose(s1['R_by_place'], [0, 0, .5, 0, 0, 0])


def _gloo_make(n_replicas, seed):
    return helpers.make_context(sx_oracle_library(), age_count_override=helpers.small_population(4000),
                                seed=seed, n_replicas=n_replicas, max_days=64)


def _gloo_worker(rank, world, port, out_dir):
    sys.path.insert(0, os.path.join(helpers.ROOT, 'tests'))
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    ctx = _gloo_make(2, ensemble.seeds_for_rank(300, 2, rank))
    ctx.run(50)
    s = ensemble.setting_summary(ctx.transmission_settings(), helpers.TorchComm(dist))
    np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), **{k: np.asarray(v) for k, v in s.items()})
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_summary_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_gloo_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / 'rank0.npz'), np.load(tmp_path / 'rank1.npz')
    ctx = _gloo_make(4, 300)                  # seeds 300..303 = rank 0 (300, 301) + rank 1 (302, 303)
    ctx.run(50)
    one = ensemble.setting_summary(ctx.transmission_settings())
    assert int(r0['n_replicas']) == 4 and one['pair_all'].sum() > 0
    for k, v in one.items():
        np.testing.assert_allclose(r0[k], v, rtol=1e-12, equal_nan=True, err_msg=k)
        np.testing.assert_array_equal(r0[k], r1[k], err_msg=k)


# ---------------------------------------------------------------- GPU
def _oracle_full_hus(args):
    scenario, variables, seed = args
    ctx = helpers.make_context(sx_oracle_library(), area='HUS', scenario=scenario, seed=seed, max_days=181, variables=variables)
    ctx.run(180)
    return ctx.transmission_settings(), ctx.infection_places(0)


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
    s, t = gpu.transmission_settings(), gpu.transmission_stats()
    places = {r: gpu.infection_places(r) for r in (0, 255)}
    gpu.close()
    with ProcessPoolExecutor(2, mp_context=multiprocessing.get_context('spawn')) as ex:
        ref = dict(zip((0, 255), ex.map(_oracle_full_hus, [(scenario, variables, seed + r) for r in (0, 255)])))
    for r in (0, 255):
        for k in SETTINGS:
            assert np.array_equal(s[k][r], ref[r][0][k][0]), (scenario, initial, r, k)
        assert np.array_equal(places[r], ref[r][1]), (scenario, initial, r)
    for r in range(256):
        check_invariants(s, t, r)
    assert s['pair_all'].sum() > 256 * 100000          # the epidemic happened


@pytest.mark.gpu
def test_every_intervention_type_equal_oracle(cuda_lib, sx_oracle):
    """Several mobility epochs, masks, both variants, vaccination and contact tracing, three replicas side by side."""
    kw = stress_kw()
    gpu = helpers.make_context(cuda_lib, seed=11, n_replicas=3, max_days=130, **kw)
    for _ in range(4):
        gpu.run(30)
    s, t = gpu.transmission_settings(), gpu.transmission_stats()
    assert len(set(gpu._epoch_of_day().tolist())) > 3
    for r in range(3):
        cpu = helpers.make_context(sx_oracle, seed=11 + r, max_days=130, **kw)
        cpu.run(120)
        c = cpu.transmission_settings()
        for k in SETTINGS:
            assert np.array_equal(s[k][r], c[k][0]), (r, k)
        assert np.array_equal(gpu.infection_places(r), cpu.infection_places(0)), r
        check_invariants(s, t, r, int((gpu._engine.read_agents(r)['infector'] >= 0).sum()))
    assert (s['pair_all'].sum(axis=(0, 2, 3)) > 0).all()


@pytest.mark.gpu
def test_bad_epochs_are_refused(cuda_lib):
    """A wrong number of days or an epoch without a contact table is an error, not a fault."""
    ctx = helpers.make_context(cuda_lib, seed=5, max_days=40, **stress_kw(20000))
    ctx.run(30)
    ep = ctx._epoch_of_day()
    for bad in (ep[:-1], np.where(np.arange(ep.size) == 20, 99, ep), np.where(np.arange(ep.size) == 3, -1, ep)):
        with pytest.raises(_abi.EngineError):
            ctx._engine.transmission_settings(bad)
        with pytest.raises(_abi.EngineError):
            ctx._engine.read_infection_places(0, bad)
    assert ctx.transmission_settings()['pair_all'].sum() > 0        # the engine is fine afterwards


@pytest.mark.gpu
def test_tables_survive_save_load_and_reset(cuda_lib):
    """load_state into a fresh Context: the device never saw the past days' schedule, the epochs come from the replayed
    plan."""
    kw = dict(stress_kw(60000), seed=21, n_replicas=2, max_days=100)
    a = helpers.make_context(cuda_lib, **kw)
    a.run(47)
    blob, s47 = a.save_state(), a.transmission_settings()
    b = helpers.make_context(cuda_lib, **kw)
    b.load_state(blob)
    sb = b.transmission_settings()
    assert all(np.array_equal(s47[k], sb[k]) for k in SETTINGS)
    assert np.array_equal(a.infection_places(1), b.infection_places(1))
    a.run(43)
    b.run(43)
    s90 = a.transmission_settings()
    sb = b.transmission_settings()
    assert all(np.array_equal(s90[k], sb[k]) for k in SETTINGS)
    a.reset(21)                                 # the sparse reset, then the same run again
    assert a.transmission_settings()['pair_all'].sum() == 0
    a.run(90)
    sa = a.transmission_settings()
    assert all(np.array_equal(s90[k], sa[k]) for k in SETTINGS)
    assert np.array_equal(a.infection_places(1), b.infection_places(1))


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
        q.put([(c.transmission_settings(), c.infection_places(0)) for c in ctxs])
    except Exception:
        q.put(traceback.format_exc())


@pytest.mark.gpu
@pytest.mark.parametrize('world', [2, 4])
def test_local_ranks_on_one_gpu(cuda_lib, sx_oracle, monkeypatch, world):
    """Population-sharded mode (several ranks on one GPU): every rank returns the single-engine tables and places."""
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
    ref = helpers.make_context(sx_oracle, **dict(stress_kw(), seed=11, max_days=130))
    ref.run(120)
    s, places = ref.transmission_settings(), ref.infection_places(0)
    for rank, (sr, pr) in enumerate(out):
        for k in SETTINGS:
            assert np.array_equal(sr[k], s[k]), (rank, k)
        assert np.array_equal(pr, places), rank


@pytest.mark.gpu
def test_school_closure_gpu(cuda_lib, sx_oracle):
    kw = dict(school_kw(), n_replicas=2, max_days=70)
    gpu = helpers.make_context(cuda_lib, seed=8, **kw)
    gpu.run(60)
    s = gpu.transmission_settings()
    check_school_closure(gpu, s)
    cpu = helpers.make_context(sx_oracle, seed=8, **kw)
    cpu.run(60)
    c = cpu.transmission_settings()
    assert all(np.array_equal(s[k], c[k]) for k in SETTINGS)
