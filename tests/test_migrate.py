"""Moving replicas between engines and GPUs (rb_replica_bytes / rb_export_replicas / rb_import_replicas /
rb_copy_replicas / rb_comm_move_replicas; Context.export_replicas / import_replicas / copy_replicas_from) and one particle
filter over several Contexts or ranks (ensemble.migration_plan, particle_filter with a list of Contexts or a comm).

CPU: migration_plan is assign_slots on one rank, writes only from survivors and moves the fewest replicas; a reference
replica exported and imported (or copied) into another engine continues as it would have; the filter over two reference
Contexts -- in one process, or in two gloo processes through host records -- equals a replay of its ancestors and seeds
on one Context holding all replicas; bad moves are refused and leave the engine usable.  GPU: the same on the CUDA
engine, against the reference, at the bench geometry and between two NCCL ranks where there are two GPUs.

The CPU reference is tests/oracle_migrate.c over the reference of test_branch.py, compiled into a library of its own in
the temporary directory, keyed by the hash of the sources."""
import hashlib
import multiprocessing
import os
import shutil
import socket
import subprocess
import sys
import tempfile
import traceback

import numpy as np
import pytest

import helpers
from reina_b200 import _abi, ensemble
from test_branch import assert_same_ensemble, replica_state
from test_transmission import stress_kw
from test_transmission_settings import ORACLE_PROBES

_mg_oracle = None


def mg_oracle_library():
    """The probed oracle plus the transmission, settings, branch and migration entry points, built once per source state."""
    global _mg_oracle
    if _mg_oracle is None:
        files = [('oracle', 'reina_oracle.c'), ('tests', 'oracle_transmission.c'), ('tests', 'oracle_settings.c'),
                 ('tests', 'oracle_branch.c'), ('tests', 'oracle_migrate.c'), ('include', 'reina_b200.h')]
        src = {f: open(os.path.join(helpers.ROOT, *f), 'rb').read().decode() for f in files}
        key = hashlib.sha1(''.join(src[f] for f in files).encode() + repr(ORACLE_PROBES).encode()).hexdigest()[:16]
        lib = os.path.join(tempfile.gettempdir(), 'reina_mg_oracle_%d_%s.so' % (os.getuid(), key))
        if not os.path.exists(lib):
            text = src[('oracle', 'reina_oracle.c')]
            for anchor, line in ORACLE_PROBES:
                assert text.count(anchor) == 1, 'oracle probe anchor not found exactly once: %r' % anchor
                text = text.replace(anchor, anchor + line)
            src[('oracle', 'reina_oracle.c')] = text
            tree = tempfile.mkdtemp(prefix='reina_mg_oracle_')
            try:
                for f in files:
                    os.makedirs(os.path.join(tree, f[0]), exist_ok=True)
                    with open(os.path.join(tree, *f), 'w') as fh:
                        fh.write(src[f])
                tmp = '%s.%d.tmp' % (lib, os.getpid())
                subprocess.run([os.environ.get('CC', 'gcc'), '-O2', '-fPIC', '-std=c11', '-ffp-contract=off', '-fno-fast-math',
                                '-shared', '-o', tmp, os.path.join(tree, 'tests', 'oracle_migrate.c'), '-lm'], check=True)
                os.replace(tmp, lib)
            finally:
                shutil.rmtree(tree, ignore_errors=True)
        _mg_oracle = _abi.Library(lib, 'ro_')
        _mg_oracle.bind_transmission()
        _mg_oracle.bind_settings()
        _mg_oracle.bind_branch()
        _mg_oracle.bind_migrate()
    return _mg_oracle


@pytest.fixture(scope='module')
def mg_oracle():
    return mg_oracle_library()


class SendRecvComm(helpers.TorchComm):
    """TorchComm plus the optional sendrecv of the particle filter's host-record path: point-to-point gloo messages,
    their sizes agreed by one all-gather first."""

    def sendrecv(self, payload):
        import torch
        sizes = np.zeros(self.size, dtype=np.int64)
        for p, b in payload.items():
            sizes[p] = len(b)
        table = self.allgather(sizes)                         # [from, to]
        reqs, bufs = [], {}
        for p, b in payload.items():
            reqs.append(self.dist.isend(torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()), p))
        for p in range(self.size):
            if p != self.rank and table[p, self.rank] > 0:
                bufs[p] = torch.empty(int(table[p, self.rank]), dtype=torch.uint8)
                reqs.append(self.dist.irecv(bufs[p], p))
        for r in reqs:
            r.wait()
        return {p: t.numpy().tobytes() for p, t in bufs.items()}


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def full_state(ctx, r):
    return dict(replica_state(ctx, r), seeds_all=ctx._engine.read_seeds()[r])


def _cross_moves(anc, R):
    g = np.arange(anc.shape[1])
    return int(((anc // R) != (g // R)[None]).sum())


# ---------------------------------------------------------------- CPU
@pytest.mark.parametrize('seed', range(4))
def test_migration_plan(seed):
    rng = np.random.default_rng(seed)
    for K, R in ((1, 1), (1, 9), (2, 4), (3, 7), (8, 16)):
        for _ in range(20):
            w = rng.random(K * R) ** 6
            w[rng.random(K * R) < 0.3] = 0
            if not w.sum() > 0:
                w[0] = 1
            c = ensemble.systematic_resample(w, rng)
            src = ensemble.migration_plan(c, K)
            if K == 1:
                assert np.array_equal(src, ensemble.assign_slots(c))
            assert np.array_equal(np.bincount(src, minlength=K * R), c)
            assert (c[src] > 0).all() and (src[src] == src).all()               # every source is a survivor
            dropped = (c == 0).reshape(K, R).sum(1)
            extras = np.maximum(c - 1, 0).reshape(K, R).sum(1)
            assert _cross_moves(src[None], R) == np.maximum(dropped - extras, 0).sum()
    assert ensemble.migration_plan([0, 0, 2, 2, 0, 1, 1, 2], 2).tolist() == [2, 3, 2, 3, 7, 5, 6, 7]
    with pytest.raises(ValueError):
        ensemble.migration_plan([1, 1, 1], 2)


def test_oracle_record_continues_in_another_engine(mg_oracle):
    """Export / import and the engine-to-engine copy: the written slot, given its source's seed, continues for 20 days
    exactly as the source -- rows, agents, queue, capacity, seed history and places of infection."""
    kw = dict(stress_kw(30000), max_days=80)
    a = helpers.make_context(mg_oracle, seed=40, n_replicas=3, **kw)
    b = helpers.make_context(mg_oracle, seed=90, n_replicas=2, **kw)
    a.run(38)
    b.run(38)
    rec = a.export_replicas([1])
    assert rec.shape == (1, a._engine.replica_bytes())
    assert b.import_replicas([0], rec, [41]).tolist() == [41]
    assert b.copy_replicas_from(a, [2], [1], [42]).tolist() == [42]
    assert a._engine.read_queue(1).size > 0 or a._engine.read_queue(2).size > 0
    a.run(20)
    b.run(20)
    for ra, rb in ((1, 0), (2, 1)):
        x, y = full_state(a, ra), full_state(b, rb)
        for k in x:
            assert np.array_equal(x[k], y[k]), (ra, k)
        assert np.array_equal(a.infection_places(ra), b.infection_places(rb))
    # fresh seeds: none the destination or the record ever used
    rec = a.export_replicas([0])
    s = b.import_replicas([1], rec)
    used = set(b._engine.read_seeds()[0].tolist()) | set(a._engine.read_seeds().ravel().tolist())
    assert int(s[0]) not in used - {int(s[0])} and b._engine.read_seeds()[1, b.day] == s[0]


def test_oracle_refusals_leave_the_engine_usable(mg_oracle):
    kw = dict(stress_kw(20000), max_days=60)
    a = helpers.make_context(mg_oracle, seed=9, n_replicas=3, **kw)
    b = helpers.make_context(mg_oracle, seed=19, n_replicas=3, **kw)
    c = helpers.make_context(mg_oracle, seed=29, n_replicas=3, **dict(kw, age_count_override=helpers.small_population(21000)))
    ref = helpers.make_context(mg_oracle, seed=19, n_replicas=3, **kw)
    for x in (a, b, c, ref):
        x.run(10)
    rec = a.export_replicas([0, 1])
    bad = [lambda: b.import_replicas([0, 0], rec, [1, 2]),                    # duplicate slots
           lambda: b.import_replicas([0, 3], rec, [1, 2]),                    # slot out of range
           lambda: b.import_replicas([0], rec[:1, :-4], [1]),                 # wrong size
           lambda: c.import_replicas([0], rec[:1], [1]),                      # another shape
           lambda: a.export_replicas([3]),
           lambda: b._engine.copy_replicas_from(a._engine, [0, 5], [0, 1], [1, 2])]
    for f in bad:
        with pytest.raises(_abi.EngineError):
            f()
    with pytest.raises(ValueError):
        b.copy_replicas_from(b, [0], [1])
    with pytest.raises(_abi.EngineError):
        c.copy_replicas_from(a, [0], [1])                                    # another population
    a.run(1)
    with pytest.raises(_abi.EngineError):                                    # a record of another day
        b.import_replicas([0], a.export_replicas([0]), [1])
    with pytest.raises(ValueError):
        b.copy_replicas_from(a, [0], [1])
    b.run(15)
    ref.run(15)
    assert not helpers.diff_report(b, ref, 25)


def _split_filter_case(lib, R, seed0, truth_seed, n_agents=20000, days=(6, 12, 18, 24, 30), names=('in_ward', 'all_detected'),
                       **extra):
    kw = dict(age_count_override=helpers.small_population(n_agents), max_days=days[-1] + 20, **extra)
    truth = helpers.make_context(mg_oracle_library(), seed=truth_seed, **kw)
    truth.run(days[-1] + 1)
    t = truth.series(0, days[-1] + 1)
    obs = {d: {n: int(ensemble._model_counts(truth, t[:, d], n)[0]) for n in names} for d in days}
    parts = [helpers.make_context(lib, seed=seed0 + k * R, n_replicas=R, **kw) for k in range(2)]
    return parts, obs, kw


def _replay(lib, out, R_total, seed0, kw, end):
    one = helpers.make_context(lib, seed=seed0, n_replicas=R_total, **kw)
    for k, d in enumerate(out['days']):
        if out['resampled'][k]:
            one.run(int(d) - one.day)
            one.branch(out['ancestors'][k], out['seeds'][k])
    one.run(end - one.day)
    return one


def _assert_split_equals(parts, one, R):
    for g in range(one.n_replicas):
        a, b = full_state(parts[g // R], g % R), full_state(one, g)
        for k in a:
            assert np.array_equal(a[k], b[k]), (g, k)


def test_oracle_filter_over_two_contexts_equals_replay(mg_oracle):
    R, seed0 = 6, 500
    parts, obs, kw = _split_filter_case(mg_oracle, R, seed0, 4242)
    out = ensemble.particle_filter(parts, obs, seed=3, ess_threshold=0.95)
    assert out['ancestors'].shape == (5, 2 * R) and out['seeds'].shape == (5, 2 * R)
    assert _cross_moves(out['ancestors'], R) > 0, 'the case moves no replica between the Contexts'
    for p in parts:
        p.run(40 - p.day)
    one = _replay(mg_oracle, out, 2 * R, seed0, kw, 40)
    _assert_split_equals(parts, one, R)
    # one Context of 2R replicas filtered directly weighs the same particles (its plan keeps copies on its one Context)
    whole = helpers.make_context(mg_oracle, seed=seed0, n_replicas=2 * R, **kw)
    o2 = ensemble.particle_filter(whole, obs, seed=3, ess_threshold=0.95)
    assert np.array_equal(out['loglik'][0], o2['loglik'][0]) and np.array_equal(out['resampled'][:1], o2['resampled'][:1])


def _gloo_worker(rank, world, port, out_dir, R, seed0):
    sys.path.insert(0, os.path.join(helpers.ROOT, 'tests'))
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        parts, obs, kw = _split_filter_case(mg_oracle_library(), R, seed0, 4242)
        ctx = parts[rank]
        out = ensemble.particle_filter(ctx, obs, seed=3, ess_threshold=0.95, comm=SendRecvComm(dist))
        ctx.run(40 - ctx.day)
        st = {'%s_%d' % (k, r): v for r in range(R) for k, v in full_state(ctx, r).items()}
        np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), log_evidence=out['log_evidence'],
                 **{k: out[k] for k in ('ancestors', 'loglik', 'seeds', 'ess', 'resampled', 'days')}, **st)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_oracle_filter_over_two_gloo_ranks_equals_replay(tmp_path):
    import torch.multiprocessing as mp
    R, seed0 = 6, 500
    mp.spawn(_gloo_worker, args=(2, _free_port(), str(tmp_path), R, seed0), nprocs=2, join=True)
    r = [np.load(tmp_path / ('rank%d.npz' % k)) for k in range(2)]
    for k in ('ancestors', 'loglik', 'seeds', 'ess', 'resampled', 'log_evidence'):
        assert np.array_equal(r[0][k], r[1][k]), k
    assert _cross_moves(r[0]['ancestors'], R) > 0
    _, _, kw = _split_filter_case(mg_oracle_library(), R, seed0, 4242)
    out = {k: r[0][k] for k in ('ancestors', 'seeds', 'resampled', 'days')}
    one = _replay(mg_oracle_library(), out, 2 * R, seed0, kw, 40)
    for g in range(2 * R):
        b = full_state(one, g)
        for k in b:
            assert np.array_equal(r[g // R]['%s_%d' % (k, g % R)], b[k]), (g, k)


def test_filter_refuses_a_list_with_a_multi_rank_comm(mg_oracle):
    class Two:
        rank, size = 0, 2
    parts, obs, _ = _split_filter_case(mg_oracle, 2, 1, 4242, n_agents=4000)
    with pytest.raises(ValueError):
        ensemble.particle_filter(parts, obs, comm=Two())


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_round_trip_and_copy_continue_as_the_source(cuda_lib):
    """Host round trip and rb_copy_replicas on device 0, each slot given its source's seed: for 30 days the written
    slots equal their sources in every series, agent, queue, seed history, transmission and settings table."""
    kw = dict(stress_kw(), max_days=100)
    a = helpers.make_context(cuda_lib, seed=11, n_replicas=4, **kw)
    b = helpers.make_context(cuda_lib, seed=11, n_replicas=4, **kw)
    c = helpers.make_context(cuda_lib, seed=77, n_replicas=4, **kw)
    for x in (a, b, c):
        x.run(40)
    seeds = a.replica_seeds()
    c.import_replicas([0, 2], a.export_replicas([0, 2]), seeds[[0, 2]])
    c.copy_replicas_from(a, [1, 3], [1, 3], seeds[[1, 3]])
    for x in (b, c):
        x.run(30)
    assert_same_ensemble(c, b, 'moved')


@pytest.mark.gpu
def test_gpu_filter_over_two_engines_equals_oracle_and_replay(cuda_lib, mg_oracle):
    """Every-intervention schedule, 2 x 8 replicas: the CUDA filter over two engines equals the reference's over two
    reference Contexts and the replay on one 16-replica CUDA engine."""
    R, seed0 = 8, 11
    extra = dict(variables=stress_kw()['variables'], interventions=helpers.stress_interventions())
    outs = []
    for lib in (cuda_lib, mg_oracle):
        parts, obs, kw = _split_filter_case(lib, R, seed0, 8888, n_agents=80000, days=(14, 21, 28, 35, 42, 49), **extra)
        out = ensemble.particle_filter(parts, obs, seed=2, ess_threshold=0.9)
        for p in parts:
            p.run(kw['max_days'] - p.day)                    # to the last day the Contexts hold
        outs.append((out, parts))
    (a, pa), (b, pb) = outs
    assert _cross_moves(a['ancestors'], R) > 0
    for k in ('ancestors', 'loglik', 'seeds', 'ess', 'resampled'):
        assert np.array_equal(a[k], b[k]), k
    for g, c in zip(pa, pb):
        assert_same_ensemble(g, c, 'gpu vs oracle')
    one = _replay(cuda_lib, a, 2 * R, seed0, kw, kw['max_days'])
    _assert_split_equals(pa, one, R)


@pytest.mark.gpu
def test_gpu_bench_geometry_filter_equals_replay(cuda_lib):
    """2 engines x 128 HUS replicas, 180 days, weekly in_ward / in_icu of a truth run: every row equals the replay on
    one 256-replica engine (the split run first, then the replay, so that at most ~45 GB are held at once)."""
    R, seed0, days = 128, 1000, list(range(7, 180, 7))
    kw = dict(max_days=181)
    truth = helpers.make_context(cuda_lib, seed=999999, **kw)
    truth.run(180)
    t = truth.series(0, 180)
    truth.close()
    obs = {d: {n: int(ensemble._model_counts(truth, t[:, d], n)[0]) for n in ('in_ward', 'in_icu')} for d in days}
    parts = [helpers.make_context(cuda_lib, seed=seed0 + k * R, n_replicas=R, **kw) for k in range(2)]
    out = ensemble.particle_filter(parts, obs, seed=5)
    for p in parts:
        p.run(180 - p.day)
    rows = np.concatenate([p.series(0, 180) for p in parts])
    for p in parts:
        p.close()
    assert _cross_moves(out['ancestors'], R) > 0
    one = _replay(cuda_lib, out, 2 * R, seed0, kw, 180)
    assert np.array_equal(rows, one.series(0, 180))
    one.close()


@pytest.mark.gpu
def test_gpu_refusals_leave_the_engine_usable(cuda_lib, mg_oracle):
    kw = dict(stress_kw(20000), max_days=60)
    a = helpers.make_context(cuda_lib, seed=9, n_replicas=3, **kw)
    b = helpers.make_context(cuda_lib, seed=19, n_replicas=3, **kw)
    c = helpers.make_context(cuda_lib, seed=29, n_replicas=3, **dict(kw, age_count_override=helpers.small_population(21000)))
    ref = helpers.make_context(mg_oracle, seed=19, n_replicas=3, **kw)
    for x in (a, b, c, ref):
        x.run(10)
    rec = a.export_replicas([0, 1])
    bad = [lambda: b.import_replicas([0, 0], rec, [1, 2]),
           lambda: b.import_replicas([0, 3], rec, [1, 2]),
           lambda: b.import_replicas([0], rec[:1, :-4], [1]),
           lambda: c.import_replicas([0], rec[:1], [1]),
           lambda: a.export_replicas([3]),
           lambda: b._engine.copy_replicas_from(a._engine, [0, 5], [0, 1], [1, 2]),
           lambda: b._engine.copy_replicas_from(a._engine, [0, 1], [2, 2], [1, 2]),
           lambda: b._engine.copy_replicas_from(b._engine, [0], [1], [1]),
           lambda: c._engine.copy_replicas_from(a._engine, [0], [1], [1]),
           lambda: b._engine.comm_move_replicas([0], [1], [], [], [])]       # no communicator
    for f in bad:
        with pytest.raises(_abi.EngineError):
            f()
    a.run(1)
    with pytest.raises(_abi.EngineError):
        b.import_replicas([0], a.export_replicas([0]), [1])
    with pytest.raises(_abi.EngineError):
        b._engine.copy_replicas_from(a._engine, [0], [1], [1])
    b.run(15)
    ref.run(15)
    assert not helpers.diff_report(b, ref, 25)


def _sharded_worker(q):
    try:
        from reina_b200 import sharded
        kw = dict(stress_kw(20000), seed=9, max_days=60)
        ctxs = [helpers.make_context(helpers.cuda_library(), device=0, **kw) for _ in range(2)]
        sharded.join_local(ctxs)
        refused = 0
        for f in (lambda: ctxs[0].export_replicas([0]), lambda: ctxs[0]._engine.import_replicas([0], [5], np.zeros(ctxs[0]._engine.replica_bytes(), np.uint8)),
                  lambda: ctxs[0]._engine.copy_replicas_from(ctxs[1]._engine, [0], [0], [5])):
            try:
                f()
            except _abi.EngineError:
                refused += 1
        sharded.run_local(ctxs, 20)
        q.put((refused, [c.series(0, 20) for c in ctxs]))
    except Exception:
        q.put(traceback.format_exc())


@pytest.mark.gpu
def test_gpu_sharded_engine_refuses_moves(cuda_lib, oracle_lib, monkeypatch):
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
    assert refused == 3
    ref = helpers.make_context(oracle_lib, **dict(stress_kw(20000), seed=9, max_days=60))
    ref.run(20)
    for r in rows:
        assert np.array_equal(r, ref.series(0, 20))


def _nccl_worker(rank, world, uid, q):
    try:
        from reina_b200 import comm as _comm
        R, seed0 = 8, 11
        extra = dict(variables=stress_kw()['variables'], interventions=helpers.stress_interventions())
        parts, obs, kw = _split_filter_case(helpers.cuda_library(), R, seed0, 8888, n_agents=80000, days=(14, 21, 28, 35, 42, 49),
                                            device=rank, **extra)
        ctx = parts[rank]
        for k, p in enumerate(parts):
            if k != rank:
                p.close()
        c = _comm.connect(ctx._engine, rank=rank, size=world, unique_id=uid)
        out = ensemble.particle_filter(ctx, obs, seed=2, ess_threshold=0.9, comm=c)
        ctx.run(kw['max_days'] - ctx.day)
        q.put((rank, dict(out=out, rows=ctx.series(0, kw['max_days']), seeds=ctx._engine.read_seeds(),
                          agents=[ctx._engine.read_agents(r) for r in range(R)])))
    except Exception:
        q.put((rank, traceback.format_exc()))


@pytest.mark.gpu
def test_gpu_nccl_move_between_two_ranks_equals_replay(cuda_lib):
    """rb_comm_move_replicas: the filter of test_gpu_filter_over_two_engines... over two NCCL ranks, one GPU each,
    equals the replay on one 16-replica engine.  Needs two GPUs."""
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
    assert _cross_moves(out['ancestors'], R) > 0
    for k in ('ancestors', 'loglik', 'seeds'):
        assert np.array_equal(out[k], res[1]['out'][k]), k
    _, _, kw = _split_filter_case(cuda_lib, R, seed0, 8888, n_agents=80000, days=(14, 21, 28, 35, 42, 49),
                                  variables=stress_kw()['variables'], interventions=helpers.stress_interventions())
    one = _replay(cuda_lib, out, 2 * R, seed0, kw, kw['max_days'])
    rows = one.series(0, kw['max_days'])
    seeds = one._engine.read_seeds()
    for k in range(2):
        assert np.array_equal(res[k]['rows'], rows[k * R:(k + 1) * R]), k
        assert np.array_equal(res[k]['seeds'], seeds[k * R:(k + 1) * R]), k
        for r in range(R):
            assert np.array_equal(res[k]['agents'][r], one._engine.read_agents(k * R + r)), (k, r)
