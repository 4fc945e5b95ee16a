"""The reference's real caller, calc/simulation.py:148-290 `simulate_individuals` (imported UNMODIFIED from
/root/reference by tests/ref_caller_shim.py, with stand-ins only for flask / flask_babel / flask_caching / xlrd),
driven over `reina_b200.model` bound as `cythonsim.model` -- the one-line integration INTEGRATION.md section 1 describes --
side by side with the same call over the unmodified Cython engine (oracle/_ref).

The live comparisons need the reference source tree ($REF) and skip where it is absent; the engine under the shim is the
CPU oracle library, injected through the test-only `_library` seam.  The CUDA engine runs behind exactly the same Python
surface (tests/test_gpu_*.py compare the two bit for bit).  The deterministic cells they compare are also checked without
the reference tree, against the reference engine's own output stored in tests/golden.
"""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

import helpers

REF = os.environ.get('REF', '/root/reference')
SHIM = os.path.join(helpers.ROOT, 'tests', 'ref_caller_shim.py')

needs_reference_tree = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'calc')), reason='needs the reference tree')
# the unmodified reference engine, Varsinais-Suomi with the default interventions, 256 seeds (tests/golden/make_golden.py)
REF_GOLD = os.path.join(helpers.ROOT, 'tests', 'golden', 'ref_ensemble_varsinais_suomi_default_n256.npz')


def _run(engine, out, days, area='Varsinais-Suomi', seed=3):
    r = subprocess.run([sys.executable, SHIM, engine, str(out), '--days', str(days), '--area', area, '--seed', str(seed)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    with open(out, 'rb') as f:
        return pickle.load(f)


@needs_reference_tree
def test_real_caller_over_the_shim_matches_the_reference_engine(tmp_path):
    from oracle import ref_harness
    if not ref_harness.available():
        pytest.skip('oracle/_ref not built')
    days = 30
    ref = _run('ref', tmp_path / 'ref.pkl', days)
    shim = _run('shim-oracle', tmp_path / 'shim.pkl', days)
    assert ref['engine_file'].startswith(os.path.join(helpers.ROOT, 'oracle', '_ref'))
    assert shim['engine_file'] == os.path.join(helpers.ROOT, 'reina_b200', 'model.py')
    a, b = ref['df'], shim['df']
    # identical frames as far as a caller can tell: columns, order, dtypes, index, shapes
    assert list(a.columns) == list(b.columns) and a.shape == b.shape == (days, 26)
    assert a.index.equals(b.index) and a.dtypes.equals(b.dtypes)
    aa, ab = ref['adf'], shim['adf']
    assert aa.columns.equals(ab.columns) and aa.index.equals(ab.index) and aa.dtypes.equals(ab.dtypes) and aa.shape == (days, 12 * 9)
    # deterministic cells agree exactly; the two engines use different random streams, so the rest is compared in
    # distribution by tests/test_oracle_pinned.py against >= 64 reference seeds
    assert a['susceptible'].iloc[0] == b['susceptible'].iloc[0] == 479861
    for col in ('total_icu_units', 'mobility_limitation', 'vaccinated'):
        assert np.array_equal(a[col].to_numpy(dtype=float), b[col].to_numpy(dtype=float)), col
    assert np.array_equal(aa['susceptible'].iloc[0].to_numpy(), ab['susceptible'].iloc[0].to_numpy())
    for f in (a, b):                                   # imports of 2020-02-22 .. 03-15 (default interventions) took hold in both
        assert f['all_infected'].iloc[-1] > 200 and f['susceptible'].iloc[-1] + f['all_infected'].iloc[-1] == 479861

    # the per-day API the real caller uses (generate_state + iterate, one day at a time) gives the same numbers as this
    # repo's batched caller (reina_b200/simulation.py: one run, one fetch) on the same engine and seed
    from reina_b200 import inputs, simulation
    v = inputs.default_variables(simulation_days=days, area_name='Varsinais-Suomi', random_seed=3)
    ctx = simulation.make_context(v, _library=helpers.oracle_library())
    df2, adf2 = simulation.simulate_individuals(v, context=ctx)
    cols = [c for c in b.columns if c != 'us_per_infected']
    assert np.array_equal(b[cols].to_numpy(dtype=float), df2[cols].to_numpy(dtype=float))
    assert np.array_equal(ab.to_numpy(), adf2.to_numpy()) and ab.columns.equals(adf2.columns)


@needs_reference_tree
@pytest.mark.gpu
def test_real_caller_over_the_cuda_shim(tmp_path):
    """Only where a GPU and the reference tree meet (never on the driver's boxes): the same call over the shipped module."""
    days = 30
    cuda = _run('shim-cuda', tmp_path / 'cuda.pkl', days)
    orac = _run('shim-oracle', tmp_path / 'shim.pkl', days)
    cols = [c for c in cuda['df'].columns if c != 'us_per_infected']
    assert np.array_equal(cuda['df'][cols].to_numpy(dtype=float), orac['df'][cols].to_numpy(dtype=float))
    assert np.array_equal(cuda['adf'].to_numpy(), orac['adf'].to_numpy())


@pytest.mark.parametrize('engine', ['oracle', pytest.param('cuda', marks=pytest.mark.gpu)])
def test_caller_frames_hold_the_reference_engine_cells(engine):
    """The deterministic cells of the live comparison above, without the reference tree: this repo's caller
    (reina_b200.simulation, same area, days and seed) over the CPU oracle and over the CUDA engine, against the output of
    the unmodified reference engine stored in REF_GOLD.  There these cells take the same value in all 256 seeds."""
    from reina_b200 import inputs, simulation
    gold = np.load(REF_GOLD)
    names = list(gold['names'])
    days = 30
    v = inputs.default_variables(simulation_days=days, area_name='Varsinais-Suomi', random_seed=3)
    lib = helpers.oracle_library() if engine == 'oracle' else helpers.cuda_library()
    df, adf = simulation.simulate_individuals(v, context=simulation.make_context(v, _library=lib))
    assert df.shape == (days, 26) and adf.shape == (days, 12 * 9)
    for col in ('total_icu_units', 'mobility_limitation', 'vaccinated'):
        j = names.index(col)
        assert (gold['std'][:days, j] == 0).all(), col
        assert np.array_equal(df[col].to_numpy(dtype=float), gold['mean'][:days, j]), col
    j = names.index('susceptible')
    assert gold['std'][0, j] == 0 and df['susceptible'].iloc[0] == gold['mean'][0, j] == 479861
    assert adf['susceptible'].iloc[0].sum() == 479861
    # the imports of 2020-02-22 .. 03-15 (default interventions) took hold
    assert df['all_infected'].iloc[-1] > 200 and df['susceptible'].iloc[-1] + df['all_infected'].iloc[-1] == 479861
