"""Drop-in for the reference's `cythonsim.model` module (= cythonsim/main.pyx, cythonsim/__init__.py:5-8).

`calc.simulation` uses this module surface (SURVEY.md section 8b): `DISEASE_PARAMS`, `__file__`,
`Context(population_params, healthcare_params, disease_params, start_date, random_seed)`,
`ctx.add_intervention(iv)`, `ctx.iterate()`, `ctx.generate_state()`, `ctx.get_date_for_today()`,
`ctx.get_population_stats(what)`, `ctx.sample(what, age, severity)`, `ctx.apply_intervention(iv)`,
`SimulationFailed`, `SEVERITY_TO_STR`, `STATE_TO_STR`, `PROBLEM_TO_STR`.

Everything per-agent runs in hand-written CUDA behind the C-ABI of include/reina_b200.h
(libreina_b200.so, bound with ctypes).  The host side only does what the reference does in Python:
parameter marshalling, the intervention schedule (apply_intervention, main.pyx:1880-1960) and the
contact-probability tables (ContactMatrix.generate_contact_probabilities, main.pyx:1184-1235, here in
numpy instead of pandas).  There is no CPU fallback: constructing a Context without the built CUDA
library raises.

Extensions beyond the reference surface (all optional keyword arguments / extra methods):
  * `n_replicas=R`: R ensemble members (seeds random_seed .. random_seed+R-1) advanced by the same kernel
    launches; `generate_state(replica=r)`, `run(days)`, `series()`.
"""
import math
from datetime import date, timedelta

import numpy as np

from . import _abi
from ._abi import ATTRS, DayParams, Variant, Config, EngineError  # noqa: F401
from .inputs import DISEASE_PARAMS  # noqa: F401  (main.pyx:777-785)

# main.pyx:81-121
CONTACT_PLACE_TO_STR = {100: 'all', 0: 'home', 1: 'work', 2: 'school', 3: 'transport', 4: 'leisure', 5: 'other'}
_STR_TO_PLACE = {v: k for k, v in CONTACT_PLACE_TO_STR.items()}
PLACE_ALL = 100
STATE_TO_STR = {0: 'SUSCEPTIBLE', 1: 'INCUBATION', 2: 'ILLNESS', 3: 'HOSPITALIZED', 4: 'IN_ICU',
                5: 'RECOVERED', 6: 'DEAD'}
SEVERITY_TO_STR = {0: 'ASYMPTOMATIC', 1: 'MILD', 2: 'SEVERE', 3: 'CRITICAL', 4: 'FATAL'}
STR_TO_SEVERITY = {v: k for k, v in SEVERITY_TO_STR.items()}
# the columns of Context.set_severity_scale / severity_scale: the observed series each one mainly moves is in_ward,
# in_icu and dead
SEVERITY_SCALES = ('severe', 'critical', 'fatal')
PROBLEM_TO_STR = {
    0: 'No problemos', 1: 'Too many infectees', 2: 'Too many contacts', 3: 'Hospital accounting failure',
    4: 'Negative number of contacts', 5: 'Malloc failure', 6: 'Other failure', 7: 'Wrong state',
    8: 'Contact probability failure', 9: 'Infectees mismatch',
}
NO_TESTING, ALL_WITH_SYMPTOMS_CT, ALL_WITH_SYMPTOMS, ONLY_SEVERE_SYMPTOMS = range(4)   # main.pyx:441-445

# main.pyx:660-682
INFECTIOUSNESS_OVER_TIME = (
    (-10, 0.00183), (-9, 0.00280), (-8, 0.00446), (-7, 0.00742), (-6, 0.01291), (-5, 0.02350),
    (-4, 0.04419), (-3, 0.08247), (-2, 0.14018), (-1, 0.19032), (0, 0.18539), (1, 0.13091),
    (2, 0.07538), (3, 0.04018), (4, 0.02144), (5, 0.01185), (6, 0.00686), (7, 0.00415),
    (8, 0.00262), (9, 0.00172), (10, 0.00117),
)

SAMPLE_KINDS = {'contacts_per_day': 0, 'symptom_severity': 1, 'incubation_period': 2, 'illness_period': 3,
                'hospitalization_period': 4, 'icu_period': 5, 'onset_to_removed_period': 6}

f32 = np.float32


class SimulationFailed(Exception):   # main.pyx:124
    pass


# ---------------------------------------------------------------------------------------------------
# Disease parameters -> rb_variant  (variant_init, main.pyx:820-850; cv_* helpers :684-730, :808-817)
# ---------------------------------------------------------------------------------------------------
def _greatest_lte_table(pairs, n_ages):
    """cv_get_greatest_lte (main.pyx:721-730) evaluated for every single-year age; values are stored as
    C floats by cv_init (:690-702)."""
    classes = [int(k) for k, _ in pairs]
    values = [f32(v) for _, v in pairs]
    out = np.zeros(_abi.RB_MAX_AGES, dtype=np.float32)
    for age in range(n_ages):
        idx = len(classes) - 1
        for i, k in enumerate(classes):
            if k > age:
                idx = i - 1
                break
        out[age] = values[idx]
    return out


def _cv_div(a, b):
    assert [x[0] for x in a] == [x[0] for x in b]
    return [(ka, va / vb) for (ka, va), (_, vb) in zip(a, b)]


def _gamma_params(mu, cv):
    """RandomPool.gamma, simrandom.pyx:46-55, in C float arithmetic."""
    mu, cv = f32(mu), f32(cv)
    sigma = f32(cv * mu)
    theta = f32(f32(sigma * sigma) / mu)
    kappa = f32(mu / theta)
    return kappa, theta


def make_variant(params, n_ages):
    v = Variant()
    v.p_hospital_death_no_beds = params['p_hospital_death_no_beds']
    v.p_icu_death_no_beds = params['p_icu_death_no_beds']
    v.infectiousness_multiplier = params['infectiousness_multiplier']
    v.p_asymptomatic_infection = params['p_asymptomatic_infection']
    v.p_mask_protects_others = params['p_mask_protects_others']
    v.p_mask_protects_wearer = params['p_mask_protects_wearer']
    v.ratio_in_ward = params['ratio_of_duration_in_ward']
    v.ratio_before_hospitalisation = params['ratio_of_duration_before_hospitalisation']
    v.incubation_kappa, v.incubation_theta = _gamma_params(params['mean_incubation_duration'], 0.86)
    v.onset_death_kappa, v.onset_death_theta = _gamma_params(params['mean_duration_from_onset_to_death'], 0.45)
    v.onset_recovery_kappa, v.onset_recovery_theta = _gamma_params(
        params['mean_duration_from_onset_to_recovery'], 0.45)
    for kappa in (v.incubation_kappa, v.onset_death_kappa, v.onset_recovery_kappa):
        if not kappa > 1.0:
            raise ValueError('gamma shape <= 1 is outside the Marsaglia-Tsang branch the engine implements')
    for day, val in INFECTIOUSNESS_OVER_TIME:
        v.iot[day + 10] = val
    tabs = {
        _abi.T_SUSCEPTIBILITY: params['p_susceptibility'],
        _abi.T_SYMPTOMATIC: params['p_symptomatic'],
        # absolute -> conditional probabilities, main.pyx:834-843
        _abi.T_SEVERE: _cv_div(params['p_severe'], params['p_symptomatic']),
        _abi.T_CRITICAL: _cv_div(params['p_critical'], params['p_severe']),
        _abi.T_FATAL: _cv_div(params['p_fatal'], params['p_critical']),
        _abi.T_DEATH_OUTSIDE_HOSPITAL: params['p_death_outside_hospital'],
    }
    for t, pairs in tabs.items():
        arr = _greatest_lte_table([tuple(x) for x in pairs], n_ages)
        for age in range(_abi.RB_MAX_AGES):
            v.tab[t][age] = arr[age]
        if t == _abi.T_SUSCEPTIBILITY:
            v.reserved[0] = float(arr[:n_ages].max())      # upper bound used by the contact kernel's coarse filter
    return v


# ---------------------------------------------------------------------------------------------------
# Contact matrix (ContactMatrix, main.pyx:1119-1288) -- numpy instead of pandas
# ---------------------------------------------------------------------------------------------------
class ContactMatrix:
    def __init__(self, contacts_per_day, n_ages):
        self.n_ages = n_ages
        recs = self._records(contacts_per_day)
        # rows are ordered as `set_index([...]).sort_index()` orders them (main.pyx:1213): by place name,
        # then by contact band
        keys = sorted({(p, band) for p, _, band, _ in recs})
        if len(keys) > _abi.RB_MAX_ROWS:
            raise ValueError('more than %d contact rows per age' % _abi.RB_MAX_ROWS)
        self.keys = keys
        kidx = {k: i for i, k in enumerate(keys)}
        self.base = np.full((n_ages, len(keys)), np.nan)
        for p, age, band, c in recs:
            self.base[age, kidx[(p, band)]] = c
        if np.isnan(self.base).any():
            raise ValueError('contacts_per_day must list every (place, band) for every participant age')
        self.row_place = np.array([_STR_TO_PLACE[p] for p, _ in keys], dtype=np.uint8)
        self.row_lo = np.array([b[0] for _, b in keys], dtype=np.int32)
        self.row_hi = np.array([b[1] for _, b in keys], dtype=np.int32)
        self.mobility_factor = f32(1.0)           # cdef float, main.pyx:1128
        self.mobility_factors = []                # [place, min_age, max_age, factor(f32)]
        self.mobility_factor_changed = False
        self.mask_probabilities = np.zeros((n_ages, _abi.RB_N_PLACES))   # main.pyx:1178-1182

    @staticmethod
    def _records(cpd):
        if hasattr(cpd, 'itertuples'):     # pandas DataFrame as calc.simulation passes it
            return [(t.place_type, int(t.participant_age), tuple(int(x) for x in t.contact_age), float(t.contacts))
                    for t in cpd.itertuples()]
        return [(p, int(a), tuple(int(x) for x in b), float(c)) for p, a, b, c in cpd]

    def set_mobility_factor(self, factor, place=None, min_age=None, max_age=None):   # main.pyx:1250-1266
        self.mobility_factor = f32(factor)
        place = PLACE_ALL if place is None else place
        min_age = 0 if min_age is None else min_age
        max_age = self.n_ages - 1 if max_age is None else max_age
        for mf in self.mobility_factors:
            if mf[0] == place and mf[1] == min_age and mf[2] == max_age:
                mf[3] = f32(factor)
                break
        else:
            self.mobility_factors.append([place, min_age, max_age, f32(factor)])
        self.mobility_factor_changed = True

    def set_mask_probability(self, p, place=None, min_age=None, max_age=None):   # main.pyx:1268-1283
        min_age = 0 if min_age is None else min_age
        max_age = self.n_ages - 1 if max_age is None else max_age
        places = list(range(_abi.RB_N_PLACES)) if place is None else [place]
        for pl in places:
            self.mask_probabilities[min_age:max_age + 1, pl] = p

    def generate(self):
        """generate_contact_probabilities, main.pyx:1184-1235 -> arrays for rb_set_contact_table."""
        n_ages, nk = self.base.shape
        contacts = self.base.copy()
        ages = np.arange(n_ages)
        for place, min_age, max_age, factor in self.mobility_factors:
            if factor == 1.0:
                continue
            rows = (ages >= min_age) & (ages <= max_age)
            cols = np.ones(nk, dtype=bool) if place == PLACE_ALL else (self.row_place == place)
            contacts[np.ix_(rows, cols)] *= float(factor)
        total = contacts.sum(axis=1)
        with np.errstate(invalid='ignore', divide='ignore'):
            cum = np.cumsum(contacts / total[:, None], axis=1)
        R = _abi.RB_MAX_ROWS
        t = dict(
            n_rows=np.full(n_ages, nk, dtype=np.int32),
            cum_p=np.zeros((n_ages, R), dtype=np.float64),
            age_lo=np.zeros((n_ages, R), dtype=np.int32),
            age_hi=np.zeros((n_ages, R), dtype=np.int32),
            place=np.zeros((n_ages, R), dtype=np.uint8),
            mask_p=np.zeros((n_ages, R), dtype=np.float32),
            nr_contacts=np.ascontiguousarray(total, dtype=np.float64),
        )
        t['cum_p'][:, :nk] = cum
        t['age_lo'][:, :nk] = self.row_lo
        t['age_hi'][:, :nk] = np.minimum(self.row_hi, n_ages - 1)
        t['place'][:, :nk] = self.row_place
        t['mask_p'][:, :nk] = self.mask_probabilities[:, self.row_place].astype(np.float32)
        t['ncontact_cdf'] = ncontact_cdf(total)
        return t


def ncontact_cdf(nr_contacts_by_age):
    """Distribution of ContactMatrix.get_nr_contacts (main.pyx:1308-1320), tabulated.

    n = min(limit, int(max(1, L * c * factor)) - 1) with L ~ lognormal(0, 0.5), c = nr_contacts_by_age[age]:
    n <= k  <=>  L * c * factor < k + 2  <=>  z < 2 ln((k + 2) / (c * factor)), z standard normal, hence
    P(n <= k) = Phi(2 ln((k + 2) / (c * factor))).  Class 0: factor 1, limit 100; class 1: factor 0.5, limit 5
    (Disease.get_exposed_people, main.pyx:945-953).  Returns float64 [n_ages, 2, RB_NCDF]."""
    n_ages = len(nr_contacts_by_age)
    out = np.ones((n_ages, 2, _abi.RB_NCDF), dtype=np.float64)
    for age in range(n_ages):
        for cls, (factor, limit) in enumerate(((1.0, 100), (0.5, 5))):
            c = float(nr_contacts_by_age[age]) * factor
            if not c > 0:
                continue
            for k in range(limit):
                x = 2.0 * math.log((k + 2) / c)
                out[age, cls, k] = 0.5 * (1.0 + math.erf(x / math.sqrt(2.0)))
    return out


# ---------------------------------------------------------------------------------------------------
# Context
# ---------------------------------------------------------------------------------------------------
def fresh_seeds(hist, n):
    """n seeds none of which occurs in the seed history `hist` (any shape): counting up from its largest seed, skipping
    used ones (modulo 2^32).  Context.branch gives these to the replicas whose state it changes."""
    h = np.asarray(hist, dtype=np.uint32)
    used = set(h.ravel().tolist())
    nxt = int(h.max()) + 1 if h.size else 0
    out = np.zeros(n, dtype=np.int64)
    for j in range(n):
        while (nxt & 0xFFFFFFFF) in used:
            nxt += 1
        out[j] = nxt & 0xFFFFFFFF
        used.add(int(out[j]))
    return out


class Context:
    """model.Context (main.pyx:1746-2101) over the CUDA engine."""

    # places of infection in transmission_settings() / infection_places(): the contact places, then the roots
    PLACE_NAMES = [CONTACT_PLACE_TO_STR[i] for i in range(_abi.RB_N_PLACES)] + ['imported/initial']

    def __init__(self, population_params, healthcare_params, disease_params, start_date,
                 random_seed=4321, n_replicas=1, device=0, max_days=600, contact_capacity=0.0,
                 shard=None, _library=None):
        lib = _library if _library is not None else _abi.cuda_library()
        ipc = population_params.pop('initial_population_condition', None)   # main.pyx:1765 (mutates, as the reference)

        age_structure = population_params['age_structure']
        items = list(age_structure.items())
        n_ages = int(max(a for a, _ in items)) + 1           # main.pyx:1355
        age_counts = np.zeros(n_ages, dtype=np.int64)
        for a, c in items:
            age_counts[int(a)] = int(c)
        if n_ages > _abi.RB_MAX_AGES:
            raise ValueError('more than %d ages' % _abi.RB_MAX_AGES)
        n_agents = int(age_counts.sum())
        if n_agents >= 2 ** 31:
            raise ValueError('population does not fit int32 indices (main.pyx:28)')

        # Disease(params): wild-type + variants (main.pyx:868-881)
        self.variant_names = ['wild-type']
        variants = [make_variant(disease_params, n_ages)]
        for var in disease_params['variants']:
            vp = dict(disease_params)
            vp.update(var)
            variants.append(make_variant(vp, n_ages))
            self.variant_names.append(var['name'])
        if len(variants) > _abi.RB_MAX_VARIANTS:
            raise ValueError('more than %d variants' % _abi.RB_MAX_VARIANTS)

        self.age_group_labels = list(population_params['age_groups']['labels'])
        group_of_age = np.asarray(population_params['age_groups']['age_indices'], dtype=np.int32)
        assert len(group_of_age) >= n_ages

        # imported_infection_ages -> cumulative classes (main.pyx:1376-1384, :1632-1650)
        ages = population_params['imported_infection_ages']
        wsum = sum(x[1] for x in ages)
        cum, total = [], 0.0
        for _, w in ages:
            w = w / wsum
            cum.append(f32(w + total))
            total += w
        lo = [int(a) for a, _ in ages]
        hi = [lo[i + 1] - 1 for i in range(len(lo) - 1)] + [n_ages - 1]

        cfg = Config()
        cfg.n_agents, cfg.n_ages, cfg.n_groups = n_agents, n_ages, len(self.age_group_labels)
        cfg.n_variants, cfg.n_replicas = len(variants), int(n_replicas)
        cfg.seed = int(random_seed) & 0xFFFFFFFF
        cfg.hospital_beds = int(healthcare_params['hospital_beds'])
        cfg.icu_units = int(healthcare_params['icu_units'])
        cfg.max_days, cfg.n_import_classes, cfg.device = int(max_days), len(lo), int(device)
        cfg.contact_capacity = float(contact_capacity)
        self._engine = _abi.Engine(lib, cfg, age_counts, group_of_age[:n_ages], variants, lo, hi, cum)
        if ipc is not None and ipc.has_initial_state():      # main.pyx:1780-1781
            self._engine.set_initial_state([getattr(ipc, k) for k in
                                            ('dead', 'in_icu', 'in_ward', 'confirmed_cases', 'incubating', 'ill', 'recovered')])
        if shard is not None:
            # population-sharded mode: shard = (rank, nranks, nccl_unique_id[, exchange_capacity]); every rank builds the
            # same Context (same inputs, interventions and seed) on its own GPU and makes the same calls
            self._engine.shard_init(int(shard[0]), int(shard[1]), shard[2], float(shard[3]) if len(shard) > 3 else 0.0)

        self.n_agents, self.n_ages, self.n_replicas = n_agents, n_ages, int(n_replicas)
        self._group_of_age = group_of_age[:n_ages].copy()
        self._age_start = np.concatenate([[0], np.cumsum(age_counts)])      # agents are stored age-sorted
        self.max_days = int(max_days)
        self.start_date = start_date
        self.day = 0
        self.interventions = []
        self._direct = []       # apply_intervention() calls made directly by the caller, with the day they were made on
        self._contacts_per_day = ContactMatrix._records(population_params['contacts_per_day'])
        self._n_variants = len(variants)
        self._reset_host_state()
        self._state_day = -1    # day whose stats row is known to be on the device

    def _reset_host_state(self):
        """Host half of a fresh Context: HealthcareSystem / Population settings and the contact matrix."""
        self.contact_matrix = ContactMatrix(self._contacts_per_day, self.n_ages)
        for entry in self._direct:
            entry[2] = False
        # HealthcareSystem host-side settings (main.pyx:461-471)
        self._testing_mode = NO_TESTING
        self._p_detected_anyway = f32(0)
        self._p_successful_tracing = f32(1.0)
        self._vaccinations = []
        # Population import settings (main.pyx:1366-1369)
        self._weekly_amount = 0
        self._weekly_leftover = [0.0] * (self._n_variants + 1)
        self._weekly_shares = [0.0] * self._n_variants
        self._weekly_shares[0] = 1.0
        # pending one-day effects collected by apply_intervention
        self._pending = dict(beds=0, icu=0, imports=[])
        self._epoch = 0
        self._epoch_mobility = {0: 1 - float(self.contact_matrix.mobility_factor)}
        self._tables = {0: self.contact_matrix.generate()}
        self._engine.set_contact_table(0, self._tables[0])
        self._plan = []         # DayParams of every day planned so far (the schedule does not depend on the seed)

    # -- reference surface ------------------------------------------------------------------------
    def get_date_for_today(self):                      # main.pyx:1806-1808
        d = date.fromisoformat(self.start_date)
        return (d + timedelta(days=self.day)).isoformat()

    def add_intervention(self, iv):                    # main.pyx:1810-1811
        self._replan_from_today()
        self.interventions.append(iv)

    def _replan_from_today(self):
        """Days beyond today may have been planned ahead (after reset() / load_state(), the schedule is kept because it
        does not depend on the seed): drop them, so that a change made now takes effect from today's iterate() on."""
        if len(self._plan) > self.day:
            done = self.day
            self._reset_host_state()
            for _ in range(done):
                self._plan_next_day()

    def find_variant(self, variant_str):               # main.pyx:1868-1878
        if variant_str is None:
            return 0
        for idx, vn in enumerate(self.variant_names):
            if variant_str == vn:
                return idx
        raise Exception('Variant %s not found' % variant_str)

    def apply_intervention(self, iv):                  # main.pyx:1880-1960
        """Part of the reference surface (calc/simulation.py:321 calls it directly): takes effect immediately, i.e. from
        the next iterate() on.  The host keeps it with the day it was made on, so that re-planning replays it."""
        self._replan_from_today()
        self._apply(iv)                                # raises for an unknown type, like the reference
        self._direct.append([self.day, iv, True])      # [day, intervention, applied to the current host state]

    def _apply(self, iv):
        params = iv.get_param_values()
        t = iv.type
        if t == 'test-all-with-symptoms':
            self._set_testing_mode(ALL_WITH_SYMPTOMS)
        elif t == 'test-only-severe-symptoms':
            self._set_testing_mode(ONLY_SEVERE_SYMPTOMS, params['mild_detection_rate'] / 100.0)
        elif t == 'test-with-contact-tracing':
            self._set_testing_mode(ALL_WITH_SYMPTOMS_CT, params['efficiency'] / 100.0)
        elif t == 'build-new-icu-units':
            self._pending['icu'] += params['units']
        elif t == 'build-new-hospital-beds':
            self._pending['beds'] += params['beds']
        elif t == 'import-infections':
            # infects immediately in the reference (main.pyx:1897-1899): the new cases get an infectee list iff contact
            # tracing is the testing mode at THIS point of the day's intervention list (person_infect, :227-233)
            self._pending['imports'].append((int(params['amount']), self.find_variant(params.get('variant')),
                                             self._testing_mode == ALL_WITH_SYMPTOMS_CT))
        elif t == 'import-infections-weekly':
            shares = [0] * len(self.variant_names)
            for pn in params.keys():
                if not pn.startswith('variant_'):
                    continue
                vid = self.find_variant(pn.replace('variant_', ''))
                share = params[pn]
                shares[vid] = share / 100 if share else 0
            shares[0] = 1 - sum(shares)
            self._weekly_amount = int(params['weekly_amount'])
            self._weekly_shares = shares
        elif t == 'limit-mobility':
            reduction = (100 - params['reduction']) / 100.0
            place = params.get('place')
            self.contact_matrix.set_mobility_factor(
                factor=reduction, min_age=params.get('min_age'), max_age=params.get('max_age'),
                place=None if place is None else _STR_TO_PLACE[place])
        elif t == 'wear-masks':
            place = params.get('place')
            self.contact_matrix.set_mask_probability(
                p=params['share_of_contacts'] / 100.0, min_age=params.get('min_age'),
                max_age=params.get('max_age'), place=None if place is None else _STR_TO_PLACE[place])
        elif t == 'vaccinate':
            self._start_vaccinating(params['weekly_vaccinations'] / 7, params.get('min_age'), params.get('max_age'))
        else:
            raise Exception()

    def iterate(self):                                 # main.pyx:2011-2018
        self.run(1)

    def generate_state(self, replica=0):               # main.pyx:1813-1857
        if self._state_day != self.day:
            self._engine.snapshot()
            self._engine.sync()
            self._state_day = self.day
        row = self._engine.read_stats(self.day, 1)[replica, 0]
        return self._row_to_state(row)

    def get_population_stats(self, what, replica=0):   # main.pyx:1859-1866
        if what not in ('dead', 'all_infected', 'all_detected'):
            raise Exception()
        self._engine.sync()
        return self._engine.read_per_age(replica, ATTRS.index(what))

    def sample(self, what, age, severity=None):        # main.pyx:2047-2101
        if what == 'infectiousness':
            # broken in the reference itself (calls a method that does not exist, main.pyx:2068)
            days = list(range(-100, 100))
            iot = dict(INFECTIOUSNESS_OVER_TIME)
            vals = [iot.get(d, 0.0) for d in days]
            return np.rec.fromarrays((days, vals), names=('day', 'val'))
        if what not in SAMPLE_KINDS:
            raise Exception('unknown sample type. supported: %s' % ', '.join(['infectiousness'] + list(SAMPLE_KINDS)))
        sev = STR_TO_SEVERITY[severity] if severity is not None else 1
        return self._engine.sample(SAMPLE_KINDS[what], int(age), sev, 10000)

    # -- extensions -------------------------------------------------------------------------------
    def run(self, days):
        """`days` x iterate() in one device-resident run (the per-day schedule is computed up front)."""
        self._prepare_run(days)
        self._launch_run(days)
        self._finish_run()

    # run() in three parts, for callers that drive several engines at once (sharded.run_local): everything that may
    # allocate, upload or synchronise first; then the asynchronous launches; then the wait and the error check.
    def _prepare_run(self, days):
        if self.day + days > self.max_days:
            raise ValueError('max_days=%d exceeded' % self.max_days)
        while len(self._plan) < self.day + days:
            self._plan_next_day()
        self._engine.set_schedule(self.day, self._plan[self.day:self.day + days])

    def _launch_run(self, days):
        self._engine.step(days)
        self.day += days

    def _finish_run(self):
        self._engine.sync()
        problems = self._engine.problem()
        if problems.any():                              # main.pyx:2017-2018
            raise SimulationFailed(PROBLEM_TO_STR.get(int(problems[problems != 0][0]), 'Other failure'))

    def series(self, day0=0, days=None):
        """Raw stats rows [replica, day, row] for days [day0, day0+days) (rows of completed days)."""
        days = self.day - day0 if days is None else days
        self._engine.sync()
        return self._engine.read_stats(day0, days)

    def moments(self, day0=0, days=None, reduce=False):
        """Ensemble moments reduced on the device: (sum, sum of squares, n_replicas) of every stats column per day.
        reduce=True sums them over the ranks of the engine's NCCL communicator as well (rb_reduce_moments)."""
        days = self.day - day0 if days is None else days
        if reduce:
            return self._engine.reduce_moments(day0, days)
        s1, s2 = self._engine.read_moments(day0, days)
        return s1, s2, self.n_replicas

    def transmission_stats(self):
        """Who infected whom and when, per replica, from the infection tree of the current state (k_transmission; all
        arrays int64 with a leading replica axis):

          cohort_infected[r, d]    agents infected on day d, d = 0 .. today
          cohort_offspring[r, d]   the people those agents have infected so far
          cohort_open[r, d]        those agents still incubating or ill, i.e. still able to infect: while it is not 0 the
                                   cohort's offspring count can grow (right-censored)
          offspring_hist[r, k]     closed cases (no longer able to infect) that infected k people; k = 64 means >= 64
          generation_interval_hist[r, k]   infected agents whose infector was infected k days earlier (64: >= 64)
          group_closed / group_offspring[r, g]       closed cases and their offspring by age group (age_group_labels)
          variant_closed / variant_offspring[r, v]   the same by variant (variant_names)

        ensemble.transmission_summary() turns these into cohort reproduction numbers, dispersion and the
        generation-interval distribution."""
        t = self._engine.transmission_stats().astype(np.int64)
        M, B, G, V = self.max_days + 1, _abi.RB_TX_BINS, len(self.age_group_labels), _abi.RB_MAX_VARIANTS
        parts, k = {}, 0
        for name, n in (('cohort_infected', M), ('cohort_offspring', M), ('cohort_open', M), ('offspring_hist', B),
                        ('generation_interval_hist', B), ('group_closed', G), ('group_offspring', G),
                        ('variant_closed', V), ('variant_offspring', V)):
            parts[name] = t[:, k:k + n]
            k += n
        assert k == t.shape[1]
        for name in ('cohort_infected', 'cohort_offspring', 'cohort_open'):
            parts[name] = parts[name][:, :self.day + 1]
        for name in ('variant_closed', 'variant_offspring'):
            parts[name] = parts[name][:, :len(self.variant_names)]
        return parts

    def transmission_tree(self, replica=0):
        """The line list of one replica: every agent infected so far, as arrays agent (index), infector (-1 for imports
        and the initial state), day (of infection) and age."""
        days = self._engine.read_infection_days(replica)
        agent = np.flatnonzero(days >= 0)
        infector = self._engine.read_agents(replica)['infector'][agent]
        age = np.searchsorted(self._age_start, agent, side='right') - 1
        return dict(agent=agent.astype(np.int64), infector=infector.astype(np.int64), day=days[agent].astype(np.int64),
                    age=age.astype(np.int64))

    def _epoch_of_day(self):
        # the contact-table epoch of every completed day, from the plan (load_state replays it; the device keeps no
        # schedule of the days before a load)
        return np.array([dp.table_epoch for dp in self._plan[:self.day]], dtype=np.int32)

    def transmission_settings(self):
        """Where infections happened and who infected whom, per replica, from the infection tree of the current state
        (k_transmission_settings; all arrays int64 with a leading replica axis, places in PLACE_NAMES order):

          by_day_place[r, d, p]       agents infected on day d (d = 0 .. today) at place p; p = 6 (RB_PLACE_ROOT) are
                                      imports and the initial state
          pair_all[r, p, i, j]        infections at place p of a person of age group j by one of age group i
          pair_closed[r, p, i, j]     the same, only by infectors that can no longer infect (closed cases)
          closed_by_group[r, i]       closed cases of age group i: the denominator of the next-generation matrix

        ensemble.setting_summary() turns these into shares by place, the next-generation matrix and its spectral
        radius with and without each place."""
        t = self._engine.transmission_settings(self._epoch_of_day()).astype(np.int64)
        R, M, P, G = self.n_replicas, self.max_days + 1, _abi.RB_N_PLACES, len(self.age_group_labels)
        k0, k1, k2 = M * (P + 1), M * (P + 1) + P * G * G, M * (P + 1) + 2 * P * G * G
        assert t.shape[1] == k2 + G
        return dict(by_day_place=t[:, :k0].reshape(R, M, P + 1)[:, :self.day + 1],
                    pair_all=t[:, k0:k1].reshape(R, P, G, G), pair_closed=t[:, k1:k2].reshape(R, P, G, G),
                    closed_by_group=t[:, k2:])

    def infection_places(self, replica=0):
        """Place of infection (index into PLACE_NAMES) of every agent of transmission_tree(replica)['agent'], in that
        order: 0..5 the contact's place, 6 an import or the initial state."""
        p = self._engine.read_infection_places(replica, self._epoch_of_day())
        return p[p >= 0].astype(np.int64)

    def branch(self, source, seeds=None):
        """Many futures of one present (rb_branch): replica j continues from the current state of replica source[j] --
        agents, infection tree, test queue, counters and its stats rows so far -- and draws with its own seed from the
        next iterate() on.  `source` is an int array of length n_replicas, or one int: every replica from that one.  A
        replica that is copied from keeps its own state (source[source[j]] == source[j]).

        seeds None: every replica whose state changes (source[j] != j) gets a seed this engine has never used, the others
        keep theirs; else an array of n_replicas seeds (a copy given its source's seed continues exactly as the source).
        Returns the seeds now in force.  Rows of days before today are the source's; today's row is written by the next
        iterate() or generate_state()."""
        R = self.n_replicas
        src = np.full(R, int(source), dtype=np.int64) if np.ndim(source) == 0 else np.asarray(source, dtype=np.int64)
        if src.shape != (R,):
            raise ValueError('source must be one int or %d ints' % R)
        if seeds is None:
            hist = self._engine.read_seeds()
            seeds = hist[:, self.day].copy()
            changed = np.flatnonzero(src != np.arange(R))
            seeds[changed] = fresh_seeds(hist, changed.size)
        seeds = np.asarray(seeds, dtype=np.int64)
        if seeds.shape != (R,) or (seeds < 0).any() or (seeds > 0xFFFFFFFF).any():
            raise ValueError('seeds must be %d unsigned 32-bit ints' % R)
        self._engine.branch(src, seeds.astype(np.uint32))
        self._state_day = -1
        return seeds.astype(np.uint32)

    # -- moving replicas between Contexts, engines and GPUs --------------------------------------------------------
    def _check_movable(self, other):
        """Refuses two Contexts the engines cannot tell apart but a moved replica would notice: a different schedule of
        the days run so far, or different contact tables of those days' epochs (inputs, not state)."""
        if other.day != self.day:
            raise ValueError('the Contexts are at days %d and %d' % (self.day, other.day))
        if len(self._plan) < self.day or len(other._plan) < other.day or \
                any(bytes(a) != bytes(b) for a, b in zip(self._plan[:self.day], other._plan[:other.day])):
            raise ValueError('the Contexts ran different schedules (interventions) so far')
        for ep in sorted({0} | {dp.table_epoch for dp in self._plan[:self.day]}):
            a, b = self._tables.get(ep), other._tables.get(ep)
            if a is None or b is None or a.keys() != b.keys() or any(not np.array_equal(a[k], b[k]) for k in a):
                raise ValueError('the Contexts use different contact tables (epoch %d)' % ep)

    def _import_seeds(self, slots, seeds, foreign_hist):
        """The seeds of written slots: as given, or (None) seeds neither this engine nor the incoming replicas' seed
        histories ever used -- Context.branch's rule over both."""
        if seeds is None:
            hist = self._engine.read_seeds()
            seeds = fresh_seeds(np.concatenate([hist, foreign_hist.reshape(-1, hist.shape[1])]), len(slots))
        seeds = np.asarray(seeds, dtype=np.int64)
        if seeds.shape != (len(slots),) or (seeds < 0).any() or (seeds > 0xFFFFFFFF).any():
            raise ValueError('seeds must be %d unsigned 32-bit ints' % len(slots))
        return seeds.astype(np.uint32)

    def export_replicas(self, idx):
        """Replica records (rb_export_replicas) of replicas `idx`: uint8 [len(idx), record bytes].  Everything a replica
        needs to continue -- agents, infection tree, test queue, counters, sweep-order keys, stats rows so far and its
        seed history, which ends every record -- for import_replicas() into a Context built the same way, at the same day,
        in this process or another one."""
        return self._engine.export_replicas(np.atleast_1d(np.asarray(idx, dtype=np.int64)))

    def import_replicas(self, slots, records, seeds=None):
        """Write export_replicas() records into `slots` (rb_import_replicas): each slot continues from its record with
        seed seeds[j] from today on (the record's own seed: exactly as the replica it came from).  seeds None: seeds
        that neither this engine nor the records' seed histories have used.  Returns the seeds given."""
        slots = np.atleast_1d(np.asarray(slots, dtype=np.int64))
        rec = np.ascontiguousarray(records, dtype=np.uint8).reshape(len(slots), -1) if len(slots) else np.zeros((0, 0), np.uint8)
        foreign = rec[:, rec.shape[1] - 4 * (self.max_days + 1):].copy().view(np.uint32) if len(slots) else np.zeros((0, self.max_days + 1), np.uint32)
        seeds = self._import_seeds(slots, seeds, foreign)
        self._engine.import_replicas(slots, seeds, rec)
        self._state_day = -1
        return seeds

    def copy_replicas_from(self, other, src_idx, slots, seeds=None):
        """Replicas src_idx of Context `other` (another Context of this process, on this GPU or another one) into
        `slots` of this one, device to device (rb_copy_replicas); seeds as in import_replicas().  Returns the seeds
        given."""
        if other is self:
            raise ValueError('copy_replicas_from: the same Context (Context.branch copies within one)')
        self._check_movable(other)
        src_idx = np.atleast_1d(np.asarray(src_idx, dtype=np.int64))
        slots = np.atleast_1d(np.asarray(slots, dtype=np.int64))
        if src_idx.shape != slots.shape:
            raise ValueError('src_idx and slots differ in length')
        seeds = self._import_seeds(slots, seeds, other._engine.read_seeds() if seeds is None else np.zeros((0, self.max_days + 1), np.uint32))
        self._engine.copy_replicas_from(other._engine, src_idx, slots, seeds)
        self._state_day = -1
        return seeds

    def replica_seeds(self):
        """The seed every replica draws with from today on (random_seed + r until a branch changes it)."""
        return self._engine.read_seeds()[:, self.day].copy()

    def set_transmission_scale(self, values):
        """Every replica's transmission scale f (rb_set_transmission_scale): one value for all replicas or n_replicas
        values, each finite and in (0, 16].  Replica r's infectors then transmit with probability min(1, f_r p) where
        they would with p, at every place and for every variant, from the next iterate() on.  The scale is part of the
        replica's state: branch(), export / import, copy_replicas_from() and save_state() / load_state() carry it, and
        reset() and a fresh Context give 1.  Refused values raise EngineError and change nothing."""
        R = self.n_replicas
        v = np.full(R, values, dtype=np.float64) if np.ndim(values) == 0 else np.asarray(values, dtype=np.float64)
        if v.shape != (R,):
            raise ValueError('transmission scale: one value or %d values' % R)
        with np.errstate(over='ignore'):                  # a value beyond float32 becomes inf, which the engine refuses
            self._engine.set_transmission_scale(v.astype(np.float32))

    def transmission_scale(self):
        """float32 [n_replicas]: the scales in force, as the engine applies them (1 + (f - 1) in float: f itself for
        0.5 <= f <= 2)."""
        return self._engine.read_transmission_scale()

    def set_severity_scale(self, severe=None, critical=None, fatal=None):
        """Every replica's severity scales (rb_set_severity_scale), column by column: each argument is None (keep the
        scales in force), one value for all replicas or n_replicas values, each finite and in (0, 16].  Where an
        infection's severity is drawn -- transmissions, imports and the initial state (rb_set_initial_state, which reads
        the scales when it runs) -- the wild-type variant's conditional probabilities of the infected age become
        min(x s, max(x, 1)): p_severe times `severe`, p_critical times `critical`, and both p_fatal and
        p_death_outside_hospital times `fatal`, in force from the next iterate() on.  A scaled probability never passes 1
        unless the table's already does, and a scale of 1 draws exactly as an unscaled Context does.  `severe` moves
        in_ward, `critical` in_icu and `fatal` dead; FATAL is nested inside CRITICAL and every FATAL case dies outside
        hospital, so raising `fatal` turns critical cases into deaths and in_icu falls.  sample('symptom_severity') stays
        unscaled.  The scales are part of the replica's state: branch(), export / import, copy_replicas_from() and
        save_state() / load_state() carry them, and reset() and a fresh Context give 1.  The full [n_replicas, 3] is
        built from severity_scale() and the given columns and set in one engine call: refused values raise EngineError
        and change nothing, the columns left as None included."""
        R = self.n_replicas
        s = self.severity_scale().astype(np.float64)
        for j, values in enumerate((severe, critical, fatal)):
            if values is None:
                continue
            v = np.full(R, values, dtype=np.float64) if np.ndim(values) == 0 else np.asarray(values, dtype=np.float64)
            if v.shape != (R,):
                raise ValueError('severity scale %s: one value or %d values' % (SEVERITY_SCALES[j], R))
            s[:, j] = v
        with np.errstate(over='ignore'):                  # a value beyond float32 becomes inf, which the engine refuses
            self._engine.set_severity_scale(s.astype(np.float32))

    def severity_scale(self):
        """float32 [n_replicas, 3]: the severe, critical and fatal scales in force (SEVERITY_SCALES order), as the engine
        applies them (1 + (s - 1) in float)."""
        return self._engine.read_severity_scale()

    def row_layout(self):
        G = len(self.age_group_labels)
        names = ['%s[%s]' % (a, g) for a in ATTRS for g in self.age_group_labels]
        names += _abi.SCALARS + ['exposures_%s' % CONTACT_PLACE_TO_STR[i] for i in range(_abi.RB_N_PLACES)]
        names += ['infected_by_variant_%d' % i for i in range(_abi.RB_MAX_VARIANTS)]
        assert len(names) == len(ATTRS) * G + _abi.RB_N_SCALARS
        return names

    def reset(self, random_seed):
        """A fresh Context(random_seed=...) with the same inputs and interventions, without reallocating
        device memory.  The planned schedule is kept (it does not depend on the seed); interventions applied directly
        with apply_intervention() belong to the old run and are dropped."""
        if self._direct:
            self._direct = []
            self._reset_host_state()
        self._engine.reset(random_seed)
        self.day = 0
        self._state_day = -1

    def save_state(self):
        """Checkpoint: the engine's whole device state between two iterate() calls as one uint8 array (np.save it).
        Interventions, inputs and max_days are not part of it: load it into a Context built the same way."""
        return self._engine.save_state()

    def load_state(self, blob):
        """Resume from a save_state() blob: this Context continues at the saved day."""
        self._engine.load_state(blob)
        self.day = self._engine.day()
        self._state_day = -1
        while len(self._plan) < self.day:         # replays the host half (interventions, contact tables) up to that day
            self._plan_next_day()

    def upload_inputs(self):
        """Re-send every contact table to the device (bench.py: per-step host->device input copy)."""
        for epoch, t in self._tables.items():
            self._engine.set_contact_table(epoch, t)
        return sum(sum(a.nbytes for a in t.values()) for t in self._tables.values())

    def close(self):
        self._engine.close()

    # -- internals --------------------------------------------------------------------------------
    def _set_testing_mode(self, mode, p=1.0):           # main.pyx:623-628
        self._testing_mode = mode
        if mode == ALL_WITH_SYMPTOMS_CT:
            self._p_successful_tracing = f32(p)
        elif mode == ONLY_SEVERE_SYMPTOMS:
            self._p_detected_anyway = f32(p)

    def _start_vaccinating(self, daily, min_age, max_age):   # main.pyx:585-593
        for v in self._vaccinations:
            if min_age != v.get('min_age') or max_age != v.get('max_age'):
                continue
            break
        else:
            v = dict(min_age=min_age, max_age=max_age, slot=len(self._vaccinations))
            if v['slot'] >= _abi.RB_MAX_VACC:
                raise ValueError('more than %d vaccination programmes' % _abi.RB_MAX_VACC)
            self._vaccinations.append(v)
        v['nr_daily'] = daily

    def _plan_next_day(self):
        """Host half of one iterate(): interventions dated that day (main.pyx:2012-2015), then the settings
        Population.init_day (:1687-1699) and HealthcareSystem.iterate (:547-558) read.  Appends to the plan."""
        index = len(self._plan)
        today = (date.fromisoformat(self.start_date) + timedelta(days=index)).isoformat()
        for entry in self._direct:                     # re-planning: direct apply_intervention() calls made before that day's iterate()
            if entry[0] == index and not entry[2]:
                self._apply(entry[1])
                entry[2] = True
        for iv in self.interventions:
            if iv.date == today:
                self._apply(iv)
        dp = DayParams()
        dp.testing_mode = self._testing_mode
        dp.p_detected_anyway = self._p_detected_anyway
        dp.p_successful_tracing = self._p_successful_tracing
        dp.beds_delta, dp.icu_delta = self._pending['beds'], self._pending['icu']
        imports = self._pending['imports']
        if len(imports) > _abi.RB_MAX_IMPORT_EVENTS:
            raise ValueError('more than %d import events on one day' % _abi.RB_MAX_IMPORT_EVENTS)
        dp.n_imports = len(imports)
        dp.import_traced = 0
        for i, (amount, variant, traced) in enumerate(imports):
            dp.import_amount[i], dp.import_variant[i] = amount, variant
            dp.import_traced |= int(bool(traced)) << i
        self._pending = dict(beds=0, icu=0, imports=[])
        # ContactMatrix.init_day, main.pyx:1285-1288
        cm = self.contact_matrix
        if cm.mobility_factor_changed:
            self._epoch += 1
            self._tables[self._epoch] = cm.generate()
            self._engine.set_contact_table(self._epoch, self._tables[self._epoch])
            self._epoch_mobility[self._epoch] = 1 - float(cm.mobility_factor)
            cm.mobility_factor_changed = False
        dp.table_epoch = self._epoch
        # infect_people_daily, main.pyx:1671-1685 (C float accumulator, Python-float arithmetic)
        for vid in range(len(self.variant_names)):
            leftover = f32(self._weekly_leftover[vid])
            leftover = f32(float(leftover) + self._weekly_amount / 7.0 * self._weekly_shares[vid])
            amount_today = int(leftover)
            if amount_today:
                leftover = f32(leftover - f32(amount_today))
            assert leftover >= 0
            self._weekly_leftover[vid] = float(leftover)
            dp.trickle[vid] = amount_today
        # vaccination programmes, main.pyx:547-558
        n = 0
        for v in self._vaccinations:
            if not v['nr_daily']:
                continue
            dp.vacc_nr[n] = int(v['nr_daily'])
            dp.vacc_min_age[n] = 0 if v['min_age'] is None else int(v['min_age'])
            dp.vacc_max_age[n] = self.n_ages - 1 if v['max_age'] is None else int(v['max_age'])
            dp.vacc_slot[n] = v['slot']
            n += 1
        dp.n_vacc = n
        self._plan.append(dp)
        return dp

    def _row_to_state(self, row):
        G = len(self.age_group_labels)
        sc = row[len(ATTRS) * G:]
        S = {name: int(sc[i]) for i, name in enumerate(_abi.SCALARS)}
        r = S['total_infections'] / S['total_infectors'] if S['total_infectors'] > 5 else 0   # main.pyx:1817
        s = dict(
            available_icu_units=S['available_icu_units'],
            available_hospital_beds=S['available_hospital_beds'],
            total_icu_units=S['total_icu_units'],
            r=r,
            exposed_per_day=S['exposed_per_day'],
            ct_cases_per_day=S['ct_cases_per_day'],
            mobility_limitation=self._epoch_mobility_for_row(S),
        )
        for i, attr in enumerate(ATTRS):
            s[attr] = np.array(row[i * G:(i + 1) * G], dtype=np.int32)
        s['infected_by_variant'] = {self.variant_names[i]: int(sc[_abi.RB_S_VARIANT0 + i])
                                    for i in range(len(self.variant_names))}
        s['daily_contacts'] = {CONTACT_PLACE_TO_STR[i]: int(sc[_abi.RB_S_CONTACTS0 + i])
                               for i in range(_abi.RB_N_PLACES)}
        return s

    def _epoch_mobility_for_row(self, S):
        # mobility_limitation = 1 - (last factor passed to set_mobility_factor), main.pyx:1251,1842; the
        # value changes on the day the intervention is applied, i.e. with the table epoch of that day
        return self._epoch_mobility.get(S['table_epoch'], 0.0)
