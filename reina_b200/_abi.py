"""ctypes mirror of include/reina_b200.h.

`Engine` binds one shared library that exports the C-ABI with a given prefix: the product binds
`libreina_b200.so` (prefix `rb_`, CUDA); tests bind the CPU oracle (`ro_`) through the very same class
to compare the two on identical inputs.  Nothing in this package ever loads the oracle.
"""
import ctypes as C
import os

import numpy as np

RB_MAX_AGES = 128
RB_MAX_VARIANTS = 4
RB_MAX_ROWS = 96
RB_NCDF = 100
RB_MAX_IMPORT_EVENTS = 8
RB_MAX_VACC = 8
RB_MAX_IMPORT_CLASSES = 16
RB_N_PLACES = 6
RB_IOT_LEN = 21
RB_N_TABLES = 6
RB_TX_BINS = 65      # offspring / generation-interval histograms: bins 0..63 and ">= 64"
RB_PLACE_ROOT = RB_N_PLACES   # place index of imports and the initial state (no infector)

ATTRS = ['susceptible', 'vaccinated', 'infected', 'all_infected', 'detected', 'all_detected',
         'in_icu', 'cum_icu', 'in_ward', 'dead', 'recovered', 'non_hospital_deaths', 'new_infections']
RB_N_ATTRS = len(ATTRS)
SCALARS = ['available_icu_units', 'available_hospital_beds', 'total_icu_units', 'total_hospital_beds',
           'total_infections', 'total_infectors', 'exposed_per_day', 'ct_cases_per_day', 'table_epoch',
           'day']
RB_S_CONTACTS0 = len(SCALARS)
RB_S_VARIANT0 = RB_S_CONTACTS0 + RB_N_PLACES
RB_N_SCALARS = RB_S_VARIANT0 + RB_MAX_VARIANTS

T_SUSCEPTIBILITY, T_SYMPTOMATIC, T_SEVERE, T_CRITICAL, T_FATAL, T_DEATH_OUTSIDE_HOSPITAL = range(6)


class Variant(C.Structure):
    _fields_ = [
        ('p_icu_death_no_beds', C.c_float), ('p_hospital_death_no_beds', C.c_float),
        ('infectiousness_multiplier', C.c_float), ('p_asymptomatic_infection', C.c_float),
        ('p_mask_protects_wearer', C.c_float), ('p_mask_protects_others', C.c_float),
        ('ratio_before_hospitalisation', C.c_float), ('ratio_in_ward', C.c_float),
        ('incubation_kappa', C.c_float), ('incubation_theta', C.c_float),
        ('onset_death_kappa', C.c_float), ('onset_death_theta', C.c_float),
        ('onset_recovery_kappa', C.c_float), ('onset_recovery_theta', C.c_float),
        ('reserved', C.c_float * 2),
        ('iot', C.c_float * (RB_IOT_LEN + 3)),
        ('tab', (C.c_float * RB_MAX_AGES) * RB_N_TABLES),
    ]


class Config(C.Structure):
    _fields_ = [
        ('n_agents', C.c_int32), ('n_ages', C.c_int32), ('n_groups', C.c_int32),
        ('n_variants', C.c_int32), ('n_replicas', C.c_int32), ('seed', C.c_uint32),
        ('hospital_beds', C.c_int32), ('icu_units', C.c_int32), ('max_days', C.c_int32),
        ('n_import_classes', C.c_int32), ('device', C.c_int32), ('contact_capacity', C.c_float),
        ('reserved', C.c_int32 * 4),
    ]


class DayParams(C.Structure):
    _fields_ = [
        ('testing_mode', C.c_int32), ('p_detected_anyway', C.c_float),
        ('p_successful_tracing', C.c_float), ('beds_delta', C.c_int32), ('icu_delta', C.c_int32),
        ('table_epoch', C.c_int32), ('n_imports', C.c_int32),
        ('import_amount', C.c_int32 * RB_MAX_IMPORT_EVENTS),
        ('import_variant', C.c_int32 * RB_MAX_IMPORT_EVENTS),
        ('trickle', C.c_int32 * RB_MAX_VARIANTS), ('n_vacc', C.c_int32),
        ('vacc_nr', C.c_int32 * RB_MAX_VACC), ('vacc_min_age', C.c_int32 * RB_MAX_VACC),
        ('vacc_max_age', C.c_int32 * RB_MAX_VACC), ('vacc_slot', C.c_int32 * RB_MAX_VACC),
        ('import_traced', C.c_int32), ('reserved', C.c_int32 * 3),
    ]


AGENT_DTYPE = np.dtype([
    ('infector', '<i4'), ('n_infected', '<i4'), ('days_left', '<i2'), ('day_of_illness', '<i2'),
    ('day_of_vaccination', '<i2'), ('state', 'u1'), ('severity', 'u1'), ('variant', 'u1'),
    ('flags', 'u1'), ('ward_days', 'u1'), ('icu_days', 'u1')], align=True)
assert AGENT_DTYPE.itemsize == 20, AGENT_DTYPE.itemsize

_HERE = os.path.dirname(os.path.abspath(__file__))
# REINA_B200_LIB: measurement aid (tools/variants.sh builds the library with different tuning macros)
CUDA_LIB_PATH = os.environ.get('REINA_B200_LIB') or os.path.join(_HERE, 'libreina_b200.so')

SYMBOLS = ['create', 'destroy', 'reset', 'set_initial_state', 'step_profiled', 'set_contact_table', 'set_schedule', 'step', 'sync', 'day',
           'snapshot', 'row_len', 'read_stats', 'read_moments', 'read_per_age', 'problem', 'sample', 'read_agents',
           'read_queue', 'read_available', 'last_step_ms', 'launch_count', 'last_error', 'rng_block']


# transmission statistics from the infection tree; their CPU reference is test code (tests/oracle_transmission.c)
TX_SYMBOLS = ['transmission_len', 'transmission_stats', 'read_infection_days']
# the same tree by place of infection and age group; CPU reference: tests/oracle_settings.c (which includes the above)
SX_SYMBOLS = ['transmission_settings_len', 'transmission_settings', 'read_infection_places']
# branching replicas from the current state; CPU reference: tests/oracle_branch.c (which includes the above)
BRANCH_SYMBOLS = ['branch', 'read_seeds']
# replica records moved between engines; CPU reference: tests/oracle_migrate.c (which includes the above).  The NCCL move
# is CUDA only.
MIGRATE_SYMBOLS = ['replica_bytes', 'export_replicas', 'import_replicas', 'copy_replicas']
# the per-replica transmission scale; CPU reference: tests/oracle_tscale.c (which includes the above)
TSCALE_SYMBOLS = ['set_transmission_scale', 'read_transmission_scale']
# the per-replica severity scales; CPU reference: tests/oracle_sscale.c (which includes the above)
SSCALE_SYMBOLS = ['set_severity_scale', 'read_severity_scale']
# exported by the CUDA library only: population-sharded mode (the sequential CPU oracle has no ranks) and the rest below
SHARD_SYMBOLS = ['shard_unique_id', 'shard_init', 'shard_init_local', 'shard_rank', 'shard_nranks', 'shard_message_bytes', 'shard_exchange',
                 # checkpoint / resume of the device-resident state
                 'state_bytes', 'save_state', 'load_state',
                 # ensemble communicator (NCCL), production-geometry timing, measurement aids
                 'comm_init', 'comm_rank', 'comm_size', 'comm_allreduce', 'comm_allgather', 'reduce_moments',
                 'step_timed', 'debug_flag', 'debug_phase_cycles', 'copied_bytes', 'comm_move_replicas'] + TX_SYMBOLS + SX_SYMBOLS + BRANCH_SYMBOLS + MIGRATE_SYMBOLS + TSCALE_SYMBOLS + SSCALE_SYMBOLS
SH_SHIFT = 12      # ownership stripes of 4096 agents, dealt round-robin over the ranks (engine.cu owns())


def owner_of(agent_index, nranks):
    """Rank that owns (sweeps) each agent in population-sharded mode."""
    return (np.asarray(agent_index) >> SH_SHIFT) % nranks


class EngineError(RuntimeError):
    pass


def _ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


class Library:
    """A loaded shared library exporting the C-ABI under `prefix`."""

    def __init__(self, path, prefix):
        if not os.path.exists(path):
            raise EngineError(
                '%s not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                '(there is no CPU fallback)' % path)
        self.path, self.prefix = path, prefix
        self.dll = C.CDLL(path)
        f = {}
        for name in SYMBOLS:
            f[name] = getattr(self.dll, prefix + name)   # AttributeError if a symbol is missing
        vp = C.c_void_p
        f['create'].argtypes = [C.POINTER(Config), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.POINTER(Variant), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.POINTER(C.c_float), C.POINTER(vp)]
        f['destroy'].argtypes = [vp]
        f['destroy'].restype = None
        f['set_contact_table'].argtypes = [vp, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                           C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                           C.POINTER(C.c_uint8), C.POINTER(C.c_float),
                                           C.POINTER(C.c_double), C.POINTER(C.c_double)]
        f['set_schedule'].argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(DayParams)]
        f['step'].argtypes = [vp, C.c_int32]
        f['reset'].argtypes = [vp, C.c_uint32]
        f['set_initial_state'].argtypes = [vp, C.POINTER(C.c_int32)]
        f['step_profiled'].argtypes = [vp, C.c_int32, C.POINTER(C.c_float)]
        f['sync'].argtypes = [vp]
        f['day'].argtypes = [vp]
        f['day'].restype = C.c_int32
        f['snapshot'].argtypes = [vp]
        f['row_len'].argtypes = [vp]
        f['row_len'].restype = C.c_int32
        f['read_stats'].argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]
        f['read_moments'].argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        f['read_per_age'].argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]
        f['problem'].argtypes = [vp, C.POINTER(C.c_int32)]
        f['sample'].argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]
        f['rng_block'].argtypes = [C.c_int32, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        f['read_agents'].argtypes = [vp, C.c_int32, C.c_void_p]
        f['read_queue'].argtypes = [vp, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]
        f['read_available'].argtypes = [vp, C.c_int32, C.POINTER(C.c_int32)]
        f['last_step_ms'].argtypes = [vp]
        f['last_step_ms'].restype = C.c_float
        f['launch_count'].argtypes = [vp]
        f['launch_count'].restype = C.c_int64
        f['last_error'].argtypes = []
        f['last_error'].restype = C.c_char_p
        if prefix == 'rb_':
            for name in SHARD_SYMBOLS:
                f[name] = getattr(self.dll, prefix + name)
            f['shard_unique_id'].argtypes = [C.c_char_p]
            f['shard_init'].argtypes = [vp, C.c_int32, C.c_int32, C.c_char_p, C.c_float]
            f['shard_init_local'].argtypes = [C.POINTER(vp), C.c_int32, C.c_float]
            f['shard_rank'].argtypes = [vp]
            f['shard_nranks'].argtypes = [vp]
            f['shard_message_bytes'].argtypes = [vp]
            f['shard_message_bytes'].restype = C.c_int64
            f['shard_exchange'].argtypes = [vp]
            f['state_bytes'].argtypes = [vp]
            f['state_bytes'].restype = C.c_int64
            f['save_state'].argtypes = [vp, C.c_void_p, C.c_int64]
            f['load_state'].argtypes = [vp, C.c_void_p, C.c_int64]
            f['comm_init'].argtypes = [vp, C.c_int32, C.c_int32, C.c_char_p]
            f['comm_rank'].argtypes = [vp]
            f['comm_size'].argtypes = [vp]
            f['comm_allreduce'].argtypes = [vp, C.POINTER(C.c_double), C.c_int64, C.c_int32]
            f['comm_allgather'].argtypes = [vp, C.c_void_p, C.c_void_p, C.c_int64]
            f['reduce_moments'].argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]
            f['step_timed'].argtypes = [vp, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_float)]
            f['debug_flag'].argtypes = [vp, C.c_int32]
            f['debug_flag'].restype = None
            f['debug_phase_cycles'].argtypes = [vp, C.c_int32, C.c_void_p]
            f['copied_bytes'].argtypes = [vp, C.c_int32]
            f['copied_bytes'].restype = C.c_int64
            i32p = C.POINTER(C.c_int32)
            f['comm_move_replicas'].argtypes = [vp, C.c_int32, i32p, i32p, C.c_int32, i32p, i32p, C.POINTER(C.c_uint32)]
        self.f = f
        if prefix == 'rb_':
            self.bind_transmission()
            self.bind_settings()
            self.bind_branch()
            self.bind_migrate()
            self.bind_tscale()
            self.bind_sscale()

    def bind_transmission(self):
        """Bind the transmission-statistics entry points (the CUDA library exports them; a test library that adds them
        to the CPU oracle calls this itself)."""
        f, vp = self.f, C.c_void_p
        for name in TX_SYMBOLS:
            f[name] = getattr(self.dll, self.prefix + name)
        f['transmission_len'].argtypes = [vp]
        f['transmission_len'].restype = C.c_int32
        f['transmission_stats'].argtypes = [vp, C.POINTER(C.c_int32)]
        f['read_infection_days'].argtypes = [vp, C.c_int32, C.POINTER(C.c_int32)]

    def bind_settings(self):
        """Bind the entry points of the tables by place of infection and age group (like bind_transmission)."""
        f, vp = self.f, C.c_void_p
        for name in SX_SYMBOLS:
            f[name] = getattr(self.dll, self.prefix + name)
        f['transmission_settings_len'].argtypes = [vp]
        f['transmission_settings_len'].restype = C.c_int32
        f['transmission_settings'].argtypes = [vp, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]
        f['read_infection_places'].argtypes = [vp, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]

    def bind_branch(self):
        """Bind rb_branch / rb_read_seeds (like bind_transmission)."""
        f, vp = self.f, C.c_void_p
        for name in BRANCH_SYMBOLS:
            f[name] = getattr(self.dll, self.prefix + name)
        f['branch'].argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_uint32)]
        f['read_seeds'].argtypes = [vp, C.POINTER(C.c_uint32)]

    def bind_migrate(self):
        """Bind the replica-record entry points (like bind_transmission)."""
        f, vp, i32p = self.f, C.c_void_p, C.POINTER(C.c_int32)
        for name in MIGRATE_SYMBOLS:
            f[name] = getattr(self.dll, self.prefix + name)
        f['replica_bytes'].argtypes = [vp]
        f['replica_bytes'].restype = C.c_int64
        f['export_replicas'].argtypes = [vp, C.c_int32, i32p, vp, C.c_int64]
        f['import_replicas'].argtypes = [vp, C.c_int32, i32p, C.POINTER(C.c_uint32), vp, C.c_int64]
        f['copy_replicas'].argtypes = [vp, vp, C.c_int32, i32p, i32p, C.POINTER(C.c_uint32)]

    def bind_tscale(self):
        """Bind rb_set_transmission_scale / rb_read_transmission_scale (like bind_transmission)."""
        f, vp = self.f, C.c_void_p
        for name in TSCALE_SYMBOLS:
            f[name] = getattr(self.dll, self.prefix + name)
        f['set_transmission_scale'].argtypes = [vp, C.POINTER(C.c_float)]
        f['read_transmission_scale'].argtypes = [vp, C.POINTER(C.c_float)]

    def bind_sscale(self):
        """Bind rb_set_severity_scale / rb_read_severity_scale (like bind_transmission)."""
        f, vp = self.f, C.c_void_p
        for name in SSCALE_SYMBOLS:
            f[name] = getattr(self.dll, self.prefix + name)
        f['set_severity_scale'].argtypes = [vp, C.POINTER(C.c_float)]
        f['read_severity_scale'].argtypes = [vp, C.POINTER(C.c_float)]

    def check(self, rc, what):
        if rc != 0:
            raise EngineError('%s%s failed (%d): %s' % (
                self.prefix, what, rc, (self.f['last_error']() or b'').decode(errors='replace')))


_cuda_lib = None


def cuda_library():
    """The product library.  Raises if it has not been built -- there is no CPU fallback."""
    global _cuda_lib
    if _cuda_lib is None:
        _cuda_lib = Library(CUDA_LIB_PATH, 'rb_')
    return _cuda_lib


class Engine:
    """Thin object wrapper over one engine handle."""

    def __init__(self, lib, cfg, age_counts, group_of_age, variants, import_lo, import_hi, import_cum):
        self.lib = lib
        self.cfg = cfg
        self.n_agents, self.n_ages = cfg.n_agents, cfg.n_ages
        self.n_groups, self.n_replicas = cfg.n_groups, cfg.n_replicas
        age_counts = np.ascontiguousarray(age_counts, dtype=np.int32)
        group_of_age = np.ascontiguousarray(group_of_age, dtype=np.int32)
        import_lo = np.ascontiguousarray(import_lo, dtype=np.int32)
        import_hi = np.ascontiguousarray(import_hi, dtype=np.int32)
        import_cum = np.ascontiguousarray(import_cum, dtype=np.float32)
        varr = (Variant * len(variants))(*variants)
        h = C.c_void_p()
        lib.check(lib.f['create'](C.byref(cfg), _ptr(age_counts, C.c_int32), _ptr(group_of_age, C.c_int32),
                                  varr, _ptr(import_lo, C.c_int32), _ptr(import_hi, C.c_int32),
                                  _ptr(import_cum, C.c_float), C.byref(h)), 'create')
        self.h = h
        self.rank, self.nranks = 0, 1
        self.half_joined = False         # set when a population-sharded join failed half-way
        self.row_len = lib.f['row_len'](h)

    def shard_init(self, rank, nranks, unique_id, exchange_capacity=0.0):
        """Join `nranks` engines (one per GPU / process) into one population-sharded simulation."""
        assert len(unique_id) == 128
        try:
            self.lib.check(self.lib.f['shard_init'](self.h, rank, nranks, bytes(unique_id), exchange_capacity), 'shard_init')
        except EngineError:
            self.half_joined = True      # the ownership split may already have changed: this engine must not step
            raise
        self.rank, self.nranks = rank, nranks

    def save_state(self):
        n = self.lib.f['state_bytes'](self.h)
        out = np.empty(n, dtype=np.uint8)
        self.lib.check(self.lib.f['save_state'](self.h, out.ctypes.data, n), 'save_state')
        return out

    def load_state(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self.lib.check(self.lib.f['load_state'](self.h, blob.ctypes.data, blob.size), 'load_state')

    def close(self):
        if getattr(self, 'h', None):
            self.lib.f['destroy'](self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_contact_table(self, epoch, t):
        f = self.lib.f['set_contact_table']
        self.lib.check(f(self.h, epoch, _ptr(t['n_rows'], C.c_int32), _ptr(t['cum_p'], C.c_double),
                         _ptr(t['age_lo'], C.c_int32), _ptr(t['age_hi'], C.c_int32),
                         _ptr(t['place'], C.c_uint8), _ptr(t['mask_p'], C.c_float),
                         _ptr(t['nr_contacts'], C.c_double), _ptr(t['ncontact_cdf'], C.c_double)),
                       'set_contact_table')

    def set_schedule(self, day0, params):
        arr = (DayParams * len(params))(*params)
        self.lib.check(self.lib.f['set_schedule'](self.h, day0, len(params), arr), 'set_schedule')

    def step(self, n=1):
        if self.half_joined:
            raise EngineError('this engine was left half-joined by a failed population-sharded join: create a new Context')
        self.lib.check(self.lib.f['step'](self.h, n), 'step')

    def set_initial_state(self, ipc7):
        a = np.ascontiguousarray(ipc7, dtype=np.int32)
        assert a.size == 7
        self.lib.check(self.lib.f['set_initial_state'](self.h, _ptr(a, C.c_int32)), 'set_initial_state')

    def reset(self, seed):
        self.lib.check(self.lib.f['reset'](self.h, int(seed) & 0xFFFFFFFF), 'reset')

    def step_profiled(self, n):
        out = np.zeros(5, dtype=np.float32)
        self.lib.check(self.lib.f['step_profiled'](self.h, n, _ptr(out, C.c_float)), 'step_profiled')
        return out

    def step_timed(self, n):
        """rb_step in its production launch geometry with events around every launch: (ms per kernel summed over its
        launches, launches per kernel, wall ms)."""
        ms = np.zeros(5, dtype=np.float32)
        cnt = np.zeros(5, dtype=np.int32)
        wall = C.c_float()
        self.lib.check(self.lib.f['step_timed'](self.h, n, _ptr(ms, C.c_float), _ptr(cnt, C.c_int32), C.byref(wall)), 'step_timed')
        return ms, cnt, float(wall.value)

    # -- NCCL communicator over the engine handle (CUDA library only) --------------------------------------------
    def comm_init(self, rank, nranks, unique_id):
        assert len(unique_id) == 128
        self.lib.check(self.lib.f['comm_init'](self.h, rank, nranks, bytes(unique_id)), 'comm_init')
        self.rank, self.nranks = rank, nranks

    def comm_allreduce(self, x, op='sum'):
        a = np.ascontiguousarray(x, dtype=np.float64).copy()
        self.lib.check(self.lib.f['comm_allreduce'](self.h, _ptr(a, C.c_double), a.size, {'sum': 0, 'max': 1}[op]), 'comm_allreduce')
        return a

    def comm_allgather(self, x):
        a = np.ascontiguousarray(x)
        n = self.lib.f['comm_size'](self.h) if 'comm_size' in self.lib.f else 1
        out = np.empty((n,) + a.shape, dtype=a.dtype)
        self.lib.check(self.lib.f['comm_allgather'](self.h, a.ctypes.data, out.ctypes.data, a.nbytes), 'comm_allgather')
        return out

    def reduce_moments(self, day0, n):
        """read_moments summed over the ranks of the communicator: (sum, sumsq, total number of replicas)."""
        s1 = np.empty((n, self.row_len), dtype=np.float64)
        s2 = np.empty((n, self.row_len), dtype=np.float64)
        if 'reduce_moments' not in self.lib.f:           # the sequential CPU oracle has no ranks
            s1, s2 = self.read_moments(day0, n)
            return s1, s2, self.n_replicas
        tot = C.c_int64()
        self.lib.check(self.lib.f['reduce_moments'](self.h, day0, n, _ptr(s1, C.c_double), _ptr(s2, C.c_double), C.byref(tot)), 'reduce_moments')
        return s1, s2, int(tot.value)

    def sync(self):
        self.lib.check(self.lib.f['sync'](self.h), 'sync')

    def day(self):
        return self.lib.f['day'](self.h)

    def snapshot(self):
        self.lib.check(self.lib.f['snapshot'](self.h), 'snapshot')

    def read_stats(self, day0, n):
        out = np.empty((self.n_replicas, n, self.row_len), dtype=np.int32)
        self.lib.check(self.lib.f['read_stats'](self.h, day0, n, _ptr(out, C.c_int32)), 'read_stats')
        return out

    def read_moments(self, day0, n):
        s1 = np.empty((n, self.row_len), dtype=np.float64)
        s2 = np.empty((n, self.row_len), dtype=np.float64)
        self.lib.check(self.lib.f['read_moments'](self.h, day0, n, _ptr(s1, C.c_double), _ptr(s2, C.c_double)), 'read_moments')
        return s1, s2

    def read_per_age(self, replica, attr):
        out = np.empty(self.n_ages, dtype=np.int32)
        self.lib.check(self.lib.f['read_per_age'](self.h, replica, attr, _ptr(out, C.c_int32)), 'read_per_age')
        return out

    def problem(self):
        out = np.zeros(self.n_replicas, dtype=np.int32)
        self.lib.check(self.lib.f['problem'](self.h, _ptr(out, C.c_int32)), 'problem')
        return out

    def sample(self, what, age, severity, n=10000):
        out = np.empty(n, dtype=np.int32)
        self.lib.check(self.lib.f['sample'](self.h, what, age, severity, n, _ptr(out, C.c_int32)), 'sample')
        return out

    def read_agents(self, replica=0):
        out = np.empty(self.n_agents, dtype=AGENT_DTYPE)
        self.lib.check(self.lib.f['read_agents'](self.h, replica, out.ctypes.data), 'read_agents')
        return out

    def read_queue(self, replica=0):
        cap = max(1024, self.n_agents)
        out = np.empty(cap, dtype=np.int32)
        n = C.c_int32()
        self.lib.check(self.lib.f['read_queue'](self.h, replica, _ptr(out, C.c_int32), cap, C.byref(n)), 'read_queue')
        return out[:n.value].copy()

    def read_available(self, replica=0):
        out = np.zeros(2, dtype=np.int32)
        self.lib.check(self.lib.f['read_available'](self.h, replica, _ptr(out, C.c_int32)), 'read_available')
        return out

    def transmission_stats(self):
        """[replica, rb_transmission_len] int32: the transmission tables of every replica (reina_b200.h)."""
        out = np.empty((self.n_replicas, self.lib.f['transmission_len'](self.h)), dtype=np.int32)
        self.lib.check(self.lib.f['transmission_stats'](self.h, _ptr(out, C.c_int32)), 'transmission_stats')
        return out

    def read_infection_days(self, replica=0):
        """Infection day of every agent of one replica, -1 = never infected."""
        out = np.empty(self.n_agents, dtype=np.int32)
        self.lib.check(self.lib.f['read_infection_days'](self.h, replica, _ptr(out, C.c_int32)), 'read_infection_days')
        return out

    def transmission_settings(self, epoch_of_day):
        """[replica, rb_transmission_settings_len] int32: the tables by place of infection and age group of every replica
        (reina_b200.h); epoch_of_day = contact-table epoch of every completed day."""
        ep = np.ascontiguousarray(epoch_of_day, dtype=np.int32)
        out = np.empty((self.n_replicas, self.lib.f['transmission_settings_len'](self.h)), dtype=np.int32)
        self.lib.check(self.lib.f['transmission_settings'](self.h, _ptr(ep, C.c_int32), ep.size, _ptr(out, C.c_int32)),
                       'transmission_settings')
        return out

    def read_infection_places(self, replica, epoch_of_day):
        """Place of infection of every agent of one replica: -1 never infected, 0..5 a contact place, 6 a root."""
        ep = np.ascontiguousarray(epoch_of_day, dtype=np.int32)
        out = np.empty(self.n_agents, dtype=np.int32)
        self.lib.check(self.lib.f['read_infection_places'](self.h, replica, _ptr(ep, C.c_int32), ep.size, _ptr(out, C.c_int32)),
                       'read_infection_places')
        return out

    def branch(self, src, seeds):
        """Replica j continues from the current state of replica src[j] with seed seeds[j] (rb_branch)."""
        s = np.ascontiguousarray(src, dtype=np.int32)
        k = np.ascontiguousarray(seeds, dtype=np.uint32)
        assert s.shape == k.shape == (self.n_replicas,)
        self.lib.check(self.lib.f['branch'](self.h, _ptr(s, C.c_int32), _ptr(k, C.c_uint32)), 'branch')

    def read_seeds(self):
        """[replica, max_days + 1] uint32: the draw seed of every replica on every day (rb_read_seeds)."""
        out = np.empty((self.n_replicas, self.cfg.max_days + 1), dtype=np.uint32)
        self.lib.check(self.lib.f['read_seeds'](self.h, _ptr(out, C.c_uint32)), 'read_seeds')
        return out

    # -- replica records (rb_replica_bytes / rb_export_replicas / rb_import_replicas / rb_copy_replicas) ----------
    def replica_bytes(self):
        return int(self.lib.f['replica_bytes'](self.h))

    def export_replicas(self, idx):
        """uint8 [n, replica_bytes]: the records of replicas idx."""
        i = np.ascontiguousarray(idx, dtype=np.int32).ravel()
        out = np.empty((i.size, self.replica_bytes()), dtype=np.uint8)
        self.lib.check(self.lib.f['export_replicas'](self.h, i.size, _ptr(i, C.c_int32), out.ctypes.data, out.size), 'export_replicas')
        return out

    def import_replicas(self, slots, seeds, records):
        s = np.ascontiguousarray(slots, dtype=np.int32).ravel()
        k = np.ascontiguousarray(seeds, dtype=np.uint32).ravel()
        b = np.ascontiguousarray(records, dtype=np.uint8)
        assert s.shape == k.shape
        self.lib.check(self.lib.f['import_replicas'](self.h, s.size, _ptr(s, C.c_int32), _ptr(k, C.c_uint32), b.ctypes.data, b.size),
                       'import_replicas')

    def copy_replicas_from(self, src, src_idx, slots, seeds):
        """Replicas src_idx of Engine `src` into slots of this engine (rb_copy_replicas)."""
        i = np.ascontiguousarray(src_idx, dtype=np.int32).ravel()
        s = np.ascontiguousarray(slots, dtype=np.int32).ravel()
        k = np.ascontiguousarray(seeds, dtype=np.uint32).ravel()
        assert i.shape == s.shape == k.shape
        self.lib.check(self.lib.f['copy_replicas'](self.h, src.h, i.size, _ptr(i, C.c_int32), _ptr(s, C.c_int32), _ptr(k, C.c_uint32)),
                       'copy_replicas')

    def comm_move_replicas(self, send_idx, send_peer, recv_slot, recv_peer, recv_seed):
        """Collective replica moves over the engine's NCCL communicator (rb_comm_move_replicas)."""
        a = [np.ascontiguousarray(x, dtype=np.int32).ravel() for x in (send_idx, send_peer, recv_slot, recv_peer)]
        k = np.ascontiguousarray(recv_seed, dtype=np.uint32).ravel()
        assert a[0].shape == a[1].shape and a[2].shape == a[3].shape == k.shape
        self.lib.check(self.lib.f['comm_move_replicas'](self.h, a[0].size, _ptr(a[0], C.c_int32), _ptr(a[1], C.c_int32),
                                                        a[2].size, _ptr(a[2], C.c_int32), _ptr(a[3], C.c_int32), _ptr(k, C.c_uint32)),
                       'comm_move_replicas')

    def set_transmission_scale(self, scale):
        """float32 [n_replicas]: every replica's transmission scale, in force from the next step."""
        s = np.ascontiguousarray(scale, dtype=np.float32)
        assert s.shape == (self.n_replicas,)
        self.lib.check(self.lib.f['set_transmission_scale'](self.h, _ptr(s, C.c_float)), 'set_transmission_scale')

    def read_transmission_scale(self):
        out = np.empty(self.n_replicas, dtype=np.float32)
        self.lib.check(self.lib.f['read_transmission_scale'](self.h, _ptr(out, C.c_float)), 'read_transmission_scale')
        return out

    def set_severity_scale(self, scale):
        """float32 [n_replicas, 3]: every replica's severe, critical and fatal scales, in force from the next step."""
        s = np.ascontiguousarray(scale, dtype=np.float32)
        assert s.shape == (self.n_replicas, 3)
        self.lib.check(self.lib.f['set_severity_scale'](self.h, _ptr(s, C.c_float)), 'set_severity_scale')

    def read_severity_scale(self):
        out = np.empty((self.n_replicas, 3), dtype=np.float32)
        self.lib.check(self.lib.f['read_severity_scale'](self.h, _ptr(out, C.c_float)), 'read_severity_scale')
        return out

    def last_step_ms(self):
        return float(self.lib.f['last_step_ms'](self.h))

    def launch_count(self):
        return int(self.lib.f['launch_count'](self.h))

    def copied_bytes(self):
        """(host -> device, device -> host) bytes copied by this handle so far."""
        f = self.lib.f['copied_bytes']
        return int(f(self.h, 0)), int(f(self.h, 1))


def shard_init_local(engines, exchange_capacity=0.0):
    """Join the Engine objects of THIS process into one population-sharded simulation: rank k = engines[k]
    (rb_shard_init_local: plain device pointers instead of NCCL + CUDA IPC).  Step each from its own thread."""
    lib = engines[0].lib
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    try:
        lib.check(lib.f['shard_init_local'](arr, len(engines), exchange_capacity), 'shard_init_local')
    except EngineError:
        for e in engines:
            e.half_joined = True         # some ranks may already own only their stripes: none of them may step
        raise
    for k, e in enumerate(engines):
        e.rank, e.nranks = k, len(engines)


def shard_unique_id(lib=None):
    """A fresh NCCL unique id (128 bytes): rank 0 creates it and hands it to the other ranks."""
    lib = lib or cuda_library()
    buf = C.create_string_buffer(128)
    lib.check(lib.f['shard_unique_id'](buf), 'shard_unique_id')
    return buf.raw
