/*
 * reina_b200.h -- C-ABI of the B200-native per-day agent loop (libreina_b200.so).
 *
 * The reference has no FFI for this path: `calc.simulation` talks to the Cython extension module
 * `cythonsim.main` (imported as `model`, cythonsim/__init__.py:5-8) through Python objects.  This
 * header is the boundary a maintainer binds instead: `reina_b200/model.py` mirrors the Python surface
 * (`Context`, `add_intervention`, `iterate`, `generate_state`, ...) and calls these entry points through
 * ctypes.  Plain C types only, caller-owned buffers, int return codes (0 = ok), no global state:
 * one handle = one CUDA device + one stream, so 8 handles drive 8 GPUs from one process.
 *
 * Each entry point cites the reference interface it replaces (paths relative to the reference root).
 *
 * The CPU oracle (oracle/reina_oracle.c, test infrastructure) exports the same functions with the
 * `ro_` prefix and the same struct layouts, so tests can drive both through one ctypes wrapper.
 */
#ifndef REINA_B200_H
#define REINA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RB_MAX_AGES 128      /* single-year ages 0..n_ages-1 (reference: 101, main.pyx:1355) */
#define RB_MAX_VARIANTS 4    /* wild-type + configured variants (main.pyx:868-881) */
#define RB_MAX_ROWS 96       /* contact rows per participant age: 6 places x 15 bands = 90 (main.pyx:1094-1103) */
#define RB_NCDF 100          /* contacts per infector per day are capped at 100 (get_contacts limit, main.pyx:1539) */
#define RB_MAX_IMPORT_EVENTS 8
#define RB_MAX_VACC 8
#define RB_MAX_IMPORT_CLASSES 16
#define RB_N_PLACES 6        /* ContactPlace HOME..OTHER, main.pyx:64-70 */
#define RB_IOT_LEN 21        /* INFECTIOUSNESS_OVER_TIME days -10..+10, main.pyx:660-682 */

/* enum SymptomSeverity / PersonState / SimulationProblem / TestingMode: main.pyx:33-61, 441-445 */
enum { RB_ASYMPTOMATIC = 0, RB_MILD, RB_SEVERE, RB_CRITICAL, RB_FATAL };
enum { RB_SUSCEPTIBLE = 0, RB_INCUBATION, RB_ILLNESS, RB_HOSPITALIZED, RB_IN_ICU, RB_RECOVERED, RB_DEAD };
enum { RB_NO_PROBLEMOS = 0, RB_TOO_MANY_INFECTEES, RB_TOO_MANY_CONTACTS, RB_HOSPITAL_ACCOUNTING_FAILURE,
       RB_NEGATIVE_CONTACTS, RB_MALLOC_FAILURE, RB_OTHER_FAILURE, RB_WRONG_STATE,
       RB_CONTACT_PROBABILITY_FAILURE, RB_INFECTEES_MISMATCH };
enum { RB_NO_TESTING = 0, RB_ALL_WITH_SYMPTOMS_CT, RB_ALL_WITH_SYMPTOMS, RB_ONLY_SEVERE_SYMPTOMS };

/* Per-age population counters, in the order generate_state lists them (main.pyx:1819-1833). */
enum { RB_A_SUSCEPTIBLE = 0, RB_A_VACCINATED, RB_A_INFECTED, RB_A_ALL_INFECTED, RB_A_DETECTED,
       RB_A_ALL_DETECTED, RB_A_IN_ICU, RB_A_CUM_ICU, RB_A_IN_WARD, RB_A_DEAD, RB_A_RECOVERED,
       RB_A_NON_HOSPITAL_DEATHS, RB_A_NEW_INFECTIONS, RB_N_ATTRS };

/* Scalars appended to every stats row after the RB_N_ATTRS x n_groups block (main.pyx:1835-1855). */
enum { RB_S_AVAILABLE_ICU = 0, RB_S_AVAILABLE_BEDS, RB_S_TOTAL_ICU, RB_S_TOTAL_BEDS,
       RB_S_TOTAL_INFECTIONS, RB_S_TOTAL_INFECTORS, /* r = infections/infectors if infectors > 5 (main.pyx:1817) */
       RB_S_EXPOSED_PER_DAY, RB_S_CT_CASES_PER_DAY, RB_S_TABLE_EPOCH, RB_S_DAY,
       RB_S_CONTACTS0, /* daily_contacts[6] */
       RB_S_VARIANT0 = RB_S_CONTACTS0 + RB_N_PLACES, /* infected_by_variant[RB_MAX_VARIANTS] */
       RB_N_SCALARS = RB_S_VARIANT0 + RB_MAX_VARIANTS };

/* Disease parameters of one variant (struct Variant, main.pyx:787-806; variant_init :820-850).
 * Per-age tables are the ClassifiedValues expanded with cv_get_greatest_lte (:721-730). */
enum { RB_T_SUSCEPTIBILITY = 0, RB_T_SYMPTOMATIC, RB_T_SEVERE, RB_T_CRITICAL, RB_T_FATAL,
       RB_T_DEATH_OUTSIDE_HOSPITAL, RB_N_TABLES };
typedef struct rb_variant {
    float p_icu_death_no_beds, p_hospital_death_no_beds;
    float infectiousness_multiplier, p_asymptomatic_infection;
    float p_mask_protects_wearer, p_mask_protects_others;
    float ratio_before_hospitalisation, ratio_in_ward;
    /* gamma(mu, cv) as simrandom.pyx:46-55 parametrises it: kappa = mu/theta, theta = (cv mu)^2/mu */
    float incubation_kappa, incubation_theta;      /* main.pyx:977-986  (cv 0.86) */
    float onset_death_kappa, onset_death_theta;    /* main.pyx:989-1001 (cv 0.45, FATAL) */
    float onset_recovery_kappa, onset_recovery_theta;
    float reserved[2];                             /* [0] = max over ages of tab[RB_T_SUSCEPTIBILITY] (transmission upper bound) */
    float iot[RB_IOT_LEN + 3];                     /* index = day + 10 */
    float tab[RB_N_TABLES][RB_MAX_AGES];
} rb_variant;

typedef struct rb_config {
    int32_t n_agents;      /* total_people, main.pyx:1449 */
    int32_t n_ages;        /* nr_ages, main.pyx:1355 */
    int32_t n_groups;      /* len(age_groups.labels), calc/simulation.py:156-161 */
    int32_t n_variants;    /* Disease.nr_variants, main.pyx:870 */
    int32_t n_replicas;    /* ensemble members advanced by the same launches; replica r uses seed + r */
    uint32_t seed;         /* Context(random_seed=...), main.pyx:1759-1760 */
    int32_t hospital_beds, icu_units;   /* HealthcareSystem.__init__, main.pyx:461-465 */
    int32_t max_days;      /* capacity of the per-day stats buffer */
    int32_t n_import_classes;           /* imported_infection_ages, main.pyx:1376-1384 */
    int32_t device;        /* CUDA device ordinal (ignored by the oracle) */
    float contact_capacity;  /* capacity of the per-day contact work list, in units of n_agents (0 = default) */
    int32_t reserved[4];
} rb_config;

/* Everything the host-side intervention schedule decides for one simulated day
 * (Context.iterate / apply_intervention, main.pyx:1880-1960, 2011-2016; Population.init_day :1687-1699;
 *  HealthcareSystem.iterate :547-558). */
typedef struct rb_day_params {
    int32_t testing_mode;            /* set_testing_mode, main.pyx:623-628 */
    float p_detected_anyway;
    float p_successful_tracing;
    int32_t beds_delta, icu_delta;   /* build-new-hospital-beds / build-new-icu-units, :1891-1896 */
    int32_t table_epoch;             /* contact table in force today (set_mobility_factor + init_day, :1250-1288) */
    int32_t n_imports;               /* 'import-infections' events dated today, in list order (:1897-1899) */
    int32_t import_amount[RB_MAX_IMPORT_EVENTS];
    int32_t import_variant[RB_MAX_IMPORT_EVENTS];
    int32_t trickle[RB_MAX_VARIANTS];   /* infect_people_daily amounts per variant (:1671-1685) */
    int32_t n_vacc;                  /* active vaccination programmes (:548-558) */
    int32_t vacc_nr[RB_MAX_VACC], vacc_min_age[RB_MAX_VACC], vacc_max_age[RB_MAX_VACC];
    int32_t vacc_slot[RB_MAX_VACC];  /* stable programme id */
    /* bit i: testing mode was test-with-contact-tracing at the moment import event i was applied (interventions of one
     * date are applied in list order, main.pyx:2012-2015, and person_infect gives the new case an infectee list only
     * under contact tracing, :227-233) */
    int32_t import_traced;
    int32_t reserved[3];
} rb_day_params;

/* One agent in canonical (layout-independent) form, for parity tests (struct Person, main.pyx:132-144). */
typedef struct rb_agent {
    int32_t infector;            /* agent index in age-sorted order, -1 = none */
    int32_t n_infected;          /* other_people_infected */
    int16_t days_left;
    int16_t day_of_illness;      /* saturates at 31 */
    int16_t day_of_vaccination;  /* -1 = not vaccinated */
    uint8_t state, severity, variant;
    uint8_t flags;               /* bit0 detected, 1 queued_for_testing, 2 included_in_totals, 3 has infectee list */
    uint8_t ward_days, icu_days; /* durations fixed at symptom onset (main.pyx:1016-1039) */
} rb_agent;

typedef struct rb_engine rb_engine;

/* Context.__init__ (main.pyx:1759-1781): Disease + Population (_init_stats, _create_agents) + HealthcareSystem.
 * age_counts[n_ages]; group_of_age[n_ages]; variants[n_variants];
 * import classes: age band [lo,hi] and cumulative weight (Population.__init__ :1376-1384, get_import_infection_person :1632-1650). */
int rb_create(const rb_config *cfg, const int32_t *age_counts, const int32_t *group_of_age,
              const rb_variant *variants, const int32_t *import_lo, const int32_t *import_hi,
              const float *import_cum, rb_engine **out);
void rb_destroy(rb_engine *e);

/* Re-initialise every replica to the state right after rb_create with a new base seed (a fresh
 * Context(random_seed=seed), main.pyx:1759-1781) without reallocating; schedule and contact tables are kept. */
int rb_reset(rb_engine *e, uint32_t seed);

/* Population.set_initial_state (main.pyx:1452-1516, called by Context.__init__ :1780-1781): start the run with an
 * epidemic already under way.  ipc = {dead, in_icu, in_ward, confirmed_cases, incubating, ill, recovered}
 * (InitialPopulationCondition, calc/datasets.py:107-135).  Once, before the first rb_step; rb_reset re-applies it. */
int rb_set_initial_state(rb_engine *e, const int32_t *ipc7);

/* ContactMatrix.generate_contact_probabilities output (main.pyx:1184-1235) for one mobility epoch:
 * per participant age `n_rows[age]` rows of {cum_p, contact band [lo,hi], place, mask_p}, arrays are
 * [n_ages][RB_MAX_ROWS]; nr_contacts[age] = nr_contacts_by_age (main.pyx:1209-1211).
 * ncontact_cdf[age][cls][k] = P(number of contacts <= k) for ContactMatrix.get_nr_contacts (main.pyx:1308-1320:
 * n = min(limit, int(max(1, lognormal(0, 0.5) * nr_contacts_by_age[age] * factor)) - 1)), tabulated by the host in
 * double precision so that the device draws n with one uniform and a binary search instead of evaluating
 * exp/log per infector.  cls 0: factor 1, limit 100 (incubating / asymptomatic); cls 1: factor 0.5, limit 5
 * (symptomatic, Disease.get_exposed_people :945-953).  Array is [n_ages][2][RB_NCDF]. */
int rb_set_contact_table(rb_engine *e, int32_t epoch, const int32_t *n_rows, const double *cum_p,
                         const int32_t *age_lo, const int32_t *age_hi, const uint8_t *place,
                         const float *mask_p, const double *nr_contacts, const double *ncontact_cdf);

/* Host-side schedule for days [day0, day0 + n). */
int rb_set_schedule(rb_engine *e, int32_t day0, int32_t n, const rb_day_params *params);

/* Context.iterate() x n (main.pyx:2011-2018, _iterate :1994-2009).  Asynchronous on the handle's stream;
 * a stats row is recorded at the start of every day (= generate_state() before iterate(),
 * calc/simulation.py:195,270). */
int rb_step(rb_engine *e, int32_t n_days);
int rb_sync(rb_engine *e);
int32_t rb_day(rb_engine *e);

/* Context.generate_state() (main.pyx:1813-1857): record the stats row of the current day without stepping. */
int rb_snapshot(rb_engine *e);
int32_t rb_row_len(rb_engine *e);   /* RB_N_ATTRS * n_groups + RB_N_SCALARS */
/* out[replica][day][row_len], days [day0, day0+n) */
int rb_read_stats(rb_engine *e, int32_t day0, int32_t n, int32_t *out);

/* Ensemble moments of the stats rows, reduced on the device: for days [day0, day0+n) and every row column,
 * sum[day][col] = sum over replicas of x and sumsq[day][col] = sum of x^2 (doubles, [n][row_len] each).  This is what a
 * Monte-Carlo run returns (mean / std curves); it replaces the D2H copy of every replica's rows. */
int rb_read_moments(rb_engine *e, int32_t day0, int32_t n, double *sum, double *sumsq);

/* Context.get_population_stats(what) (main.pyx:1859-1866): per single-year age counter of one replica. */
int rb_read_per_age(rb_engine *e, int32_t replica, int32_t attr, int32_t *out);

/* Sticky SimulationProblem per replica (main.pyx:51-61, 2017-2018). */
int rb_problem(rb_engine *e, int32_t *out);

/* Context.sample(what, age, severity) (main.pyx:2047-2101).  what: 0 contacts_per_day, 1 symptom_severity,
 * 2 incubation_period, 3 illness_period, 4 hospitalization_period, 5 icu_period, 6 onset_to_removed_period. */
int rb_sample(rb_engine *e, int32_t what, int32_t age, int32_t severity, int32_t n, int32_t *out);

/* The counter-based random block behind every draw (replaces RandomPool, simrandom.pyx:13-55), computed on the host by
 * the function the kernels inline: words = 4 -> Philox4x32-10 with key (key, 0x5EEDB200) and counter ctr[0..3] (other
 * widths are refused).  No device needed: the CPU tests pin the generator to the Random123 known-answer vectors through
 * this call. */
int rb_rng_block(int32_t words, uint32_t key, const uint32_t *ctr, uint32_t *out);

/* Transmission statistics of the state after the last completed rb_step, from the infection tree every run keeps (no
 * reference counterpart: main.pyx only reports r = total_infections / total_infectors, which mixes infection days).
 * Per replica one int32 row of rb_transmission_len entries, M = max_days + 1:
 *   cohort_infected[M], cohort_offspring[M], cohort_open[M]   by infection day d: infected agents, the sum of their
 *                                                             other_people_infected, those still INCUBATION / ILLNESS
 *   offspring_hist[RB_TX_BINS]                                closed cases (neither INCUBATION nor ILLNESS) by
 *                                                             min(other_people_infected, 64)
 *   gi_hist[RB_TX_BINS]                                       agents with an infector by min(d - d(infector), 64)
 *   group_closed[n_groups], group_offspring[n_groups]         closed cases and their offspring by age group
 *   variant_closed[RB_MAX_VARIANTS], variant_offspring[RB_MAX_VARIANTS]   the same by variant
 * Identical on every rank of a population-sharded simulation.  CUDA library only: the tests' CPU reference is the oracle
 * plus these three entry points as plain loops (tests/oracle_transmission.c). */
#define RB_TX_BINS 65        /* histogram bins 0..63 and ">= 64" */
int32_t rb_transmission_len(rb_engine *e);   /* 3 (max_days + 1) + 2 RB_TX_BINS + 2 n_groups + 2 RB_MAX_VARIANTS */
/* out[n_replicas][rb_transmission_len] */
int rb_transmission_stats(rb_engine *e, int32_t *out);
/* Infection day of every agent of one replica (-1 = never infected): with rb_read_agents' infector, the transmission tree. */
int rb_read_infection_days(rb_engine *e, int32_t replica, int32_t *out);

/* Transmission by setting and age of the state after the last completed rb_step (no reference counterpart: main.pyx
 * only counts daily_contacts[place], contacts made rather than infections).  The place of a child's infection is
 * recomputed from its infector, infection day and winning contact slot, which every run keeps, against the contact
 * table of the epoch in force on that day.  Per replica one int32 row of rb_transmission_settings_len entries,
 * M = max_days + 1, P = RB_N_PLACES, G = n_groups:
 *   by_day_place[M][P + 1]     infected agents by infection day and place of infection (column RB_PLACE_ROOT: imports and
 *                              the initial state, which have no infector)
 *   pair_all[P][G][G]          children by place, infector's age group, child's age group
 *   pair_closed[P][G][G]       the same, only children of closed infectors (neither INCUBATION nor ILLNESS)
 *   closed_by_group[G]         closed cases by age group (equals group_closed of rb_transmission_stats)
 * epoch_of_day[0 .. n_days): the contact-table epoch (rb_set_contact_table) in force on each completed day, as the caller
 * scheduled it (rb_day_params.table_epoch); n_days must equal rb_day(e) and every epoch must have a table, else 1.
 * Identical on every rank of a population-sharded simulation.  CUDA library only: the tests' CPU reference is the
 * oracle, which records the place where it infects, plus these three entry points as plain loops
 * (tests/oracle_settings.c). */
#define RB_PLACE_ROOT RB_N_PLACES
int32_t rb_transmission_settings_len(rb_engine *e);   /* (max_days + 1)(RB_N_PLACES + 1) + 2 RB_N_PLACES n_groups^2 + n_groups */
/* out[n_replicas][rb_transmission_settings_len] */
int rb_transmission_settings(rb_engine *e, const int32_t *epoch_of_day, int32_t n_days, int32_t *out);
/* Place of infection of every agent of one replica: -1 never infected, 0 .. RB_N_PLACES - 1, RB_PLACE_ROOT. */
int rb_read_infection_places(rb_engine *e, int32_t replica, const int32_t *epoch_of_day, int32_t n_days, int32_t *out);

/* Parity/debug exports. */
int rb_read_agents(rb_engine *e, int32_t replica, rb_agent *out);
int rb_read_queue(rb_engine *e, int32_t replica, int32_t *out, int32_t cap, int32_t *n);   /* test queue, in order */
int rb_read_available(rb_engine *e, int32_t replica, int32_t *beds_icu);  /* {available_beds, available_icu_units} */
/* timing of the last rb_step measured with CUDA events on the handle's stream (ms); oracle: wall clock */
float rb_last_step_ms(rb_engine *e);
/* Like rb_step, but brackets every kernel with CUDA events and returns the summed device time per kernel
 * (ms_per_kernel[RB_N_KERNELS], order: pre, sweep, expose, resolve, post).  One kernel at a time on one stream with
 * full-wave grids: what each kernel costs when it has the GPU to itself.  Measurement aid for bench.py. */
#define RB_N_KERNELS 5
int rb_step_profiled(rb_engine *e, int32_t n_days, float *ms_per_kernel);
/* The same measurement in the PRODUCTION launch geometry of rb_step (replica groups on concurrent, staggered streams
 * with rb_step's grids; kernels launched one by one so that events can sit between them).  ms_per_kernel[k] sums the
 * event-to-event time of kernel k over launches_per_kernel[k] launches; wall_ms is the whole run.  Launches of different
 * groups overlap, so the per-kernel sums add up to more than wall_ms.  CUDA library only. */
int rb_step_timed(rb_engine *e, int32_t n_days, float *ms_per_kernel, int32_t *launches_per_kernel, float *wall_ms);
/* ---- Ensemble across GPUs (BASELINE configs[3]; replaces the reference's multiprocessing.Pool over seeds,
 * calc/simulation.py:376-377).  The ensemble shards as independent replicas, one process and one engine per GPU, with no
 * data-path collective; the only exchange is the final reduce of the daily curves, done here with NCCL on device buffers
 * (libnccl.so.2 is loaded at run time by these calls only).  rb_comm_init joins the engine to a communicator: rank 0 gets
 * a 128-byte unique id from rb_shard_unique_id and hands it to the other ranks by any host-side means
 * (reina_b200/comm.py: a file under /tmp for the ranks of one node).  rb_reduce_moments = rb_read_moments summed over all
 * ranks (sum, sum of squares and the replica count in ONE ncclAllReduce); rb_comm_allreduce (op 0 sum, 1 max; n = 1 makes
 * it a barrier) and rb_comm_allgather move small host buffers over the same communicator.  Without a communicator all
 * of them act on the local engine alone. */
int rb_comm_init(rb_engine *e, int32_t rank, int32_t nranks, const uint8_t *unique_id128);
int32_t rb_comm_rank(rb_engine *e);
int32_t rb_comm_size(rb_engine *e);
int rb_comm_allreduce(rb_engine *e, double *inout, int64_t n, int32_t op);
int rb_comm_allgather(rb_engine *e, const void *in, void *out, int64_t bytes_per_rank);
int rb_reduce_moments(rb_engine *e, int32_t day0, int32_t n, double *sum, double *sumsq, int64_t *n_replicas);

/* ---- Population-sharded mode (BASELINE configs[4]; no reference counterpart: the reference is one process, SURVEY 2.2).
 * One process per GPU; every rank creates the same engine (same inputs, seed, schedule, n_replicas = 1) and then joins:
 * rank 0 obtains a 128-byte NCCL unique id with rb_shard_unique_id and hands it to the others by any means; each rank
 * calls rb_shard_init(e, rank, nranks, id, exchange_capacity) before the first rb_step.  Agents are dealt to the ranks in
 * stripes of 4096 (age-sorted order, so every rank holds ~1/nranks of every age).  A rank sweeps and samples contacts only
 * for the agents it owns; once per simulated day the ranks exchange their day's cross-shard events -- successful
 * transmissions, state changes, test-queue entries, capacity events, counter deltas -- and every rank applies all of them,
 * so counters, queues and every rb_read_* result are identical on all ranks and bit-identical to a single-GPU run.
 * The exchange runs over NVLink peer memory: every rank maps every other rank's message buffer (CUDA IPC, set up through
 * the NCCL communicator), publishes a per-day flag when its message is complete, and the merge kernel pulls exactly the
 * bytes each message holds.  Where peer mapping is not possible (ranks inside one process, no peer access, or
 * RB_SHARD_EXCHANGE=nccl) the fixed-size message slots travel through one ncclAllGather per day instead.
 * Per-agent day counters and severity are authoritative on the owning rank only (rb_read_agents: take agent a from rank
 * (a >> 12) % nranks).  exchange_capacity scales the per-day message capacity (0 = default); overflow sets RB_OTHER_FAILURE.
 * libnccl.so.2 is loaded at run time by these calls only. */
int rb_shard_unique_id(uint8_t *out128);
int rb_shard_init(rb_engine *e, int32_t rank, int32_t nranks, const uint8_t *unique_id128, float exchange_capacity);
/* The same join for `nranks` engines of ONE process (rank k = engines[k]): no NCCL and no CUDA IPC, every rank reads the
 * others' message buffers through plain device pointers (engines on one device, or on devices with peer access, which
 * this call enables).  Each engine must then be stepped from its own host thread (a rank's day ends only after every
 * rank's sweep of that day has been launched), and all of them must be idle before any one is destroyed.  This is how a
 * single-GPU box exercises the multi-rank exchange: several ranks, each on its own stream of the one device. */
int rb_shard_init_local(rb_engine **engines, int32_t nranks, float exchange_capacity);
int32_t rb_shard_rank(rb_engine *e);
int32_t rb_shard_nranks(rb_engine *e);
int64_t rb_shard_message_bytes(rb_engine *e);   /* capacity of one rank's daily message (what the all-gather path moves) */
int32_t rb_shard_exchange(rb_engine *e);        /* 0 = not sharded, 1 = ncclAllGather, 2 = NVLink peer memory */

/* ---- Checkpoint / resume (SURVEY 8f rank 4; the reference keeps its state only in process memory).
 * The blob holds the whole mutable state between two rb_step calls (packed words, agent records, bitmaps, counters, test
 * queues, stats rows so far, day).  It can be loaded into any engine created with the same inputs, replica count and
 * max_days; contact tables and the schedule are inputs, not state, and are set by the caller as usual. */
int64_t rb_state_bytes(rb_engine *e);
int rb_save_state(rb_engine *e, void *out, int64_t capacity);
int rb_load_state(rb_engine *e, const void *in, int64_t n_bytes);
/* Blob version 3 appends the seed history of rb_read_seeds; a version-2 blob still loads, its history taken from the
 * loaded seeds. */

/* ---- Branching replicas (no reference counterpart: the reference runs one replica from day 0 and never copies one).
 * Replica j continues from the current state of replica src[j], drawing with seed[j] from the next rb_step on.  The copy
 * is the state of rb_save_state plus the replica's sweep-order keys, so a copy made with the source's own seed continues
 * exactly as the source does.  Requires 0 <= src[j] < R and src[src[j]] == src[j] for every j (a replica that is copied
 * from keeps its own state); identity src with the current seeds is a no-op, identity src with new seeds re-seeds the
 * futures.  Refused (return 1, rb_last_error) for a bad or chained source and in population-sharded mode; the engine
 * stays usable.  Waits for every stream of the engine first.  CUDA library only. */
int rb_branch(rb_engine *e, const int32_t *src, const uint32_t *seed);
/* out[R][max_days + 1]: the draw seed of every replica on every day (days after today: the seed in force now).  No
 * reference counterpart. */
int rb_read_seeds(rb_engine *e, uint32_t *out);

/* Measurement aids of the CUDA library (tools/phase_run.py): flag 9 makes the day-boundary kernels record the cycles
 * they spend per phase; rb_debug_phase_cycles reads the 16 accumulated counters of one replica.  No effect on results. */
void rb_debug_flag(rb_engine *e, int32_t flag);
int rb_debug_phase_cycles(rb_engine *e, int32_t replica, long long *out16);

/* number of kernel launches issued by this handle so far */
int64_t rb_launch_count(rb_engine *e);
/* bytes this handle has copied so far on the per-run path: direction 0 = host -> device (counter initialisation, contact
 * tables, schedule), 1 = device -> host (stats rows, moments, problem words).  bench.py reports their per-step deltas. */
int64_t rb_copied_bytes(rb_engine *e, int32_t direction);
const char *rb_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* REINA_B200_H */
