// reina_b200 engine: the per-day agent loop of Reina (cythonsim/main.pyx Context.iterate and everything it
// calls) as hand-written CUDA for sm_100a, behind the C-ABI of include/reina_b200.h.
//
//   state.cuh     data layout in HBM (agents stored AGE-SORTED, so age is implied by position and a contact target is
//                 age_start[band] + u32 % band_size with no indirection), the segmented active lists, per-replica
//                 counters, shared device helpers, person_infect
//   boundary.cuh  k_pre / k_post / k_between, one CTA per replica or (few replicas of a large population) a team of
//                 co-resident CTAs with a grid barrier: stats row, intervention deltas, imports, test queue + contact
//                 tracing, vaccination, sweep start; beds / ICU first-come-first-served = sort by sweep position +
//                 max-plus scan
//   sweep.cuh     k_sweep: Context._iterate_people / person_advance over the dense active lists (a warp owns whole
//                 segments); emits contact work items, capacity events and test-queue entries tagged with sweep position
//   contacts.cuh  k_expose: one thread per group of four sampled contacts (O(1) row pick, target gather, transmission
//                 draw, atomicMin(winner[target], sweep position of infector | slot)); k_resolve: winners become infected
//   shard.cuh     population-sharded mode: k_publish / k_wait (per-day flags in NVLink peer memory) and k_merge, which
//                 pulls and applies every rank's message of the day
//   setup.cuh     set_initial_state, initialisation, contact-row guide, snapshot, ensemble moments, samplers
//   transmission.cuh  k_transmission: cohort / offspring / generation-interval tables from the infection tree (not per day);
//                 k_transmission_settings: the same tree by place of infection and age group
//   branch.cuh    k_branch_copy / k_branch_rebuild: replicas continue from another replica's current state (rb_branch);
//                 k_import_fixup: replica records written into slots (rb_import_replicas, rb_copy_replicas, rb_comm_move_replicas)
//   this file     host side: engine handle, launch geometry, replica groups, CUDA graphs, NCCL binding (ensemble reduce,
//                 sharded mode), the extern "C" entry points
//
// Per day and replica group (reference order, main.pyx:1994-2016): k_sweep -> k_expose -> k_resolve -> k_between.  Every order-dependent
// step of the sequential reference is resolved through the agent's sweep position, so the result is bit-identical to the
// sequential CPU oracle and independent of scheduling.
#include "state.cuh"
#include "boundary.cuh"
#include "sweep.cuh"
#include "contacts.cuh"
#include "shard.cuh"
#include "setup.cuh"
#include "transmission.cuh"
#include "branch.cuh"

// ================================================================ host side / C-ABI
static thread_local char g_err[512];
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { snprintf(g_err, sizeof g_err, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return 1; } } while (0)

#define MAX_GROUPS 8
struct ReplicaGroup {
    int r0, R;                          // replicas [r0, r0 + R)
    int sweep_blocks, list_blocks, resolve_blocks;
    cudaStream_t stream;
    cudaEvent_t ev_stagger, ev_join;
    cudaGraphExec_t graph[2];
};

struct rb_engine {
    rb_config cfg;
    Eng G;
    cudaStream_t stream;
    cudaEvent_t ev0, ev1;
    std::vector<void *> allocs;
    std::vector<DevTable *> tables;     // host copy of the device pointer table
    std::vector<std::vector<uint8_t>> table_args, table_host;      // per epoch: the arguments last seen, the host-built part of the DevTable
    DevTable **d_tables;
    int n_table_slots;
    rb_day_params *d_sched;
    double *d_moments;                  // [2][max_days + 1][row_len] + 1: ensemble moments (rb_read_moments / rb_reduce_moments)
    void *h_stage; int n_stage;         // pinned staging ring for contact-table uploads (4 x TABLE_HOST_BYTES)
    cudaEvent_t ev_stage[4];
    std::vector<rb_day_params> h_sched;
    std::vector<int32_t> age_start, age_counts;
    std::vector<rb_variant> h_variants;
    int32_t day;
    float last_ms;
    int64_t launches;
    int64_t h2d_bytes, d2h_bytes;       // bytes this handle copied host -> device / device -> host so far (rb_copied_bytes)
    int sweep_blocks, list_blocks, resolve_blocks;     // full-wave grids over all replicas
    bool have_graphs;
    // replica groups: the ensemble is split into n_groups sets of replicas, each advanced by its own chain of launches
    // on its own stream with a grid sized for its share of the SMs.  The groups run half a day apart, so the
    // latency-bound phases of one (k_resolve, the single-CTA day boundary) overlap the sweep / contact kernels of another.
    cudaError_t launch_err;             // first failed cooperative launch (launch_boundary)
    int wide_ctas;                      // CTAs per replica of the wide day boundary (<= 1: one CTA per replica)
    int n_groups;
    ReplicaGroup grp[MAX_GROUPS];
    cudaEvent_t ev_fork;
    ncclComm_t comm;                    // NCCL communicator: the ensemble's final reduce (rb_comm_init) or the population-sharded mode
    int comm_rank, comm_size;
    bool sharded;                       // rb_shard_init joined this engine into one population-sharded simulation
    bool shard_timing; std::vector<cudaEvent_t> shard_events;
    int n_peer_open;                    // peer buffers mapped through CUDA IPC: ranks [0, n_peer_open) except the own one
    int merge_blocks;
    int prio, prio_high;                // RB_PRIO: launch the latency-bound kernels with the device's highest priority
    uint32_t xepoch; uint32_t *d_xepoch;   // host copy / device word of Eng::xepoch
    Ipc ipc; bool has_ipc;              // initial population condition, re-applied by rb_reset
    int32_t *d_tx;                      // [R][rb_transmission_len] tables of rb_transmission_stats, allocated by its first call
    int32_t *d_sx, *d_sx_epoch;         // [R][rb_transmission_settings_len] tables, [max_days + 1] epoch of each day: allocated by the first settings call
    int32_t *d_branch;                  // [R] sources then [R] seeds of rb_branch, allocated by its first call
    int32_t *d_move;                    // [3R] slots, seeds and rebuild markers of a replica import, allocated by the first one
    uint32_t *seed_of_day;              // [R][max_days + 1] seed history (branch.cuh)
};

// ---------------------------------------------------------------- NCCL, bound at run time
struct NcclApi {
    void *dl;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *);
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int);
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    const char *(*GetErrorString)(ncclResult_t);
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)(void);
    ncclResult_t (*GroupEnd)(void);
};
static NcclApi g_nccl;
static int load_nccl() {
    if (g_nccl.dl) return 0;
    // reuse a libnccl the process already mapped (torch ships one with the same soname), else load the system one
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { snprintf(g_err, sizeof g_err, "cannot load libnccl.so.2: %s", dlerror()); return 1; }
    g_nccl.GetUniqueId = (ncclResult_t(*)(ncclUniqueId *))dlsym(h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (ncclResult_t(*)(ncclComm_t *, int, ncclUniqueId, int))dlsym(h, "ncclCommInitRank");
    g_nccl.AllGather = (ncclResult_t(*)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllGather");
    g_nccl.AllReduce = (ncclResult_t(*)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllReduce");
    g_nccl.CommDestroy = (ncclResult_t(*)(ncclComm_t))dlsym(h, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char *(*)(ncclResult_t))dlsym(h, "ncclGetErrorString");
    g_nccl.Send = (ncclResult_t(*)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclSend");
    g_nccl.Recv = (ncclResult_t(*)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclRecv");
    g_nccl.GroupStart = (ncclResult_t(*)(void))dlsym(h, "ncclGroupStart");
    g_nccl.GroupEnd = (ncclResult_t(*)(void))dlsym(h, "ncclGroupEnd");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.AllReduce || !g_nccl.CommDestroy || !g_nccl.GetErrorString ||
        !g_nccl.Send || !g_nccl.Recv || !g_nccl.GroupStart || !g_nccl.GroupEnd) {
        snprintf(g_err, sizeof g_err, "libnccl.so.2 lacks a required symbol"); return 1;
    }
    g_nccl.dl = h;
    return 0;
}
#define NK(call) do { ncclResult_t r_ = (call); if (r_ != ncclSuccess) { snprintf(g_err, sizeof g_err, "%s:%d %s: %s", __FILE__, __LINE__, #call, g_nccl.GetErrorString(r_)); return 1; } } while (0)


template <typename T> static int dalloc(rb_engine *e, T **p, size_t n) {
    void *q = nullptr;
    cudaError_t err = cudaMalloc(&q, n * sizeof(T));
    if (err != cudaSuccess) { snprintf(g_err, sizeof g_err, "cudaMalloc(%zu bytes): %s", n * sizeof(T), cudaGetErrorString(err)); return 1; }
    e->allocs.push_back(q);
    *p = (T *)q;
    return 0;
}
static uint32_t pow2_at_least(uint64_t x) { uint32_t p = 1024; while (p < x) p <<= 1; return p; }

extern "C" const char *rb_last_error(void) { return g_err; }

// A fresh population on the device: counters, packed words, agent records, bitmaps, empty active lists.  `sparse`: the
// arrays hold the end of a previous run (k_init).
static int init_population(rb_engine *e, uint32_t seed, bool sparse) {
    const Eng &G = e->G;
    k_init_counters<<<G.R, 128, 0, e->stream>>>(G, seed, e->cfg.hospital_beds, e->cfg.icu_units);
    if (sparse) k_init<true><<<dim3(e->sweep_blocks, G.R), 256, 0, e->stream>>>(G);
    else k_init<false><<<dim3(e->sweep_blocks, G.R), 256, 0, e->stream>>>(G);
    k_init_bitmaps<<<dim3(8, G.R), 256, 0, e->stream>>>(G);
    k_clear_lists<<<128, 256, 0, e->stream>>>(G);
    k_init_seeds<<<G.R, 128, 0, e->stream>>>(G, e->seed_of_day, seed, 0);
    e->launches += 5;
    CK(cudaGetLastError());
    return 0;
}

static int setup_groups(rb_engine *e, int sms);
static void group_config(int R, int *n_groups, int *wave_pct);

// k_resolve is a chain of dependent scattered accesses per infection (two infections in flight per thread): it wants as
// many threads in flight as a day can bring infections -- up to ~1 / 128 of the agents -- and is indifferent to how many
// of its CTAs find nothing to do.  Measured on the peak day of 256 HUS replicas (us): 2 / 4 / 8 / 16 CTAs per SM in total
// 341 / 350 / 322 / 294; 52 CTAs per replica (13312 in all) 260.
static int resolve_grid(int n_agents, int sms, int pct, int replicas) {
    long long b = ((long long)n_agents / 128 + 255) / 256;
    long long cap = (long long)sms * 16 * pct / 100 / replicas; if (cap < 64) cap = 64;
    if (const char *s = getenv("RB_RESOLVE_BLOCKS")) cap = b = atoi(s);      // measurement aid
    if (b > cap) b = cap;
    return b < 1 ? 1 : (int)b;
}

extern "C" void rb_destroy(rb_engine *e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    cudaStreamSynchronize(e->stream);
    if (e->have_graphs) for (int g = 0; g < e->n_groups; g++) { cudaGraphExecDestroy(e->grp[g].graph[0]); cudaGraphExecDestroy(e->grp[g].graph[1]); }
    for (int g = 0; g < e->n_groups && e->n_groups > 1; g++) {
        cudaStreamDestroy(e->grp[g].stream); cudaEventDestroy(e->grp[g].ev_stagger); cudaEventDestroy(e->grp[g].ev_join);
    }
    if (e->n_groups > 1) cudaEventDestroy(e->ev_fork);
    for (int k = 0; k < e->n_peer_open; k++) if (k != e->G.rank && e->G.xpeer[k]) cudaIpcCloseMemHandle(e->G.xpeer[k]);
    if (e->comm) g_nccl.CommDestroy(e->comm);
    for (void *p : e->allocs) cudaFree(p);
    if (e->h_stage) { cudaFreeHost(e->h_stage); for (int i = 0; i < 4; i++) cudaEventDestroy(e->ev_stage[i]); }
    cudaEventDestroy(e->ev0); cudaEventDestroy(e->ev1);
    cudaStreamDestroy(e->stream);
    delete e;
}

extern "C" int rb_create(const rb_config *cfg, const int32_t *age_counts, const int32_t *group_of_age,
                         const rb_variant *variants, const int32_t *import_lo, const int32_t *import_hi,
                         const float *import_cum, rb_engine **out) {
    if (cfg->n_ages > RB_MAX_AGES || cfg->n_variants > RB_MAX_VARIANTS || cfg->n_import_classes > RB_MAX_IMPORT_CLASSES ||
        cfg->n_groups > 16 || cfg->n_replicas < 1 || cfg->n_agents < 1) {
        snprintf(g_err, sizeof g_err, "config exceeds compiled limits"); return 1;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        snprintf(g_err, sizeof g_err, "no CUDA device: reina_b200 has no CPU fallback"); return 2;
    }
    CK(cudaSetDevice(cfg->device));
    if (const char *s = getenv("RB_L2_FETCH")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(s));   // measurement aid
    rb_engine *e = new rb_engine();
    e->cfg = *cfg; e->day = 0; e->last_ms = 0; e->launches = 0; e->h2d_bytes = 0; e->d2h_bytes = 0; e->have_graphs = false; e->comm = nullptr; e->comm_rank = 0; e->comm_size = 1; e->sharded = false; e->merge_blocks = 1;
    e->has_ipc = false; e->h_stage = nullptr; e->n_stage = 0; e->n_groups = 1; e->wide_ctas = 1; e->n_peer_open = 0; e->launch_err = cudaSuccess; e->shard_timing = getenv("RB_SHARD_TIMING") != nullptr;
    e->xepoch = 0; e->d_xepoch = nullptr; e->d_tx = nullptr; e->d_sx = nullptr; e->d_sx_epoch = nullptr; e->d_branch = nullptr; e->d_move = nullptr;
    { int lo = 0, hi = 0; CK(cudaDeviceGetStreamPriorityRange(&lo, &hi)); e->prio_high = hi; e->prio = (cfg->n_replicas >= 32 && cfg->n_replicas < 128) ? 1 : 0; if (const char *s = getenv("RB_PRIO")) e->prio = atoi(s); }
    CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&e->ev0)); CK(cudaEventCreate(&e->ev1));
    Eng &G = e->G;
    memset(&G, 0, sizeof G);
    const int N = cfg->n_agents, R = cfg->n_replicas;
    G.N = N; G.Npad = (N + 3) & ~3; G.n_ages = cfg->n_ages; G.n_groups = cfg->n_groups; G.n_variants = cfg->n_variants;
    G.R = R; G.max_days = cfg->max_days; G.row_len = RB_N_ATTRS * cfg->n_groups + RB_N_SCALARS;
    G.n_import_classes = cfg->n_import_classes;
    G.rank = 0; G.nranks = 1;
    int bits = 1; while ((1u << bits) < (uint32_t)N) bits++;
    G.fhalf = (bits + 1) / 2;
    e->age_start.resize(cfg->n_ages + 1);
    int64_t tot = 0;
    for (int a = 0; a < cfg->n_ages; a++) { e->age_start[a] = (int32_t)tot; tot += age_counts[a]; }
    e->age_start[cfg->n_ages] = (int32_t)tot;
    if (tot != N) { snprintf(g_err, sizeof g_err, "age_counts sum %lld != n_agents %d", (long long)tot, N); delete e; return 1; }
    // an import class that can be drawn (positive weight, or the last one: the fallback) must hold somebody -- the pick is lo + u32 % size
    for (int i = 0; i < cfg->n_import_classes; i++) {
        const float w = import_cum[i] - (i ? import_cum[i - 1] : 0.0f);
        if (import_lo[i] < 0 || import_hi[i] >= cfg->n_ages || import_lo[i] > import_hi[i]) { snprintf(g_err, sizeof g_err, "import class %d: bad age band", i); delete e; return 1; }
        if ((w > 0.0f || i == cfg->n_import_classes - 1) && e->age_start[import_hi[i] + 1] - e->age_start[import_lo[i]] <= 0) {
            snprintf(g_err, sizeof g_err, "import class %d (ages %d-%d) can be drawn but is empty", i, import_lo[i], import_hi[i]); delete e; return 1;
        }
    }
    float cc = cfg->contact_capacity > 0 ? cfg->contact_capacity : 1.0f;
    G.cap_items = pow2_at_least((uint64_t)((double)N * cc) + 4096);
    // the day's transmissions grow with its contacts (a transmission scale above 1 grows both), so they take the same factor
    G.cap_succ = pow2_at_least((uint64_t)((double)((uint64_t)N / 8) * cc) + 4096);
    G.cap_events = pow2_at_least((uint64_t)N / 16 + 2048);
    G.cap_queue = pow2_at_least((uint64_t)N / 8 + 2048);
    const size_t RN = (size_t)R * G.Npad;
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, cfg->device));
    const int sms = prop.multiProcessorCount;
    {   // Active-list segments (state.cuh, Eng::alist)
        // two per warp of the sweep grid a replica gets in the production geometry (its replica group's share of a wave):
        // a warp streams a segment from end to end, so segments are the unit of load balance -- but every segment costs a
        // dependent round trip to memory before its first entry arrives, so there should not be many more than warps; and
        // none so small that it holds fewer than ~256 agents
        int ng, pct;
        group_config(R, &ng, &pct);
        long long ctas = (long long)sms * SW_CTAS_PER_SM * (ng > 1 ? pct : 100) / 100 / ((R + ng - 1) / ng);      // as setup_groups sizes the grid
        if (ctas < 1) ctas = 1;
        long long S = 2 * ctas * SW_WARPS, most = (long long)N / 256;
        if (S > most) S = most;
        G.n_seg = (uint32_t)(S < 1 ? 1 : S);
        G.seg_cap = ((uint32_t)N + G.n_seg - 1) / G.n_seg;        // agents a with a % n_seg == s: never more than this
    }
    G.sus_words = ((G.Npad + 31) / 32 + 32 + 3) & ~3;     // multiple of 4 words: the sweep reads the bitmaps 16 bytes at a time
    if (dalloc(e, &G.hot, RN) || dalloc(e, &G.perm, RN) || dalloc(e, &G.rec, RN) ||
        dalloc(e, &G.sus, (size_t)R * G.sus_words) || dalloc(e, &G.det, (size_t)R * G.sus_words) || dalloc(e, &G.alist, (size_t)R * 2 * G.n_seg * G.seg_cap) || dalloc(e, &G.seg_n, (size_t)R * 2 * G.n_seg) || dalloc(e, &G.items, (size_t)R * G.cap_items) || dalloc(e, &G.succ, (size_t)R * G.cap_succ) ||
        dalloc(e, &G.ev_key, (size_t)R * G.cap_events) || dalloc(e, &G.ev_agent, (size_t)R * G.cap_events) ||
        dalloc(e, &G.q_key, (size_t)R * 2 * G.cap_queue) || dalloc(e, &G.q_agent, (size_t)R * 2 * G.cap_queue) ||
        dalloc(e, &G.ctr, (size_t)R) || dalloc(e, &G.stats, (size_t)R * (cfg->max_days + 1) * G.row_len) ||
        dalloc(e, &e->seed_of_day, (size_t)R * (cfg->max_days + 1)) ||
        dalloc(e, &e->d_sched, (size_t)cfg->max_days + 1) ||
        dalloc(e, &e->d_moments, 2 * ((size_t)cfg->max_days + 1) * G.row_len + 2)) { rb_destroy(e); return 1; }
    G.sched = e->d_sched;
    e->h_sched.assign(cfg->max_days + 1, rb_day_params());
    e->n_table_slots = 1024;
    if (dalloc(e, &e->d_tables, (size_t)e->n_table_slots)) { rb_destroy(e); return 1; }
    CK(cudaMemset(e->d_tables, 0, sizeof(DevTable *) * e->n_table_slots));
    G.tables = e->d_tables;
    e->tables.assign(e->n_table_slots, nullptr);
    rb_variant *dv; int32_t *d_as, *d_ga, *d_ilo, *d_ihi; float *d_icum; uint8_t *d_ab;
    if (dalloc(e, &dv, (size_t)cfg->n_variants) || dalloc(e, &d_as, (size_t)cfg->n_ages + 1) || dalloc(e, &d_ga, (size_t)cfg->n_ages) ||
        dalloc(e, &d_ilo, (size_t)RB_MAX_IMPORT_CLASSES) || dalloc(e, &d_ihi, (size_t)RB_MAX_IMPORT_CLASSES) ||
        dalloc(e, &d_icum, (size_t)RB_MAX_IMPORT_CLASSES) || dalloc(e, &d_ab, (size_t)(G.Npad >> 10) + 2)) { rb_destroy(e); return 1; }
    {
        std::vector<uint8_t> ab((size_t)(G.Npad >> 10) + 2);
        int age = 0;
        for (size_t b = 0; b < ab.size(); b++) {
            int64_t a = (int64_t)b << 10; if (a > N - 1) a = N - 1;
            while (age < cfg->n_ages - 1 && e->age_start[age + 1] <= a) age++;
            ab[b] = (uint8_t)age;
        }
        CK(cudaMemcpy(d_ab, ab.data(), ab.size(), cudaMemcpyHostToDevice));
    }
    e->h_variants.assign(variants, variants + cfg->n_variants);
    CK(cudaMemcpy(dv, variants, sizeof(rb_variant) * cfg->n_variants, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_as, e->age_start.data(), sizeof(int32_t) * (cfg->n_ages + 1), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ga, group_of_age, sizeof(int32_t) * cfg->n_ages, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ilo, import_lo, sizeof(int32_t) * cfg->n_import_classes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ihi, import_hi, sizeof(int32_t) * cfg->n_import_classes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_icum, import_cum, sizeof(float) * cfg->n_import_classes, cudaMemcpyHostToDevice));
    G.age_blk = d_ab; G.variants = dv; G.age_start = d_as; G.group_of_age = d_ga; G.import_lo = d_ilo; G.import_hi = d_ihi; G.import_cum = d_icum;
    e->age_counts.assign(age_counts, age_counts + cfg->n_ages);
    CK(cudaMemset(G.stats, 0, sizeof(int32_t) * (size_t)R * (cfg->max_days + 1) * G.row_len));
    CK(cudaMemset(e->d_sched, 0, sizeof(rb_day_params) * ((size_t)cfg->max_days + 1)));
    // launch geometry: grid-stride kernels sized in multiples of the SM count
    // the sweep fills the GPU exactly once: SW_CTAS_PER_SM resident CTAs per SM, shared out over the replicas (a grid a
    // little larger than one wave would run its tail on a nearly empty GPU)
    // (a warp per active-list segment is the most a replica can use)
    int want = ((int)G.n_seg + SW_WARPS - 1) / SW_WARPS;
    int per_rep = sms * SW_CTAS_PER_SM / R; if (per_rep < 1) per_rep = 1;
    e->sweep_blocks = want < per_rep ? want : per_rep; if (e->sweep_blocks < 1) e->sweep_blocks = 1;
    e->list_blocks = sms * EX_CTAS_PER_SM / R; if (e->list_blocks < 2) e->list_blocks = 2;
    // k_resolve is a chain of dependent scattered accesses per infection: enough threads for one pass over the day's list
    e->resolve_blocks = resolve_grid(G.N, sms, 100, R);
    if (init_population(e, cfg->seed, false)) { rb_destroy(e); return 1; }
    CK(cudaStreamSynchronize(e->stream));
    if (setup_groups(e, sms)) { rb_destroy(e); return 1; }
    // wide day boundary: only without replica groups (two wide launches on concurrent streams could each hold half
    // the SMs and wait for the other), one CTA per SM at most
    e->wide_ctas = 1;
    // measured at 5 x 10^7 agents, one replica (ms per 180 days): 1 CTA 80.1; 16 CTAs 50.7; 32: 51.8; 64: 56.7 (the grid
    // barrier grows with the team); threshold 2048 / 8192 / 32768 entries: 47.4 / 56.7 / 59.9
    G.wide_min = 2048;
    // ... and on one HUS replica (1.7 x 10^6 agents, at most ~3000 events or tests a day) the team only costs: 10.4 ms per
    // 180 days with it, 9.5 without.  So: populations of 4 x 10^6 agents and more.
    if (e->n_groups == 1 && R * 4 <= sms && N >= 4000000) { e->wide_ctas = 16; while (e->wide_ctas * R > sms) e->wide_ctas >>= 1; }     // a power of two (team sort)
    if (const char *s = getenv("RB_WIDE_CTAS")) { int v = atoi(s); if (v >= 1 && v <= WIDE_MAX_CTAS && v * R <= sms) e->wide_ctas = v; }
    if (const char *s = getenv("RB_WIDE_MIN")) G.wide_min = atoi(s);     // 0: every day is a wide day (tests)
    *out = e;
    return 0;
}

// Replica groups (see rb_engine).  Measured on B200 (HUS, 256 replicas, ms per 180-day step): 1 group 162.7; 2 groups
// with full-wave grids 154.9; 3 x 100 % 152.6; 4 x 50 % 153.0; 4 x 100 % 152.2; 8 x 50 % 156.0 -- the grids are
// oversubscribed on purpose, a group in its latency-bound phase leaves its share of the SMs to the others.
// RB_GROUPS / RB_GROUP_WAVE_PCT override (measurement aid).  Each group's grid covers `pct` % of one wave.
// Round 2, 32 / 64 replicas (the per-GPU share of a 256-seed ensemble on 8 / 4 GPUs): 2 x 100 % 22.7 / 34.4 ms, 4 x 50 % 22.3 /
// 33.6, 4 x 50 % with the latency-bound kernels at high launch priority (rb_engine::prio) 21.5 / 33.0; at 128 and 256
// replicas the priorities gain nothing (57.2 vs 56.9, 106.4 vs 105.1): the SMs are full anyway.
static void group_config(int R, int *n_groups, int *wave_pct) {
    int ng = R >= 32 ? 4 : 1, pct = R >= 32 ? 50 : 100;
    if (const char *s = getenv("RB_GROUPS")) ng = atoi(s);
    if (const char *s = getenv("RB_GROUP_WAVE_PCT")) pct = atoi(s);
    if (pct < 1) pct = 100;
    if (ng > MAX_GROUPS) ng = MAX_GROUPS;
    if (ng > R) ng = R;
    if (ng < 1) ng = 1;
    *n_groups = ng; *wave_pct = pct;
}
static int setup_groups(rb_engine *e, int sms) {
    const int R = e->G.R;
    int ng, pct;
    group_config(R, &ng, &pct);
    e->n_groups = ng;
    if (ng == 1) {      // the whole ensemble on the engine's own stream with the full-wave grids, whatever `pct` says
        ReplicaGroup &q = e->grp[0];
        q.r0 = 0; q.R = R; q.sweep_blocks = e->sweep_blocks; q.list_blocks = e->list_blocks; q.resolve_blocks = e->resolve_blocks;
        q.stream = e->stream;
        return 0;
    }
    CK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    const Eng &G = e->G;
    const int want = ((int)G.n_seg + SW_WARPS - 1) / SW_WARPS;
    for (int g = 0; g < ng; g++) {
        ReplicaGroup &q = e->grp[g];
        q.r0 = (int)((long long)R * g / ng); q.R = (int)((long long)R * (g + 1) / ng) - q.r0;
        int per = sms * SW_CTAS_PER_SM * pct / 100 / q.R; if (per < 1) per = 1;
        q.sweep_blocks = want < per ? want : per;
        q.list_blocks = sms * EX_CTAS_PER_SM * pct / 100 / q.R; if (q.list_blocks < 2) q.list_blocks = 2;
        q.resolve_blocks = resolve_grid(G.N, sms, pct, q.R);
        CK(cudaStreamCreateWithFlags(&q.stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&q.ev_stagger, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&q.ev_join, cudaEventDisableTiming));
    }
    return 0;
}

// Every reset / state load starts a new flag epoch of the population-sharded exchange (shard.cuh).  The epoch lives in a
// device word, not in the kernel arguments, so the captured graphs of sharded days stay valid.
__global__ void k_set_word(uint32_t *p, uint32_t v) { *p = v; }
static void bump_xepoch(rb_engine *e) {
    e->xepoch++;
    if (e->d_xepoch) { k_set_word<<<1, 1, 0, e->stream>>>(e->d_xepoch, e->xepoch); e->launches++; }
}

extern "C" int rb_reset(rb_engine *e, uint32_t seed) {
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    e->cfg.seed = seed;
    e->day = 0;
    bump_xepoch(e);
    if (init_population(e, seed, true)) return 1;
    if (e->has_ipc) {
        k_initial_state<<<e->G.R, 32, 0, e->stream>>>(e->G, e->ipc);
        k_rebuild_lists<<<dim3(e->sweep_blocks, e->G.R), 256, 0, e->stream>>>(e->G);
        e->launches += 2;
    }
    CK(cudaGetLastError());
    return 0;
}

extern "C" int rb_set_initial_state(rb_engine *e, const int32_t *ipc7) {
    CK(cudaSetDevice(e->cfg.device));
    if (e->day != 0 || e->has_ipc) { snprintf(g_err, sizeof g_err, "rb_set_initial_state: once, before the first step"); return 1; }
    for (int i = 0; i < 7; i++) if (ipc7[i] < 0) { snprintf(g_err, sizeof g_err, "rb_set_initial_state: negative count"); return 1; }
    e->ipc.dead = ipc7[0]; e->ipc.in_icu = ipc7[1]; e->ipc.in_ward = ipc7[2]; e->ipc.confirmed = ipc7[3];
    e->ipc.incubating = ipc7[4]; e->ipc.ill = ipc7[5]; e->ipc.recovered = ipc7[6];
    e->has_ipc = true;
    k_initial_state<<<e->G.R, 32, 0, e->stream>>>(e->G, e->ipc);
    k_rebuild_lists<<<dim3(e->sweep_blocks, e->G.R), 256, 0, e->stream>>>(e->G);      // the active lists from the packed words
    e->launches += 2;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

#define TABLE_HOST_BYTES (offsetof(DevTable, guide))      // what the host fills and uploads; the row guide is built on the device
// A pinned staging buffer for table uploads: four slots used round-robin, each guarded by an event, so a run of uploads
// (all mobility epochs of a schedule) is queued as asynchronous copies without a host-device synchronisation per table.
static int stage_slot(rb_engine *e, DevTable **h, int *slot) {
    if (!e->h_stage) {
        CK(cudaMallocHost((void **)&e->h_stage, TABLE_HOST_BYTES * 4));
        for (int i = 0; i < 4; i++) CK(cudaEventCreateWithFlags(&e->ev_stage[i], cudaEventDisableTiming));
        e->n_stage = 0;
    }
    const int k = e->n_stage & 3;
    if (e->n_stage >= 4) CK(cudaEventSynchronize(e->ev_stage[k]));     // the copy that last used this slot has left it
    e->n_stage++;
    *h = (DevTable *)((uint8_t *)e->h_stage + TABLE_HOST_BYTES * k); *slot = k;     // only the host-filled part of a DevTable is staged
    return 0;
}

extern "C" int rb_set_contact_table(rb_engine *e, int32_t epoch, const int32_t *n_rows, const double *cum_p,
                                    const int32_t *age_lo, const int32_t *age_hi, const uint8_t *place,
                                    const float *mask_p, const double *nr_contacts, const double *ncontact_cdf) {
    if (epoch < 0 || epoch >= e->n_table_slots) { snprintf(g_err, sizeof g_err, "table epoch out of range"); return 1; }
    CK(cudaSetDevice(e->cfg.device));
    // a row that can be drawn must have somebody in its contact band: the target index is start + u32 % size
    for (int age = 0; age < e->cfg.n_ages; age++) {
        if (n_rows[age] < 0 || n_rows[age] > RB_MAX_ROWS) { snprintf(g_err, sizeof g_err, "contact table: n_rows[%d] = %d", age, n_rows[age]); return 1; }
        if (e->age_counts[age] == 0) continue;                     // nobody of this age: its rows are never used
        for (int i = 0; i < n_rows[age]; i++) {
            const int k = age * RB_MAX_ROWS + i;
            if (age_lo[k] < 0 || age_hi[k] >= e->cfg.n_ages || age_lo[k] > age_hi[k]) { snprintf(g_err, sizeof g_err, "contact table: bad band [%d, %d] (age %d row %d)", age_lo[k], age_hi[k], age, i); return 1; }
            const double p = cum_p[k] - (i ? cum_p[k - 1] : 0.0);
            const bool last = i == n_rows[age] - 1;                  // the fallback row of the search
            if ((p > 0.0 || last) && e->age_start[age_hi[k] + 1] - e->age_start[age_lo[k]] <= 0) {
                snprintf(g_err, sizeof g_err, "contact table: row %d of age %d can be drawn (p = %g) but its contact band [%d, %d] is empty", i, age, p, age_lo[k], age_hi[k]);
                return 1;
            }
        }
    }
    DevTable *h; int slot;
    if (stage_slot(e, &h, &slot)) return 1;
    // The same table is usually sent again for every new batch of seeds (Context.upload_inputs): the inputs are copied to
    // the device every time, but the derived part (integer thresholds, band offsets, guides) is only recomputed when the
    // arguments differ from what this epoch was last set to.
    const size_t nA = (size_t)e->cfg.n_ages, nAR = nA * RB_MAX_ROWS;
    const void *arg[8] = {n_rows, cum_p, age_lo, age_hi, place, mask_p, nr_contacts, ncontact_cdf};
    const size_t len[8] = {nA * 4, nAR * 8, nAR * 4, nAR * 4, nAR, nAR * 4, nA * 8, nA * 2 * RB_NCDF * 8};
    size_t total = 0; for (int i = 0; i < 8; i++) total += len[i];
    if ((size_t)epoch >= e->table_args.size()) { e->table_args.resize(epoch + 1); e->table_host.resize(epoch + 1); }
    std::vector<uint8_t> &seen = e->table_args[epoch], &built = e->table_host[epoch];
    bool same = seen.size() == total && built.size() == TABLE_HOST_BYTES;
    for (size_t i = 0, off = 0; i < 8 && same; off += len[i], i++) same = memcmp(seen.data() + off, arg[i], len[i]) == 0;
    if (same) memcpy(h, built.data(), TABLE_HOST_BYTES);
    else {
    seen.resize(total);
    for (size_t i = 0, off = 0; i < 8; off += len[i], i++) memcpy(seen.data() + off, arg[i], len[i]);
    memset(h, 0, TABLE_HOST_BYTES);
    for (int age = 0; age < e->cfg.n_ages; age++) {
        h->n_rows[age] = n_rows[age];
        h->nr_contacts[age] = (float)nr_contacts[age];
        memcpy(h->ncdf[age], ncontact_cdf + (size_t)age * 2 * RB_NCDF, sizeof(double) * 2 * RB_NCDF);
        for (int i = 0; i < n_rows[age]; i++) {
            int k = age * RB_MAX_ROWS + i;
            h->cum_p[age][i] = cum_p[k];
            {   // exact: scaling by 2^24 is exact in double, and for integer k, k < x  <=>  k < ceil(x)
                double x = cum_p[k] * 16777216.0, cx = (double)(uint64_t)x;
                if (cx < x) cx += 1.0;
                h->cum24[age][i] = cx >= 4294967295.0 ? 0xffffffffu : (uint32_t)cx;
            }
            h->start[age][i] = e->age_start[age_lo[k]];
            h->size[age][i] = e->age_start[age_hi[k] + 1] - e->age_start[age_lo[k]];
            h->place[age][i] = place[k];
            h->lo_age[age][i] = (uint8_t)age_lo[k]; h->hi_age[age][i] = (uint8_t)age_hi[k];
            bool uni = true;
            for (int v = 0; v < e->cfg.n_variants; v++)
                for (int g = age_lo[k]; g <= age_hi[k]; g++)
                    if (e->h_variants[v].tab[RB_T_SUSCEPTIBILITY][g] != e->h_variants[v].tab[RB_T_SUSCEPTIBILITY][age_lo[k]]) uni = false;
            h->susc_uniform[age][i] = uni ? 1 : 0;
            h->mask_p[age][i] = mask_p[k];
        }
    }
    for (int age = 0; age < e->cfg.n_ages; age++)
        for (int cls = 0; cls < 2; cls++)
            for (int b = 0, k = 0; b < 256; b++) {
                const int limit = cls ? 5 : 100;
                while (k < limit && !(h->ncdf[age][cls][k] > (double)b / 256.0)) k++;
                // every u of the cell, b/256 <= u < (b+1)/256, draws k iff cdf[k] reaches the cell's end (or k is the cap)
                const bool exact = k >= limit || h->ncdf[age][cls][k] >= (double)(b + 1) / 256.0;
                h->nguide[age][cls][b] = (uint8_t)(k | (exact ? 0 : 128));
            }
    built.assign((const uint8_t *)h, (const uint8_t *)h + TABLE_HOST_BYTES);
    }
    DevTable *d = e->tables[epoch];
    if (!d) {
        if (dalloc(e, &d, 1)) return 1;
        e->tables[epoch] = d;
        CK(cudaMemcpyAsync(e->d_tables + epoch, &e->tables[epoch], sizeof(DevTable *), cudaMemcpyHostToDevice, e->stream));
    }
    // stream order keeps the copy behind every kernel of earlier steps (the replica-group streams join e->stream)
    CK(cudaMemcpyAsync(d, h, TABLE_HOST_BYTES, cudaMemcpyHostToDevice, e->stream));
    CK(cudaEventRecord(e->ev_stage[slot], e->stream));
    k_build_guide<<<e->cfg.n_ages, 256, 0, e->stream>>>(d, e->cfg.n_ages); e->launches++;
    CK(cudaGetLastError());
    e->h2d_bytes += (int64_t)TABLE_HOST_BYTES;
    return 0;
}

extern "C" int rb_set_schedule(rb_engine *e, int32_t day0, int32_t n, const rb_day_params *params) {
    if (day0 < 0 || day0 + n > e->cfg.max_days + 1) { snprintf(g_err, sizeof g_err, "schedule out of range"); return 1; }
    CK(cudaSetDevice(e->cfg.device));
    memcpy(e->h_sched.data() + day0, params, sizeof(rb_day_params) * n);
    CK(cudaMemcpyAsync(e->d_sched + day0, e->h_sched.data() + day0, sizeof(rb_day_params) * n, cudaMemcpyHostToDevice, e->stream));
    e->h2d_bytes += (int64_t)sizeof(rb_day_params) * n;
    return 0;
}

// Launch of a per-day kernel.  (Programmatic dependent launch -- cudaLaunchAttributeProgrammaticStreamSerialization with a
// griddepcontrol.wait at the head of every kernel, captured into the graphs as programmatic edges -- was built and
// measured here: bit-exact, but no gain over plain graph edges for one replica (52.5 vs 50.7 us per day) and a loss for
// ensembles (256 replicas 116.9 vs 104.2 ms: the early-scheduled CTAs of a group's next kernel hold SM slots that another
// group's running kernel could use).  Removed again.)
// `urgent`: the latency-bound kernels of a day (k_resolve, the day boundary) are launched with the highest priority, so
// that their few CTAs are placed before the pending CTAs of another replica group's oversubscribed sweep / contact grids.
template <typename K>
static void launch_k(rb_engine *e, K kernel, dim3 grid, int threads, cudaStream_t st, const Eng &G, bool urgent = false) {
    if (!urgent || !e->prio) { kernel<<<grid, threads, 0, st>>>(G); return; }
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = grid; cfg.blockDim = dim3(threads); cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributePriority; at[0].val.priority = e->prio_high;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t err = cudaLaunchKernelEx(&cfg, kernel, G);
    if (err != cudaSuccess && e->launch_err == cudaSuccess) e->launch_err = err;
}

// The day boundary: one CTA per replica, or -- few replicas of a large population -- a cooperative launch of
// wide_ctas co-resident CTAs per replica (boundary.cuh, Team).  kind: 0 = k_pre, 1 = k_post, 2 = k_between.
static void launch_boundary(rb_engine *e, int kind, int R, cudaStream_t st, const Eng &G) {
    if (e->wide_ctas <= 1) {
        if (kind == 0) launch_k(e, k_pre<false>, dim3(R), PRE_THREADS, st, G, true);
        else if (kind == 1) launch_k(e, k_post<false>, dim3(R), PRE_THREADS, st, G, true);
        else launch_k(e, k_between<false>, dim3(R), PRE_THREADS, st, G, true);
        return;
    }
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(e->wide_ctas, R); cfg.blockDim = dim3(PRE_THREADS); cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;     // all CTAs co-resident: the team's grid barrier needs it
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t err;
    if (kind == 0) err = cudaLaunchKernelEx(&cfg, k_pre<true>, G);
    else if (kind == 1) err = cudaLaunchKernelEx(&cfg, k_post<true>, G);
    else err = cudaLaunchKernelEx(&cfg, k_between<true>, G);
    if (err != cudaSuccess && e->launch_err == cudaSuccess) e->launch_err = err;     // reported by the rb_step that issued it
}

// One "segment" = the grid kernels of day d followed by the fused day boundary d -> d+1, for one replica group.
// No kernel takes the day as an argument (each replica carries its own day counter and reads the schedule from
// device memory), so a captured graph of GRAPH_DAYS segments is replayed for any stretch of days.
static void launch_group_segment(rb_engine *e, const ReplicaGroup &q, bool stagger_mark) {
    Eng G = e->G; G.r0 = q.r0;
    launch_k(e, k_sweep, dim3(q.sweep_blocks, q.R), SW_THREADS, q.stream, G);
    launch_k(e, k_expose, dim3(q.list_blocks, q.R), EX_THREADS, q.stream, G);
    if (stagger_mark) cudaEventRecord(q.ev_stagger, q.stream);       // the next group starts its day here
    launch_k(e, k_resolve<true>, dim3(q.resolve_blocks, q.R), 256, q.stream, G, true);
    launch_boundary(e, 2, q.R, q.stream, G);
}

#define GRAPH_DAYS 16
static int build_graphs(rb_engine *e) {
    for (int g = 0; g < e->n_groups; g++)
        for (int which = 0; which < 2; which++) {
            ReplicaGroup &q = e->grp[g];
            int nseg = which == 0 ? GRAPH_DAYS : 1;
            cudaGraph_t gr;
            CK(cudaStreamBeginCapture(q.stream, cudaStreamCaptureModeThreadLocal));
            for (int i = 0; i < nseg; i++) launch_group_segment(e, q, false);
            CK(cudaStreamEndCapture(q.stream, &gr));
            CK(cudaGraphInstantiate(&q.graph[which], gr, e->prio ? cudaGraphInstantiateFlagUseNodePriority : 0));
            CK(cudaGraphDestroy(gr));
        }
    e->have_graphs = true;
    return 0;
}


// ---------------------------------------------------------------- ensemble communicator (BASELINE configs[3])
// The Monte-Carlo ensemble shards as independent replicas per GPU; the only exchange is the final reduce of the daily
// curves.  One process per GPU joins an NCCL communicator through its engine handle (the unique id comes from
// rb_shard_unique_id and reaches the other ranks by any host-side means), and the reduce runs on device buffers: no
// other framework is involved.
extern "C" int rb_comm_init(rb_engine *e, int32_t rank, int32_t nranks, const uint8_t *uid128) {
    if (nranks < 1 || rank < 0 || rank >= nranks) { snprintf(g_err, sizeof g_err, "bad rank %d / %d", rank, nranks); return 1; }
    if (e->comm) { snprintf(g_err, sizeof g_err, "rb_comm_init: this engine already has a communicator"); return 1; }
    if (load_nccl()) return 1;
    CK(cudaSetDevice(e->cfg.device));
    ncclUniqueId id; memcpy(&id, uid128, 128);
    NK(g_nccl.CommInitRank(&e->comm, nranks, id, rank));
    e->comm_rank = rank; e->comm_size = nranks;
    return 0;
}
extern "C" int32_t rb_comm_rank(rb_engine *e) { return e->comm_rank; }
extern "C" int32_t rb_comm_size(rb_engine *e) { return e->comm_size; }

// scratch on the device for host-buffer collectives: the moments buffer if it is large enough, else a temporary
static int comm_scratch(rb_engine *e, size_t bytes, void **p, bool *temp) {
    const size_t have = sizeof(double) * (2 * ((size_t)e->cfg.max_days + 1) * e->G.row_len + 2);
    if (bytes <= have) { *p = e->d_moments; *temp = false; return 0; }
    CK(cudaMalloc(p, bytes)); *temp = true;
    return 0;
}

// In-place all-reduce of n doubles held by the host.  op: 0 = sum, 1 = max.  Doubles as a barrier (n = 1).
extern "C" int rb_comm_allreduce(rb_engine *e, double *inout, int64_t n, int32_t op) {
    if (n < 0 || (op != 0 && op != 1)) { snprintf(g_err, sizeof g_err, "rb_comm_allreduce: bad arguments"); return 1; }
    if (!e->comm || e->comm_size == 1 || n == 0) return 0;
    CK(cudaSetDevice(e->cfg.device));
    void *d; bool temp;
    if (comm_scratch(e, sizeof(double) * (size_t)n, &d, &temp)) return 1;
    CK(cudaMemcpyAsync(d, inout, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    NK(g_nccl.AllReduce(d, d, (size_t)n, ncclDouble, op == 0 ? ncclSum : ncclMax, e->comm, e->stream));
    CK(cudaMemcpyAsync(inout, d, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (temp) cudaFree(d);
    return 0;
}

// All-gather of `bytes` bytes per rank between host buffers: out[rank k] = in of rank k.
extern "C" int rb_comm_allgather(rb_engine *e, const void *in, void *out, int64_t bytes) {
    if (bytes < 0) { snprintf(g_err, sizeof g_err, "rb_comm_allgather: bad size"); return 1; }
    if (!e->comm || e->comm_size == 1) { memcpy(out, in, (size_t)bytes); return 0; }
    CK(cudaSetDevice(e->cfg.device));
    void *d; bool temp;
    if (comm_scratch(e, (size_t)bytes * e->comm_size, &d, &temp)) return 1;
    uint8_t *mine = (uint8_t *)d + (size_t)bytes * e->comm_rank;
    CK(cudaMemcpyAsync(mine, in, (size_t)bytes, cudaMemcpyHostToDevice, e->stream));
    NK(g_nccl.AllGather(mine, d, (size_t)bytes, ncclChar, e->comm, e->stream));
    CK(cudaMemcpyAsync(out, d, (size_t)bytes * e->comm_size, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (temp) cudaFree(d);
    return 0;
}

// ---------------------------------------------------------------- population-sharded mode
extern "C" int rb_shard_unique_id(uint8_t *out128) {
    if (load_nccl()) return 1;
    ncclUniqueId id;
    NK(g_nccl.GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    memcpy(out128, &id, 128);
    return 0;
}

// What every way of joining shares: rank / size, the message capacities, the epoch word, the merge grid.
static int shard_prepare(rb_engine *e, int32_t rank, int32_t nranks, float exchange_capacity) {
    if (nranks < 1 || nranks > MAX_RANKS || rank < 0 || rank >= nranks) { snprintf(g_err, sizeof g_err, "bad rank %d / %d", rank, nranks); return 1; }
    if (e->G.R != 1) { snprintf(g_err, sizeof g_err, "population-sharded mode runs one replica (n_replicas = %d)", e->G.R); return 1; }
    // (have_graphs: stepped and reset -- grp[0].graph would hold unsharded days, build_shard_graphs puts sharded ones there)
    if (e->day != 0 || e->have_graphs || e->comm || e->sharded) { snprintf(g_err, sizeof g_err, "rb_shard_init must be the first call after rb_create"); return 1; }
    CK(cudaSetDevice(e->cfg.device));
    Eng &G = e->G;
    // message capacities: this rank's share of the agents; a day's state changes / transmissions / tests / capacity
    // events are small fractions of it (peak day of the reference epidemic: 0.9 % / 0.5 % / 0.17 % / 0.08 % of the
    // agents; ~2.3x headroom each, exchange_capacity scales them, overflow is a loud RB_OTHER_FAILURE)
    const double share = (double)G.N / nranks * (exchange_capacity > 0 ? exchange_capacity : 1.0);
    G.xcap_upd = (uint32_t)(share / 48) + 4096;
    G.xcap_succ = (uint32_t)(share / 96) + 4096;
    G.xcap_q = (uint32_t)(share / 256) + 2048;
    G.xcap_ev = (uint32_t)(share / 512) + 2048;
    G.xslot = xslot_bytes(G.xcap_q, G.xcap_ev, G.xcap_upd, G.xcap_succ);
    G.rank = rank; G.nranks = nranks;
    e->comm_rank = rank; e->comm_size = nranks;
    e->xepoch = 1;
    if (dalloc(e, &e->d_xepoch, 1)) return 1;
    CK(cudaMemcpy(e->d_xepoch, &e->xepoch, sizeof(uint32_t), cudaMemcpyHostToDevice));
    G.xepoch = e->d_xepoch;
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, e->cfg.device));
    // (the sweep needs no adjustment: a rank's active list holds only the agents it owns, ~1 / nranks of the infected)
    e->merge_blocks = prop.multiProcessorCount * 8 / nranks * nranks;      // a multiple of nranks: k_merge deals its blocks to the ranks
    return 0;
}

extern "C" int rb_shard_init(rb_engine *e, int32_t rank, int32_t nranks, const uint8_t *uid128, float exchange_capacity) {
    if (shard_prepare(e, rank, nranks, exchange_capacity)) return 1;
    if (load_nccl()) return 1;
    ncclUniqueId id; memcpy(&id, uid128, 128);
    NK(g_nccl.CommInitRank(&e->comm, nranks, id, rank));
    e->sharded = true;
    Eng &G = e->G;
    // Exchange through peer memory when every rank can map every other rank's buffer (CUDA IPC; one process per GPU on
    // one NVLink box), else -- no peer access, RB_SHARD_EXCHANGE=nccl -- through ncclAllGather.
    {
        const char *mode = getenv("RB_SHARD_EXCHANGE");
        int ok = !(mode && strcmp(mode, "nccl") == 0);
        const size_t own_bytes = XFLAG_BYTES + 2 * G.xslot;
        uint8_t *own = nullptr;
        struct Hello { cudaIpcMemHandle_t h; int32_t ok; int32_t pad[15]; };
        static_assert(sizeof(Hello) == 128, "Hello is one 128-byte record");
        std::vector<Hello> all(nranks);
        Hello *d_all = nullptr;
        if (dalloc(e, &d_all, (size_t)nranks)) return 1;
        if (ok && cudaMalloc((void **)&own, own_bytes) != cudaSuccess) { cudaGetLastError(); ok = 0; own = nullptr; }
        Hello me; memset(&me, 0, sizeof me);
        if (ok && nranks > 1 && cudaIpcGetMemHandle(&me.h, own) != cudaSuccess) { cudaGetLastError(); ok = 0; }
        me.ok = ok;
        auto gather = [&]() -> int {       // everybody learns everybody's record
            CK(cudaMemcpy(d_all + rank, &me, sizeof me, cudaMemcpyHostToDevice));
            NK(g_nccl.AllGather(d_all + rank, d_all, sizeof(Hello), ncclChar, e->comm, e->stream));
            CK(cudaStreamSynchronize(e->stream));
            CK(cudaMemcpy(all.data(), d_all, sizeof(Hello) * nranks, cudaMemcpyDeviceToHost));
            return 0;
        };
        if (gather()) return 1;
        for (int k = 0; k < nranks; k++) ok = ok && all[k].ok;
        if (ok) {
            for (int k = 0; k < nranks; k++) {
                if (k == rank) { G.xpeer[k] = own; continue; }
                void *q = nullptr;
                if (cudaIpcOpenMemHandle(&q, all[k].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
                G.xpeer[k] = (uint8_t *)q; e->n_peer_open = k + 1;
            }
            me.ok = ok;
            if (gather()) return 1;        // second round: did every rank open every handle?
            for (int k = 0; k < nranks; k++) ok = ok && all[k].ok;
        }
        if (ok) {
            e->allocs.push_back(own);
            CK(cudaMemset(own, 0, own_bytes));
            G.xbuf = own; G.xp2p = 1;
            // nobody may publish before every rank has cleared its flag line
            if (gather()) return 1;
        } else {
            for (int k = 0; k < e->n_peer_open; k++) if (k != rank && G.xpeer[k]) cudaIpcCloseMemHandle(G.xpeer[k]);
            e->n_peer_open = 0; memset(G.xpeer, 0, sizeof G.xpeer);
            if (own) cudaFree(own);
            G.xp2p = 0;
            if (dalloc(e, &G.xbuf, G.xslot * nranks)) return 1;
            CK(cudaMemset(G.xbuf, 0, G.xslot * nranks));
        }
    }
    return 0;
}

static int build_shard_graphs(rb_engine *e);

// The ranks of ONE process (a host that drives several GPUs itself, or -- the tests on a single-GPU box -- several
// engines on one device, each on its own stream): no NCCL, no CUDA IPC; a rank's message buffer is a plain device
// pointer the others read directly (same device, or peer access enabled here).  Every engine must be driven by its own
// host thread, or at least have its rb_step calls issued before anybody waits for one of them: a rank's day cannot end
// before every other rank's sweep of that day has been launched.
extern "C" int rb_shard_init_local(rb_engine **engines, int32_t nranks, float exchange_capacity) {
    if (nranks < 1 || nranks > MAX_RANKS) { snprintf(g_err, sizeof g_err, "bad number of ranks %d", nranks); return 1; }
    for (int k = 0; k < nranks; k++) {
        for (int j = 0; j < k; j++) if (engines[j] == engines[k]) { snprintf(g_err, sizeof g_err, "rb_shard_init_local: the same engine twice"); return 1; }
        if (engines[k]->G.N != engines[0]->G.N) { snprintf(g_err, sizeof g_err, "rb_shard_init_local: engines of different populations"); return 1; }
    }
    uint8_t *bufs[MAX_RANKS];
    for (int k = 0; k < nranks; k++) {
        rb_engine *e = engines[k];
        if (shard_prepare(e, k, nranks, exchange_capacity)) return 1;
        const size_t own_bytes = XFLAG_BYTES + 2 * e->G.xslot;
        if (dalloc(e, &bufs[k], own_bytes)) return 1;
        CK(cudaMemset(bufs[k], 0, own_bytes));
    }
    for (int k = 0; k < nranks; k++) {
        rb_engine *e = engines[k];
        CK(cudaSetDevice(e->cfg.device));
        for (int j = 0; j < nranks; j++) {
            const int dj = engines[j]->cfg.device;
            if (dj != e->cfg.device) {
                int can = 0; CK(cudaDeviceCanAccessPeer(&can, e->cfg.device, dj));
                if (!can) { snprintf(g_err, sizeof g_err, "rb_shard_init_local: device %d cannot access device %d", e->cfg.device, dj); return 1; }
                cudaError_t err = cudaDeviceEnablePeerAccess(dj, 0);
                if (err != cudaSuccess && err != cudaErrorPeerAccessAlreadyEnabled) { snprintf(g_err, sizeof g_err, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(err)); return 1; }
                cudaGetLastError();
            }
            e->G.xpeer[j] = bufs[j];
        }
        e->G.xbuf = bufs[k]; e->G.xp2p = 1; e->sharded = true;
    }
    // Everything a step needs is created NOW, while no rank is waiting for another: a first launch loads its kernel
    // lazily and graph instantiation allocates, both of which may synchronise with the device -- which never returns
    // while a peer's k_wait is spinning for the very rank that is stuck in the load.
    for (int k = 0; k < nranks; k++) {
        rb_engine *e = engines[k];
        CK(cudaSetDevice(e->cfg.device));
        cudaFuncAttributes fa;
        CK(cudaFuncGetAttributes(&fa, k_pre<false>)); CK(cudaFuncGetAttributes(&fa, k_pre<true>));
        CK(cudaFuncGetAttributes(&fa, k_post<false>)); CK(cudaFuncGetAttributes(&fa, k_post<true>));
        CK(cudaFuncGetAttributes(&fa, k_between<false>)); CK(cudaFuncGetAttributes(&fa, k_between<true>));
        CK(cudaFuncGetAttributes(&fa, k_sweep)); CK(cudaFuncGetAttributes(&fa, k_expose));
        CK(cudaFuncGetAttributes(&fa, k_publish)); CK(cudaFuncGetAttributes(&fa, k_wait)); CK(cudaFuncGetAttributes(&fa, k_merge));
        CK(cudaFuncGetAttributes(&fa, k_resolve<false>)); CK(cudaFuncGetAttributes(&fa, k_resolve<true>));
        CK(cudaFuncGetAttributes(&fa, k_set_word));
        if (!e->shard_timing && build_shard_graphs(e)) return 1;
    }
    for (int k = 0; k < nranks; k++) { CK(cudaSetDevice(engines[k]->cfg.device)); CK(cudaDeviceSynchronize()); }
    return 0;
}

extern "C" int32_t rb_shard_rank(rb_engine *e) { return e->G.rank; }
extern "C" int32_t rb_shard_nranks(rb_engine *e) { return e->G.nranks; }
extern "C" int64_t rb_shard_message_bytes(rb_engine *e) { return e->sharded ? (int64_t)e->G.xslot : 0; }
extern "C" int32_t rb_shard_exchange(rb_engine *e) { return !e->sharded ? 0 : (e->G.xp2p ? 2 : 1); }

// One simulated day in sharded mode: sweep and contacts over the owned stripes, the exchange of the ranks' messages
// (flags in peer memory, or one all-gather), then merge / resolve / day boundary replicated on every rank.
static int launch_day_sharded(rb_engine *e, bool last) {
    const Eng &G = e->G;
    cudaStream_t st = e->stream;
    // RB_SHARD_TIMING (measurement aid): device time per phase, summed over the days of the step, printed by rb_sync
    auto mark = [&]() { if (e->shard_timing) { cudaEvent_t ev; cudaEventCreate(&ev); cudaEventRecord(ev, st); e->shard_events.push_back(ev); } };
    mark();
    k_sweep<<<dim3(e->sweep_blocks, 1), SW_THREADS, 0, st>>>(G);
    mark();
    k_expose<<<dim3(e->list_blocks, 1), EX_THREADS, 0, st>>>(G);
    mark();
    if (G.xp2p) { k_publish<<<1, 32, 0, st>>>(G); k_wait<<<1, 32, 0, st>>>(G); }      // raise the own flag, wait for every peer's
    else NK(g_nccl.AllGather(G.xbuf + (size_t)G.rank * G.xslot, G.xbuf, G.xslot, ncclChar, e->comm, st));
    mark();
    k_merge<<<e->merge_blocks, 256, 0, st>>>(G);
    mark();
    if (last) k_resolve<false><<<dim3(e->resolve_blocks, 1), 256, 0, st>>>(G); else k_resolve<true><<<dim3(e->resolve_blocks, 1), 256, 0, st>>>(G);
    mark();
    launch_boundary(e, last ? 1 : 2, 1, st, G);
    mark();
    return 0;
}
#define SHARD_LAUNCHES_PER_DAY(G) ((G).xp2p ? 7 : 5)

// Sharded days with the peer-memory exchange are pure kernel chains (the flag wait is a kernel too) that take no
// per-day argument -- the day and the flag epoch are read from device memory -- so they are captured once, as graphs of
// GRAPH_DAYS days and of one day, and replayed like the single-GPU segments.  They are kept as the graphs of the one
// replica group a sharded engine has (one replica): its unsharded graphs are never built.
static int build_shard_graphs(rb_engine *e) {
    for (int which = 0; which < 2; which++) {
        const int nseg = which == 0 ? GRAPH_DAYS : 1;
        cudaGraph_t g;
        CK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
        for (int i = 0; i < nseg; i++) if (launch_day_sharded(e, false)) { cudaStreamEndCapture(e->stream, &g); return 1; }
        CK(cudaStreamEndCapture(e->stream, &g));
        CK(cudaGraphInstantiate(&e->grp[0].graph[which], g, 0));
        CK(cudaGraphDestroy(g));
    }
    e->have_graphs = true;
    return 0;
}

// what every stepping entry point checks first: the range of days and that each day's contact table was uploaded
static int check_days(rb_engine *e, int32_t n_days) {
    if (n_days < 0) { snprintf(g_err, sizeof g_err, "negative number of days"); return 1; }
    if (e->day + n_days > e->cfg.max_days) { snprintf(g_err, sizeof g_err, "max_days exceeded"); return 1; }
    for (int d = 0; d < n_days; d++) {
        int ep = e->h_sched[e->day + d].table_epoch;
        if (ep < 0 || ep >= e->n_table_slots || !e->tables[ep]) { snprintf(g_err, sizeof g_err, "contact table %d not set", ep); return 1; }
    }
    return 0;
}
static int check_launches(rb_engine *e) {
    CK(cudaGetLastError());
    if (e->launch_err != cudaSuccess) {
        snprintf(g_err, sizeof g_err, "cooperative launch of the day boundary failed: %s", cudaGetErrorString(e->launch_err));
        e->launch_err = cudaSuccess;
        return 1;
    }
    return 0;
}

extern "C" int rb_step(rb_engine *e, int32_t n_days) {
    CK(cudaSetDevice(e->cfg.device));
    if (check_days(e, n_days)) return 1;
    if (n_days == 0) return 0;
    if (!e->sharded && !e->have_graphs && build_graphs(e)) return 1;
    const Eng &G = e->G;
    const int R = G.R;
    if (e->sharded) {
        const bool graphs = G.xp2p && !e->shard_timing;
        if (graphs && !e->have_graphs && build_shard_graphs(e)) return 1;
        CK(cudaEventRecord(e->ev0, e->stream));
        launch_boundary(e, 0, 1, e->stream, G); e->launches++;
        int mid = n_days - 1;
        if (graphs) {
            while (mid >= GRAPH_DAYS) { CK(cudaGraphLaunch(e->grp[0].graph[0], e->stream)); mid -= GRAPH_DAYS; }
            while (mid > 0) { CK(cudaGraphLaunch(e->grp[0].graph[1], e->stream)); mid -= 1; }
        } else for (; mid > 0; mid--) if (launch_day_sharded(e, false)) return 1;
        if (launch_day_sharded(e, true)) return 1;
        e->launches += (int64_t)n_days * SHARD_LAUNCHES_PER_DAY(G);
        CK(cudaEventRecord(e->ev1, e->stream));
        if (check_launches(e)) return 1;
        e->day += n_days;
        return 0;
    }
    const int ng = e->n_groups;
    CK(cudaEventRecord(e->ev0, e->stream));
    launch_boundary(e, 0, R, e->stream, G); e->launches++;
    if (ng > 1) CK(cudaEventRecord(e->ev_fork, e->stream));
    for (int g = 0; g < ng; g++) {
        ReplicaGroup &q = e->grp[g];
        int mid = n_days - 1;
        if (ng > 1) {
            CK(cudaStreamWaitEvent(q.stream, e->ev_fork, 0));
            if (g > 0 && mid > 0) CK(cudaStreamWaitEvent(q.stream, e->grp[g - 1].ev_stagger, 0));     // half a day behind the previous group
            if (mid > 0) { launch_group_segment(e, q, g + 1 < ng); mid -= 1; e->launches += 4; }
        }
        while (mid >= GRAPH_DAYS) { CK(cudaGraphLaunch(q.graph[0], q.stream)); mid -= GRAPH_DAYS; e->launches += 4 * GRAPH_DAYS; }
        while (mid > 0) { CK(cudaGraphLaunch(q.graph[1], q.stream)); mid -= 1; e->launches += 4; }
        Eng Gq = G; Gq.r0 = q.r0;
        launch_k(e, k_sweep, dim3(q.sweep_blocks, q.R), SW_THREADS, q.stream, Gq);
        launch_k(e, k_expose, dim3(q.list_blocks, q.R), EX_THREADS, q.stream, Gq);
        launch_k(e, k_resolve<false>, dim3(q.resolve_blocks, q.R), 256, q.stream, Gq, true);
        launch_boundary(e, 1, q.R, q.stream, Gq);
        e->launches += 4;
        if (ng > 1) { CK(cudaEventRecord(q.ev_join, q.stream)); CK(cudaStreamWaitEvent(e->stream, q.ev_join, 0)); }
    }
    CK(cudaEventRecord(e->ev1, e->stream));
    if (check_launches(e)) return 1;
    e->day += n_days;
    return 0;
}

// rb_step with CUDA events around every launch, one kernel at a time on ONE stream with full-wave grids (no replica
// groups, no graphs): what each kernel costs when it has the GPU to itself.
extern "C" int rb_step_profiled(rb_engine *e, int32_t n_days, float *ms_per_kernel) {
    CK(cudaSetDevice(e->cfg.device));
    if (e->sharded) { snprintf(g_err, sizeof g_err, "rb_step_profiled: not available in population-sharded mode"); return 1; }
    if (check_days(e, n_days)) return 1;
    for (int k = 0; k < RB_N_KERNELS; k++) ms_per_kernel[k] = 0;
    if (n_days == 0) return 0;
    const Eng &G = e->G;
    const int R = G.R;
    std::vector<cudaEvent_t> ev((size_t)n_days * 6);
    for (auto &x : ev) CK(cudaEventCreate(&x));
    for (int d = 0; d < n_days; d++) {
        cudaEvent_t *v = &ev[(size_t)d * 6];
        CK(cudaEventRecord(v[0], e->stream));
        launch_boundary(e, 0, R, e->stream, G); CK(cudaEventRecord(v[1], e->stream));
        k_sweep<<<dim3(e->sweep_blocks, R), SW_THREADS, 0, e->stream>>>(G); CK(cudaEventRecord(v[2], e->stream));
        k_expose<<<dim3(e->list_blocks, R), EX_THREADS, 0, e->stream>>>(G); CK(cudaEventRecord(v[3], e->stream));
        k_resolve<false><<<dim3(e->resolve_blocks, R), 256, 0, e->stream>>>(G); CK(cudaEventRecord(v[4], e->stream));
        launch_boundary(e, 1, R, e->stream, G); CK(cudaEventRecord(v[5], e->stream));
        e->launches += 5;
    }
    const int bad = check_launches(e);
    CK(cudaStreamSynchronize(e->stream));
    if (!bad)
        for (int d = 0; d < n_days; d++)
            for (int k = 0; k < RB_N_KERNELS; k++) { float ms = 0; CK(cudaEventElapsedTime(&ms, ev[(size_t)d * 6 + k], ev[(size_t)d * 6 + k + 1])); ms_per_kernel[k] += ms; }
    for (auto &x : ev) cudaEventDestroy(x);
    if (bad) return 1;
    e->day += n_days;
    return 0;
}

// The PRODUCTION launch geometry of rb_step -- the replica groups on their concurrent streams, staggered, with the
// grids rb_step uses -- with CUDA events around every launch on the stream it is launched on (kernels are launched one
// by one instead of from graphs so that events can sit between them).  ms_per_kernel[k] sums the event-to-event time of
// kernel k over all its launches, launches_per_kernel[k] counts them (order: pre, sweep, expose, resolve, post/between);
// wall_ms is the whole run.  With several groups the launches of different groups overlap, so the sum of all kernel times
// exceeds wall_ms: a launch's duration here is what it takes WHILE sharing the GPU with the other groups' kernels.
extern "C" int rb_step_timed(rb_engine *e, int32_t n_days, float *ms_per_kernel, int32_t *launches_per_kernel, float *wall_ms) {
    CK(cudaSetDevice(e->cfg.device));
    if (e->sharded) { snprintf(g_err, sizeof g_err, "rb_step_timed: not available in population-sharded mode"); return 1; }
    if (check_days(e, n_days)) return 1;
    for (int k = 0; k < RB_N_KERNELS; k++) { ms_per_kernel[k] = 0; launches_per_kernel[k] = 0; }
    *wall_ms = 0;
    if (n_days == 0) return 0;
    const Eng &G = e->G;
    const int R = G.R;
    struct Span { cudaEvent_t a, b; int k; };
    std::vector<Span> spans;
    auto mark = [&](cudaStream_t st) { cudaEvent_t x; cudaEventCreate(&x); cudaEventRecord(x, st); return x; };
    const int ng = e->n_groups;
    CK(cudaEventRecord(e->ev0, e->stream));
    { cudaEvent_t a = mark(e->stream); launch_boundary(e, 0, R, e->stream, G); spans.push_back({a, mark(e->stream), 0}); e->launches++; }
    if (ng > 1) CK(cudaEventRecord(e->ev_fork, e->stream));
    for (int d = 0; d < n_days; d++) {
        const bool last = d == n_days - 1;
        for (int g = 0; g < ng; g++) {
            ReplicaGroup &q = e->grp[g];
            if (ng > 1 && d == 0) {
                CK(cudaStreamWaitEvent(q.stream, e->ev_fork, 0));
                if (g > 0 && n_days > 1) CK(cudaStreamWaitEvent(q.stream, e->grp[g - 1].ev_stagger, 0));
            }
            Eng Gq = G; Gq.r0 = q.r0;
            cudaEvent_t t0 = mark(q.stream);
            k_sweep<<<dim3(q.sweep_blocks, q.R), SW_THREADS, 0, q.stream>>>(Gq);
            cudaEvent_t t1 = mark(q.stream);
            k_expose<<<dim3(q.list_blocks, q.R), EX_THREADS, 0, q.stream>>>(Gq);
            cudaEvent_t t2 = mark(q.stream);
            if (ng > 1 && d == 0 && g + 1 < ng && n_days > 1) CK(cudaEventRecord(q.ev_stagger, q.stream));
            if (last) k_resolve<false><<<dim3(q.resolve_blocks, q.R), 256, 0, q.stream>>>(Gq);
            else k_resolve<true><<<dim3(q.resolve_blocks, q.R), 256, 0, q.stream>>>(Gq);
            cudaEvent_t t3 = mark(q.stream);
            launch_boundary(e, last ? 1 : 2, q.R, q.stream, Gq);
            cudaEvent_t t4 = mark(q.stream);
            spans.push_back({t0, t1, 1}); spans.push_back({t1, t2, 2}); spans.push_back({t2, t3, 3}); spans.push_back({t3, t4, 4});
            e->launches += 4;
            if (ng > 1 && last) { CK(cudaEventRecord(q.ev_join, q.stream)); CK(cudaStreamWaitEvent(e->stream, q.ev_join, 0)); }
        }
    }
    CK(cudaEventRecord(e->ev1, e->stream));
    const int bad = check_launches(e);
    CK(cudaStreamSynchronize(e->stream));
    if (!bad) {
        for (const Span &s : spans) { float ms = 0; CK(cudaEventElapsedTime(&ms, s.a, s.b)); ms_per_kernel[s.k] += ms; launches_per_kernel[s.k]++; }
        CK(cudaEventElapsedTime(wall_ms, e->ev0, e->ev1));
    }
    std::vector<cudaEvent_t> seen;
    for (const Span &s : spans) { seen.push_back(s.a); seen.push_back(s.b); }
    std::sort(seen.begin(), seen.end());
    seen.erase(std::unique(seen.begin(), seen.end()), seen.end());
    for (cudaEvent_t x : seen) cudaEventDestroy(x);
    if (bad) return 1;
    e->day += n_days;
    return 0;
}

extern "C" int rb_sync(rb_engine *e) {
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    float ms = 0;
    if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) == cudaSuccess) e->last_ms = ms; else cudaGetLastError();
    if (!e->shard_events.empty()) {
        double t[6] = {0, 0, 0, 0, 0, 0};
        for (size_t d = 0; d + 7 <= e->shard_events.size(); d += 7)
            for (int k = 0; k < 6; k++) { float x = 0; if (cudaEventElapsedTime(&x, e->shard_events[d + k], e->shard_events[d + k + 1]) == cudaSuccess) t[k] += x; }
        fprintf(stderr, "[rank %d] %zu days: sweep %.2f  expose %.2f  exchange+wait %.2f  merge %.2f  resolve %.2f  boundary %.2f ms (step %.2f)\n",
                e->G.rank, e->shard_events.size() / 7, t[0], t[1], t[2], t[3], t[4], t[5], e->last_ms);
        for (cudaEvent_t ev : e->shard_events) cudaEventDestroy(ev);
        e->shard_events.clear();
    }
    return 0;
}

extern "C" int32_t rb_day(rb_engine *e) { return e->day; }
extern "C" void rb_debug_flag(rb_engine *e, int32_t v) { e->G.dbg = v; }
extern "C" int rb_debug_phase_cycles(rb_engine *e, int32_t replica, long long *out16) {
    cudaSetDevice(e->cfg.device); cudaStreamSynchronize(e->stream);
    RepCtr c; if (cudaMemcpy(&c, &e->G.ctr[replica], sizeof c, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    memcpy(out16, c.dbg_t, sizeof c.dbg_t); return 0;
}
// The random blocks behind every draw, computed on the host by the very functions the kernels inline (rng.cuh): lets a
// CPU-only test pin them to the published Random123 known-answer vectors.
extern "C" int rb_rng_block(int32_t words, uint32_t key, const uint32_t *ctr, uint32_t *out) {
    if (words == 4) { const u32x4 x = philox(key, ctr[0], ctr[1], ctr[2], ctr[3]); out[0] = x.x; out[1] = x.y; out[2] = x.z; out[3] = x.w; return 0; }
    snprintf(g_err, sizeof g_err, "rb_rng_block: words must be 4");
    return 1;
}
extern "C" int32_t rb_row_len(rb_engine *e) { return e->G.row_len; }
extern "C" float rb_last_step_ms(rb_engine *e) { return e->last_ms; }
extern "C" int64_t rb_launch_count(rb_engine *e) { return e->launches; }
extern "C" int64_t rb_copied_bytes(rb_engine *e, int32_t direction) { return direction == 0 ? e->h2d_bytes : e->d2h_bytes; }

extern "C" int rb_snapshot(rb_engine *e) {
    CK(cudaSetDevice(e->cfg.device));
    k_snapshot<<<e->G.R, 256, 0, e->stream>>>(e->G); e->launches++;
    CK(cudaGetLastError());
    return 0;
}

extern "C" int rb_read_stats(rb_engine *e, int32_t day0, int32_t n, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    if (day0 < 0 || day0 + n > e->cfg.max_days + 1) { snprintf(g_err, sizeof g_err, "stats range"); return 1; }
    const Eng &G = e->G;
    CK(cudaMemcpy2DAsync(out, sizeof(int32_t) * (size_t)n * G.row_len,
                         G.stats + (size_t)day0 * G.row_len, sizeof(int32_t) * (size_t)(G.max_days + 1) * G.row_len,
                         sizeof(int32_t) * (size_t)n * G.row_len, G.R, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->d2h_bytes += (int64_t)sizeof(int32_t) * n * G.row_len * G.R;
    return 0;
}

extern "C" int rb_read_moments(rb_engine *e, int32_t day0, int32_t n, double *sum, double *sumsq) {
    CK(cudaSetDevice(e->cfg.device));
    if (day0 < 0 || n < 1 || day0 + n > e->cfg.max_days + 1) { snprintf(g_err, sizeof g_err, "stats range"); return 1; }
    const size_t cnt = (size_t)n * e->G.row_len;
    double *d = e->d_moments;           // allocated once by rb_create for max_days + 1 rows
    k_moments<<<n, 160, 0, e->stream>>>(e->G, day0, d, d + cnt); e->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(sum, d, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(sumsq, d + cnt, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->d2h_bytes += (int64_t)sizeof(double) * 2 * cnt;
    return 0;
}


// rb_read_moments over the whole ensemble: the moments of this GPU's replicas are reduced on the device, summed over the
// communicator's ranks with one ncclAllReduce (sum, sum of squares and the replica count travel together), and only the
// result crosses to the host.  Without a communicator it is rb_read_moments plus the local replica count.
extern "C" int rb_reduce_moments(rb_engine *e, int32_t day0, int32_t n, double *sum, double *sumsq, int64_t *n_replicas) {
    CK(cudaSetDevice(e->cfg.device));
    if (day0 < 0 || n < 1 || day0 + n > e->cfg.max_days + 1) { snprintf(g_err, sizeof g_err, "stats range"); return 1; }
    const size_t cnt = (size_t)n * e->G.row_len;
    double *d = e->d_moments;
    k_moments<<<n, 160, 0, e->stream>>>(e->G, day0, d, d + cnt); e->launches++;
    CK(cudaGetLastError());
    double nrep = (double)e->G.R;
    CK(cudaMemcpyAsync(d + 2 * cnt, &nrep, sizeof(double), cudaMemcpyHostToDevice, e->stream));
    if (e->comm && e->comm_size > 1 && !e->sharded) NK(g_nccl.AllReduce(d, d, 2 * cnt + 1, ncclDouble, ncclSum, e->comm, e->stream));
    CK(cudaMemcpyAsync(sum, d, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(sumsq, d + cnt, sizeof(double) * cnt, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(&nrep, d + 2 * cnt, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->h2d_bytes += 8; e->d2h_bytes += (int64_t)sizeof(double) * (2 * cnt + 1);
    *n_replicas = (int64_t)(nrep + 0.5);
    return 0;
}

extern "C" int rb_read_per_age(rb_engine *e, int32_t replica, int32_t attr, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    if (replica < 0 || replica >= e->G.R || attr < 0 || attr >= RB_N_ATTRS) { snprintf(g_err, sizeof g_err, "bad replica/attr"); return 1; }
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy(out, &e->G.ctr[replica].counts[attr][0], sizeof(int32_t) * e->cfg.n_ages, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int rb_problem(rb_engine *e, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    // one strided copy: the problem word of every replica's counter block
    CK(cudaMemcpy2D(out, sizeof(int32_t), &e->G.ctr[0].problem, sizeof(RepCtr), sizeof(int32_t), (size_t)e->G.R, cudaMemcpyDeviceToHost));
    e->d2h_bytes += (int64_t)sizeof(int32_t) * e->G.R;
    return 0;
}

extern "C" int rb_sample(rb_engine *e, int32_t what, int32_t age, int32_t severity, int32_t n, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    if (what < 0 || what > 6 || age < 0 || age >= e->cfg.n_ages) { snprintf(g_err, sizeof g_err, "bad sample request"); return 1; }
    int32_t *d; CK(cudaMalloc(&d, sizeof(int32_t) * n));
    int epoch = e->h_sched[e->day > 0 ? e->day - 1 : 0].table_epoch;
    k_sample<<<(n + 255) / 256, 256, 0, e->stream>>>(e->G, e->cfg.seed, what, age, severity, n, epoch, d); e->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy(out, d, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    cudaFree(d);
    return 0;
}

extern "C" int rb_read_agents(rb_engine *e, int32_t replica, rb_agent *out) {
    CK(cudaSetDevice(e->cfg.device));
    const Eng &G = e->G;
    if (replica < 0 || replica >= G.R) { snprintf(g_err, sizeof g_err, "bad replica"); return 1; }
    // the current day counters live in the active lists: write them back into the packed words first
    k_flush_lists<<<dim3(e->sweep_blocks, G.R), 256, 0, e->stream>>>(G); e->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    const int N = G.N; const size_t base = (size_t)replica * G.Npad;
    std::vector<uint32_t> hot(N), cold(N); std::vector<int32_t> inf(N); std::vector<int16_t> vd(N);
    CK(cudaMemcpy(hot.data(), G.hot + base, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost));
    {
        std::vector<AgentRec> rec(N);
        CK(cudaMemcpy(rec.data(), G.rec + base, sizeof(AgentRec) * N, cudaMemcpyDeviceToHost));
        for (int a = 0; a < N; a++) { cold[a] = rec[a].cold; inf[a] = rec[a].infector; vd[a] = rec[a].vacc_day; }
    }
    for (int a = 0; a < N; a++) {
        uint32_t h = hot[a]; rb_agent *o = &out[a];
        o->infector = inf[a]; o->n_infected = (int32_t)(cold[a] & 0xffffu);
        o->days_left = (int16_t)H_DL(h); o->day_of_illness = (int16_t)H_DOI(h); o->day_of_vaccination = vd[a];
        o->state = (uint8_t)H_STATE(h); o->severity = (uint8_t)H_SEV(h); o->variant = (uint8_t)H_VAR(h);
        o->flags = (uint8_t)(((h & H_DET) ? 1 : 0) | ((h & H_QUEUED) ? 2 : 0) | ((h & H_INCL) ? 4 : 0) | ((h & H_LIST) ? 8 : 0));
        o->ward_days = (uint8_t)((cold[a] >> 16) & 255u); o->icu_days = (uint8_t)((cold[a] >> 24) & 255u);
    }
    return 0;
}

// ---------------------------------------------------------------- transmission statistics (transmission.cuh)
extern "C" int32_t rb_transmission_len(rb_engine *e) { return tx_layout(e->cfg.max_days, e->cfg.n_groups).len; }

extern "C" int rb_transmission_stats(rb_engine *e, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    const Eng &G = e->G;
    const TxLayout L = tx_layout(G.max_days, G.n_groups);
    const size_t bytes = sizeof(int32_t) * (size_t)G.R * L.len, smem = sizeof(int32_t) * (size_t)L.len;
    if (!e->d_tx && dalloc(e, &e->d_tx, (size_t)G.R * L.len)) return 1;
    // shared counts of one replica: beyond the default 48 KB only for a max_days above ~4000
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(k_transmission, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // every state change is written to `hot` at once; the flush adds the day counters, so that these tables describe the
    // same `hot` that rb_read_agents / rb_save_state see
    k_flush_lists<<<dim3(e->sweep_blocks, G.R), 256, 0, e->stream>>>(G);
    CK(cudaMemsetAsync(e->d_tx, 0, bytes, e->stream));
    int sms = 0; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
    // about two waves of 256-thread CTAs over all replicas, and no CTA without agents
    const int per_rep = std::max(1, std::min((2 * sms * (2048 / TX_THREADS) + G.R - 1) / G.R, (G.N + TX_THREADS - 1) / TX_THREADS));
    k_transmission<<<dim3(per_rep, G.R), TX_THREADS, smem, e->stream>>>(G, L, e->d_tx);
    e->launches += 2;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, e->d_tx, bytes, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->d2h_bytes += (int64_t)bytes;
    return 0;
}

extern "C" int rb_read_infection_days(rb_engine *e, int32_t replica, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    const Eng &G = e->G;
    if (replica < 0 || replica >= G.R) { snprintf(g_err, sizeof g_err, "bad replica"); return 1; }
    k_flush_lists<<<dim3(e->sweep_blocks, G.R), 256, 0, e->stream>>>(G);
    int32_t *d; CK(cudaMallocAsync(&d, sizeof(int32_t) * G.N, e->stream));
    k_infection_days<<<(G.N + 255) / 256, 256, 0, e->stream>>>(G, replica, d);
    e->launches += 2;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d, sizeof(int32_t) * G.N, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaFreeAsync(d, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->d2h_bytes += (int64_t)sizeof(int32_t) * G.N;
    return 0;
}

extern "C" int32_t rb_transmission_settings_len(rb_engine *e) { return sx_layout(e->cfg.max_days, e->cfg.n_groups).len; }

// The epochs of the completed days come from the caller: after rb_load_state into a fresh engine the device schedule of
// the past days was never uploaded, while the caller replays its plan.  Checked against the tables that have been set,
// then copied to d_sx_epoch, after the flush of the active lists that every read of the tree starts with.
static int settings_prologue(rb_engine *e, const int32_t *epoch_of_day, int32_t n_days) {
    if (n_days != e->day) { snprintf(g_err, sizeof g_err, "transmission settings: %d epochs given, %d days completed", n_days, e->day); return 1; }
    for (int d = 0; d < n_days; d++) {
        const int ep = epoch_of_day[d];
        if (ep < 0 || ep >= e->n_table_slots || !e->tables[ep]) { snprintf(g_err, sizeof g_err, "transmission settings: day %d: contact table %d not set", d, ep); return 1; }
    }
    if (!e->d_sx_epoch && dalloc(e, &e->d_sx_epoch, (size_t)e->cfg.max_days + 1)) return 1;
    if (n_days > 0) CK(cudaMemcpyAsync(e->d_sx_epoch, epoch_of_day, sizeof(int32_t) * n_days, cudaMemcpyHostToDevice, e->stream));
    e->h2d_bytes += (int64_t)sizeof(int32_t) * n_days;
    k_flush_lists<<<dim3(e->sweep_blocks, e->G.R), 256, 0, e->stream>>>(e->G);
    e->launches++;
    return 0;
}

extern "C" int rb_transmission_settings(rb_engine *e, const int32_t *epoch_of_day, int32_t n_days, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    const Eng &G = e->G;
    const SxLayout L = sx_layout(G.max_days, G.n_groups);
    const size_t bytes = sizeof(int32_t) * (size_t)G.R * L.len, smem = sizeof(int32_t) * (size_t)L.len;
    // shared counts of one replica: 29 kB at 600 days and 16 groups; beyond 48 kB only with the opt-in
    int smem_max = 0; CK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, e->cfg.device));
    if (smem > (size_t)smem_max) { snprintf(g_err, sizeof g_err, "transmission settings: %zu bytes of tables per replica exceed %d bytes of shared memory (max_days too large)", smem, smem_max); return 1; }
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(k_transmission_settings, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (!e->d_sx && dalloc(e, &e->d_sx, (size_t)G.R * L.len)) return 1;
    if (settings_prologue(e, epoch_of_day, n_days)) return 1;
    CK(cudaMemsetAsync(e->d_sx, 0, bytes, e->stream));
    int sms = 0; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
    // the geometry of k_transmission: about two waves of 256-thread CTAs over all replicas, and no CTA without agents
    const int per_rep = std::max(1, std::min((2 * sms * (2048 / TX_THREADS) + G.R - 1) / G.R, (G.N + TX_THREADS - 1) / TX_THREADS));
    k_transmission_settings<<<dim3(per_rep, G.R), TX_THREADS, smem, e->stream>>>(G, L, e->d_sx_epoch, e->seed_of_day, e->d_sx);
    e->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, e->d_sx, bytes, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->d2h_bytes += (int64_t)bytes;
    return 0;
}

extern "C" int rb_read_infection_places(rb_engine *e, int32_t replica, const int32_t *epoch_of_day, int32_t n_days, int32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    const Eng &G = e->G;
    if (replica < 0 || replica >= G.R) { snprintf(g_err, sizeof g_err, "bad replica"); return 1; }
    if (settings_prologue(e, epoch_of_day, n_days)) return 1;
    int32_t *d; CK(cudaMallocAsync(&d, sizeof(int32_t) * G.N, e->stream));
    k_infection_places<<<(G.N + 255) / 256, 256, 0, e->stream>>>(G, replica, e->d_sx_epoch, e->seed_of_day, d);
    e->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d, sizeof(int32_t) * G.N, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaFreeAsync(d, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->d2h_bytes += (int64_t)sizeof(int32_t) * G.N;
    return 0;
}

extern "C" int rb_read_queue(rb_engine *e, int32_t replica, int32_t *out, int32_t cap, int32_t *n) {
    CK(cudaSetDevice(e->cfg.device));
    const Eng &G = e->G;
    CK(cudaStreamSynchronize(e->stream));
    RepCtr c; CK(cudaMemcpy(&c, &G.ctr[replica], sizeof c, cudaMemcpyDeviceToHost));
    *n = (int32_t)c.n_queue;
    int m = (int)c.n_queue < cap ? (int)c.n_queue : cap;
    if (m > 0) CK(cudaMemcpy(out, G.q_agent + ((size_t)replica * 2 + c.qsel) * G.cap_queue, sizeof(int32_t) * m, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int rb_read_available(rb_engine *e, int32_t replica, int32_t *o) {
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    RepCtr c; CK(cudaMemcpy(&c, &e->G.ctr[replica], sizeof c, cudaMemcpyDeviceToHost));
    o[0] = c.avail_beds; o[1] = c.avail_icu;
    return 0;
}

// ---------------------------------------------------------------- checkpoint / resume
// The reference keeps its state only in process memory (SURVEY section 5: no checkpointing); a device-resident run
// of many replicas is worth saving.  The blob is the engine's whole mutable state between two rb_step calls.
struct StateHeader {
    uint64_t magic; int32_t version, n_agents, n_replicas, n_ages, row_len, max_days, day, sus_words;
    uint32_t cap_queue; uint32_t seed; int32_t rec_bytes, ctr_bytes;
};
#define STATE_MAGIC 0x3030324252414e49ull      // "INARB200"
struct StatePart { void *dev; size_t bytes; };
static std::vector<StatePart> state_parts(rb_engine *e) {
    const Eng &G = e->G;
    const size_t RN = (size_t)G.R * G.Npad, RW = (size_t)G.R * G.sus_words, RQ = (size_t)G.R * 2 * G.cap_queue;
    return {
        {G.hot, RN * sizeof(uint32_t)}, {G.rec, RN * sizeof(AgentRec)}, {G.sus, RW * sizeof(uint32_t)}, {G.det, RW * sizeof(uint32_t)},
        {G.ctr, (size_t)G.R * sizeof(RepCtr)}, {G.q_key, RQ * sizeof(unsigned long long)}, {G.q_agent, RQ * sizeof(int32_t)},
        {G.stats, (size_t)G.R * (G.max_days + 1) * G.row_len * sizeof(int32_t)},
        {e->seed_of_day, (size_t)G.R * (G.max_days + 1) * sizeof(uint32_t)},      // since version 3: the last part
    };
}
static StateHeader state_header(rb_engine *e) {
    const Eng &G = e->G;
    StateHeader h; memset(&h, 0, sizeof h);
    h.magic = STATE_MAGIC; h.version = 3; h.n_agents = G.N; h.n_replicas = G.R; h.n_ages = G.n_ages; h.row_len = G.row_len;
    h.max_days = G.max_days; h.day = e->day; h.sus_words = G.sus_words; h.cap_queue = G.cap_queue; h.seed = e->cfg.seed;
    h.rec_bytes = (int32_t)sizeof(AgentRec); h.ctr_bytes = (int32_t)sizeof(RepCtr);
    return h;
}

extern "C" int64_t rb_state_bytes(rb_engine *e) {
    size_t n = sizeof(StateHeader);
    for (const StatePart &p : state_parts(e)) n += p.bytes;
    return (int64_t)n;
}

extern "C" int rb_save_state(rb_engine *e, void *out, int64_t capacity) {
    CK(cudaSetDevice(e->cfg.device));
    if (capacity < rb_state_bytes(e)) { snprintf(g_err, sizeof g_err, "rb_save_state: buffer of %lld bytes, need %lld", (long long)capacity, (long long)rb_state_bytes(e)); return 1; }
    // the active lists are not part of the blob: their day counters are written back into the packed words here and
    // rb_load_state rebuilds the lists from those
    k_flush_lists<<<dim3(e->sweep_blocks, e->G.R), 256, 0, e->stream>>>(e->G); e->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    uint8_t *o = (uint8_t *)out;
    const StateHeader h = state_header(e);
    memcpy(o, &h, sizeof h); o += sizeof h;
    for (const StatePart &p : state_parts(e)) { CK(cudaMemcpy(o, p.dev, p.bytes, cudaMemcpyDeviceToHost)); o += p.bytes; }
    return 0;
}

// A version-2 blob (saved before the seed history existed) lacks the last part; its history is filled from the loaded
// counters' seeds, which is what it was before any rb_branch.
extern "C" int rb_load_state(rb_engine *e, const void *in, int64_t n_bytes) {
    CK(cudaSetDevice(e->cfg.device));
    std::vector<StatePart> parts = state_parts(e);
    const int64_t v2_bytes = rb_state_bytes(e) - (int64_t)parts.back().bytes;
    StateHeader h; memset(&h, 0, sizeof h);
    if (n_bytes >= (int64_t)sizeof h) memcpy(&h, in, sizeof h);
    const bool v2 = h.version == 2 && n_bytes == v2_bytes;
    if (n_bytes != rb_state_bytes(e) && !v2) { snprintf(g_err, sizeof g_err, "rb_load_state: %lld bytes, this engine's state is %lld", (long long)n_bytes, (long long)rb_state_bytes(e)); return 1; }
    if (v2) parts.pop_back();
    StateHeader w = state_header(e); w.day = h.day; w.seed = h.seed; if (v2) w.version = 2;
    if (memcmp(&h, &w, sizeof h) != 0) { snprintf(g_err, sizeof g_err, "rb_load_state: the blob was saved by an engine of another shape (agents / replicas / max_days / build)"); return 1; }
    if (h.day < 0 || h.day > e->cfg.max_days) { snprintf(g_err, sizeof g_err, "rb_load_state: bad day"); return 1; }
    CK(cudaStreamSynchronize(e->stream));
    const uint8_t *o = (const uint8_t *)in + sizeof h;
    for (const StatePart &p : parts) { CK(cudaMemcpy(p.dev, o, p.bytes, cudaMemcpyHostToDevice)); o += p.bytes; }
    // every segment counter to zero, then lists `lsel` of every replica from the packed words
    k_clear_lists<<<128, 256, 0, e->stream>>>(e->G);
    k_rebuild_lists<<<dim3(e->sweep_blocks, e->G.R), 256, 0, e->stream>>>(e->G);
    e->launches += 2;
    if (v2) { k_init_seeds<<<e->G.R, 128, 0, e->stream>>>(e->G, e->seed_of_day, 0u, 1); e->launches++; }
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    e->day = h.day; e->cfg.seed = h.seed;
    bump_xepoch(e);
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

// ---------------------------------------------------------------- branching replicas (branch.cuh)
// Every stream that may still run a kernel of this engine: its own and those of the replica groups (a branch copies
// across groups).
static int sync_all_streams(rb_engine *e) {
    CK(cudaStreamSynchronize(e->stream));
    for (int g = 0; g < e->n_groups && e->n_groups > 1; g++) CK(cudaStreamSynchronize(e->grp[g].stream));
    return 0;
}

extern "C" int rb_branch(rb_engine *e, const int32_t *src, const uint32_t *seed) {
    CK(cudaSetDevice(e->cfg.device));
    const Eng &G = e->G;
    const int R = G.R;
    if (e->sharded) { snprintf(g_err, sizeof g_err, "rb_branch: not available in population-sharded mode (one replica, per-agent state split over the ranks)"); return 1; }
    int n_copy = 0;
    for (int j = 0; j < R; j++) {
        if (src[j] < 0 || src[j] >= R) { snprintf(g_err, sizeof g_err, "rb_branch: src[%d] = %d is not a replica (0 .. %d)", j, src[j], R - 1); return 1; }
        if (src[src[j]] != src[j]) { snprintf(g_err, sizeof g_err, "rb_branch: src[%d] = %d is itself copied from %d (chained sources)", j, src[j], src[src[j]]); return 1; }
        n_copy += src[j] != j;
    }
    if (sync_all_streams(e)) return 1;
    if (!e->d_branch && dalloc(e, &e->d_branch, 2 * (size_t)R)) return 1;
    CK(cudaMemcpyAsync(e->d_branch, src, sizeof(int32_t) * R, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(e->d_branch + R, seed, sizeof(uint32_t) * R, cudaMemcpyHostToDevice, e->stream));
    e->h2d_bytes += (int64_t)8 * R;
    const int32_t *d_src = e->d_branch; const uint32_t *d_seed = (const uint32_t *)(e->d_branch + R);
    int sms = 0; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
    // about 16 CTAs per SM over the copied replicas; the columns of replicas that keep their state exit at once
    const int per_rep = std::max(1, std::min(1024, sms * 16 / std::max(1, n_copy)));
    // the day counters live in the active lists: into the packed words first, so that the copies carry them
    k_flush_lists<<<dim3(e->sweep_blocks, R), 256, 0, e->stream>>>(G);
    k_branch_copy<<<dim3(per_rep, R), 256, 0, e->stream>>>(G, e->seed_of_day, d_src, d_seed, e->day);
    if (n_copy) k_branch_rebuild<<<dim3(e->sweep_blocks, R), 256, 0, e->stream>>>(G, d_src);
    e->launches += n_copy ? 3 : 2;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

extern "C" int rb_read_seeds(rb_engine *e, uint32_t *out) {
    CK(cudaSetDevice(e->cfg.device));
    if (sync_all_streams(e)) return 1;
    const size_t bytes = sizeof(uint32_t) * (size_t)e->G.R * (e->G.max_days + 1);
    CK(cudaMemcpy(out, e->seed_of_day, bytes, cudaMemcpyDeviceToHost));
    e->d2h_bytes += (int64_t)bytes;
    return 0;
}

// ---------------------------------------------------------------- per-replica scales (RepCtr::tscale_m1, sscale_m1)
// `k` scales per replica, stored as f - 1 in `k` consecutive floats of every replica's counter block starting at `field`
// (a member of G.ctr[0]).  One strided copy into (or out of) them, as rb_problem reads `problem`; every value is checked
// before anything is written, so a refused call changes nothing.
static int set_replica_scales(rb_engine *e, const char *fn, float *field, int k, const float *scale) {
    CK(cudaSetDevice(e->cfg.device));
    const int R = e->G.R;
    std::vector<float> m1((size_t)R * k);
    for (int i = 0; i < R * k; i++) {
        if (!(scale[i] > 0.0f && scale[i] <= 16.0f)) {
            if (k == 1) snprintf(g_err, sizeof g_err, "%s: scale[%d] = %g is not in (0, 16]", fn, i, (double)scale[i]);
            else snprintf(g_err, sizeof g_err, "%s: scale[%d][%d] = %g is not in (0, 16]", fn, i / k, i % k, (double)scale[i]);
            return 1;
        }
        m1[i] = scale[i] - 1.0f;
    }
    if (sync_all_streams(e)) return 1;
    CK(cudaMemcpy2DAsync(field, sizeof(RepCtr), m1.data(), sizeof(float) * k, sizeof(float) * k, (size_t)R, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->h2d_bytes += (int64_t)sizeof(float) * k * R;
    return 0;
}

static int read_replica_scales(rb_engine *e, const float *field, int k, float *out) {
    CK(cudaSetDevice(e->cfg.device));
    if (sync_all_streams(e)) return 1;
    CK(cudaMemcpy2D(out, sizeof(float) * k, field, sizeof(RepCtr), sizeof(float) * k, (size_t)e->G.R, cudaMemcpyDeviceToHost));
    for (int i = 0; i < e->G.R * k; i++) out[i] = 1.0f + out[i];
    e->d2h_bytes += (int64_t)sizeof(float) * k * e->G.R;
    return 0;
}

extern "C" int rb_set_transmission_scale(rb_engine *e, const float *scale) {
    return set_replica_scales(e, "rb_set_transmission_scale", &e->G.ctr[0].tscale_m1, 1, scale);
}

extern "C" int rb_read_transmission_scale(rb_engine *e, float *out) {
    return read_replica_scales(e, &e->G.ctr[0].tscale_m1, 1, out);
}

extern "C" int rb_set_severity_scale(rb_engine *e, const float *scale) {
    return set_replica_scales(e, "rb_set_severity_scale", e->G.ctr[0].sscale_m1, 3, scale);
}

extern "C" int rb_read_severity_scale(rb_engine *e, float *out) {
    return read_replica_scales(e, e->G.ctr[0].sscale_m1, 3, out);
}

// ---------------------------------------------------------------- moving replicas between engines and GPUs (branch.cuh)
// A replica record: this header, then the replica's slice of every state part, in the order of state_parts.  Every part
// is [R][per-replica bytes], so a record is read and written with one plain copy per part, straight from and into the
// state arrays.  The header holds what must match for the bytes to mean the same thing in another engine; the replica
// count and the launch geometry need not (the active lists are rebuilt in the destination's own segments).
struct ReplicaHeader {
    uint64_t magic; int32_t version, n_agents, npad, n_ages, row_len, max_days, sus_words;
    uint32_t cap_queue; int32_t rec_bytes, ctr_bytes, day, reserved[3];
};
static_assert(sizeof(ReplicaHeader) == 64, "ReplicaHeader is 64 bytes");
#define REPLICA_MAGIC 0x3150455252414e49ull    // "INARREP1"

static ReplicaHeader replica_header(rb_engine *e) {
    const Eng &G = e->G;
    ReplicaHeader h; memset(&h, 0, sizeof h);
    h.magic = REPLICA_MAGIC; h.version = 1; h.n_agents = G.N; h.npad = G.Npad; h.n_ages = G.n_ages; h.row_len = G.row_len;
    h.max_days = G.max_days; h.sus_words = G.sus_words; h.cap_queue = G.cap_queue;
    h.rec_bytes = (int32_t)sizeof(AgentRec); h.ctr_bytes = (int32_t)sizeof(RepCtr); h.day = e->day;
    return h;
}

// replica r's slice of every part of state_parts
static std::vector<StatePart> replica_parts(rb_engine *e, int r) {
    std::vector<StatePart> v = state_parts(e);
    for (StatePart &p : v) { p.bytes /= (size_t)e->G.R; p.dev = (uint8_t *)p.dev + (size_t)r * p.bytes; }
    return v;
}

extern "C" int64_t rb_replica_bytes(rb_engine *e) {
    size_t n = sizeof(ReplicaHeader);
    for (const StatePart &p : replica_parts(e, 0)) n += p.bytes;
    return (int64_t)n;
}

// The checks every move makes of the engine that is written.  Returns 1 with g_err set.
static int check_slots(rb_engine *e, const char *fn, int32_t n, const int32_t *slot) {
    const int R = e->G.R;
    if (e->sharded) { snprintf(g_err, sizeof g_err, "%s: not available in population-sharded mode", fn); return 1; }
    if (n < 0 || n > R) { snprintf(g_err, sizeof g_err, "%s: %d slots for %d replicas", fn, n, R); return 1; }
    std::vector<char> seen(R, 0);
    for (int j = 0; j < n; j++) {
        if (slot[j] < 0 || slot[j] >= R) { snprintf(g_err, sizeof g_err, "%s: slot[%d] = %d is not a replica (0 .. %d)", fn, j, slot[j], R - 1); return 1; }
        if (seen[slot[j]]) { snprintf(g_err, sizeof g_err, "%s: slot %d is written twice", fn, slot[j]); return 1; }
        seen[slot[j]] = 1;
    }
    return 0;
}
static int check_sources(rb_engine *e, const char *fn, int32_t n, const int32_t *idx) {
    if (e->sharded) { snprintf(g_err, sizeof g_err, "%s: not available in population-sharded mode", fn); return 1; }
    if (n < 0) { snprintf(g_err, sizeof g_err, "%s: negative count", fn); return 1; }
    for (int j = 0; j < n; j++)
        if (idx[j] < 0 || idx[j] >= e->G.R) { snprintf(g_err, sizeof g_err, "%s: index[%d] = %d is not a replica (0 .. %d)", fn, j, idx[j], e->G.R - 1); return 1; }
    return 0;
}
// Records of another shape, build or day than engine e's (h.day against e's day first: the more useful message).
static int check_header(rb_engine *e, const char *fn, const ReplicaHeader &h, int j) {
    ReplicaHeader w = replica_header(e);
    if (h.magic == w.magic && h.day != w.day) { snprintf(g_err, sizeof g_err, "%s: record %d is of day %d, the engine is at day %d", fn, j, h.day, w.day); return 1; }
    if (memcmp(&h, &w, sizeof h) != 0) { snprintf(g_err, sizeof g_err, "%s: record %d was made by an engine of another shape (agents / ages / max_days / build)", fn, j); return 1; }
    return 0;
}

// After the bytes of n records were queued on e->stream into slots slot[0..n): the seeds, the seed history from today
// on, then the active lists and perm of the written slots (k_branch_rebuild with -1 marking them).  Waits for the end.
static int finish_import(rb_engine *e, int32_t n, const int32_t *slot, const uint32_t *seed) {
    const Eng &G = e->G;
    const int R = G.R;
    if (n > 0) {
        if (!e->d_move && dalloc(e, &e->d_move, 3 * (size_t)R)) return 1;
        std::vector<int32_t> h(2 * (size_t)n + R);
        for (int j = 0; j < n; j++) { h[j] = slot[j]; h[n + j] = (int32_t)seed[j]; }
        for (int r = 0; r < R; r++) h[2 * n + r] = r;
        for (int j = 0; j < n; j++) h[2 * n + slot[j]] = -1;
        CK(cudaMemcpyAsync(e->d_move, h.data(), sizeof(int32_t) * h.size(), cudaMemcpyHostToDevice, e->stream));
        e->h2d_bytes += (int64_t)sizeof(int32_t) * h.size();
        k_import_fixup<<<n, 256, 0, e->stream>>>(G, e->seed_of_day, e->d_move, (const uint32_t *)(e->d_move + n), e->day);
        k_branch_rebuild<<<dim3(e->sweep_blocks, R), 256, 0, e->stream>>>(G, e->d_move + 2 * n);
        e->launches += 2;
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

// the day counters live in the active lists: into the packed words first, so that a record carries them (as rb_save_state)
static int flush_for_export(rb_engine *e) {
    if (sync_all_streams(e)) return 1;
    k_flush_lists<<<dim3(e->sweep_blocks, e->G.R), 256, 0, e->stream>>>(e->G); e->launches++;
    CK(cudaGetLastError());
    return 0;
}

extern "C" int rb_export_replicas(rb_engine *e, int32_t n, const int32_t *idx, void *out, int64_t capacity) {
    CK(cudaSetDevice(e->cfg.device));
    if (check_sources(e, "rb_export_replicas", n, idx)) return 1;
    const int64_t rb = rb_replica_bytes(e);
    if (capacity < rb * n) { snprintf(g_err, sizeof g_err, "rb_export_replicas: buffer of %lld bytes, need %lld", (long long)capacity, (long long)(rb * n)); return 1; }
    if (flush_for_export(e)) return 1;
    const ReplicaHeader h = replica_header(e);
    uint8_t *o = (uint8_t *)out;
    for (int j = 0; j < n; j++) {
        memcpy(o, &h, sizeof h); o += sizeof h;
        for (const StatePart &p : replica_parts(e, idx[j])) { CK(cudaMemcpyAsync(o, p.dev, p.bytes, cudaMemcpyDeviceToHost, e->stream)); o += p.bytes; }
    }
    CK(cudaStreamSynchronize(e->stream));
    e->d2h_bytes += (rb - (int64_t)sizeof h) * n;
    return 0;
}

extern "C" int rb_import_replicas(rb_engine *e, int32_t n, const int32_t *slot, const uint32_t *seed, const void *in, int64_t n_bytes) {
    CK(cudaSetDevice(e->cfg.device));
    if (check_slots(e, "rb_import_replicas", n, slot)) return 1;
    const int64_t rb = rb_replica_bytes(e);
    if (n_bytes != rb * n) { snprintf(g_err, sizeof g_err, "rb_import_replicas: %lld bytes for %d records of %lld", (long long)n_bytes, n, (long long)rb); return 1; }
    const uint8_t *o = (const uint8_t *)in;
    for (int j = 0; j < n; j++) {
        ReplicaHeader h; memcpy(&h, o + rb * j, sizeof h);
        if (check_header(e, "rb_import_replicas", h, j)) return 1;
    }
    if (sync_all_streams(e)) return 1;
    for (int j = 0; j < n; j++) {
        o += sizeof(ReplicaHeader);
        for (const StatePart &p : replica_parts(e, slot[j])) { CK(cudaMemcpyAsync(p.dev, o, p.bytes, cudaMemcpyHostToDevice, e->stream)); o += p.bytes; }
    }
    e->h2d_bytes += (rb - (int64_t)sizeof(ReplicaHeader)) * n;
    return finish_import(e, n, slot, seed);
}

extern "C" int rb_copy_replicas(rb_engine *dst, rb_engine *src, int32_t n, const int32_t *src_idx, const int32_t *dst_slot, const uint32_t *seed) {
    if (dst == src) { snprintf(g_err, sizeof g_err, "rb_copy_replicas: source and destination are the same engine (rb_branch copies within one)"); return 1; }
    if (check_sources(src, "rb_copy_replicas", n, src_idx) || check_slots(dst, "rb_copy_replicas", n, dst_slot)) return 1;
    if (check_header(dst, "rb_copy_replicas", replica_header(src), 0)) return 1;
    CK(cudaSetDevice(src->cfg.device));
    if (flush_for_export(src)) return 1;
    CK(cudaStreamSynchronize(src->stream));
    CK(cudaSetDevice(dst->cfg.device));
    if (sync_all_streams(dst)) return 1;
    const int ds = src->cfg.device, dd = dst->cfg.device;
    for (int j = 0; j < n; j++) {
        const std::vector<StatePart> s = replica_parts(src, src_idx[j]), d = replica_parts(dst, dst_slot[j]);
        for (size_t k = 0; k < s.size(); k++) {
            if (ds == dd) CK(cudaMemcpyAsync(d[k].dev, s[k].dev, s[k].bytes, cudaMemcpyDeviceToDevice, dst->stream));
            else CK(cudaMemcpyPeerAsync(d[k].dev, dd, s[k].dev, ds, s[k].bytes, dst->stream));
        }
    }
    return finish_import(dst, n, dst_slot, seed);
}

// Collective over the engine's communicator.  Every rank first checks its own arguments, then the ranks exchange their
// headers and verdicts (one small all-gather), so that a plan or shape one rank refuses is refused by all of them and
// nobody is left waiting in a send.  Sends and receives of every part then go in one NCCL group.
extern "C" int rb_comm_move_replicas(rb_engine *e, int32_t n_send, const int32_t *send_idx, const int32_t *send_peer,
                                     int32_t n_recv, const int32_t *recv_slot, const int32_t *recv_peer, const uint32_t *recv_seed) {
    const char *fn = "rb_comm_move_replicas";
    CK(cudaSetDevice(e->cfg.device));
    if (!e->comm || e->sharded) { snprintf(g_err, sizeof g_err, "%s: needs the ensemble communicator of rb_comm_init (and no population-sharded mode)", fn); return 1; }
    const int K = e->comm_size, me = e->comm_rank;
    int bad = check_sources(e, fn, n_send, send_idx) || check_slots(e, fn, n_recv, recv_slot);
    for (int i = 0; i < n_send && !bad; i++)
        if (send_peer[i] < 0 || send_peer[i] >= K || send_peer[i] == me) { snprintf(g_err, sizeof g_err, "%s: send_peer[%d] = %d is not another rank", fn, i, send_peer[i]); bad = 1; }
    for (int j = 0; j < n_recv && !bad; j++) {
        if (recv_peer[j] < 0 || recv_peer[j] >= K || recv_peer[j] == me) { snprintf(g_err, sizeof g_err, "%s: recv_peer[%d] = %d is not another rank", fn, j, recv_peer[j]); bad = 1; }
        for (int i = 0; i < n_send && !bad; i++)
            if (send_idx[i] == recv_slot[j]) { snprintf(g_err, sizeof g_err, "%s: replica %d is both sent and written", fn, recv_slot[j]); bad = 1; }
    }
    struct Hello { ReplicaHeader h; int32_t bad, pad[15]; };
    static_assert(sizeof(Hello) == 128, "Hello is one 128-byte record");
    Hello mine; memset(&mine, 0, sizeof mine);
    mine.h = replica_header(e); mine.bad = bad;
    if (sync_all_streams(e)) return 1;
    void *d; bool temp;
    if (comm_scratch(e, sizeof(Hello) * K, &d, &temp)) return 1;
    std::vector<Hello> all(K);
    CK(cudaMemcpyAsync((Hello *)d + me, &mine, sizeof mine, cudaMemcpyHostToDevice, e->stream));
    NK(g_nccl.AllGather((Hello *)d + me, d, sizeof(Hello), ncclChar, e->comm, e->stream));
    CK(cudaMemcpyAsync(all.data(), d, sizeof(Hello) * K, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (temp) cudaFree(d);
    if (bad) return 1;
    for (int k = 0; k < K; k++) {
        if (all[k].bad) { snprintf(g_err, sizeof g_err, "%s: rank %d refused the plan", fn, k); return 1; }
        if (memcmp(&all[k].h, &mine.h, sizeof mine.h) != 0) { snprintf(g_err, sizeof g_err, "%s: rank %d holds an engine of another shape, build or day", fn, k); return 1; }
    }
    if (n_send > 0 && flush_for_export(e)) return 1;
    NK(g_nccl.GroupStart());
    for (int i = 0; i < n_send; i++)
        for (const StatePart &p : replica_parts(e, send_idx[i])) NK(g_nccl.Send(p.dev, p.bytes, ncclChar, send_peer[i], e->comm, e->stream));
    for (int j = 0; j < n_recv; j++)
        for (const StatePart &p : replica_parts(e, recv_slot[j])) NK(g_nccl.Recv(p.dev, p.bytes, ncclChar, recv_peer[j], e->comm, e->stream));
    NK(g_nccl.GroupEnd());
    return finish_import(e, n_recv, recv_slot, recv_seed);
}
