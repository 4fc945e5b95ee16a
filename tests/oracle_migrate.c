/*
 * oracle_migrate.c -- CPU reference of moving replicas between engines (reina_b200.h rb_replica_bytes /
 * rb_export_replicas / rb_import_replicas / rb_copy_replicas).  TEST INFRASTRUCTURE ONLY: tests/test_migrate.py compiles
 * it, with the probes of tests/test_transmission_settings.py, into a library of its own in a temporary directory.
 *
 * A record is this file's own serialisation of one oracle Replica, not the CUDA engine's byte layout: a header, the
 * Replica's scalars, every Agent record (the infectee list pointer replaced by a flag), a fixed table of MAX_INFECTEES
 * entries per agent for the infectee lists, the sweep order and its inverse, the test queue (at most n_agents entries),
 * the replica's stats rows and, last, its row of the seed history (oracle_branch.c's side table).  Records are fixed in
 * size, so n records are n * ro_replica_bytes bytes.  Import writes a record into a slot exactly as ro_branch writes a
 * copy, then gives the slot its seed from today on.
 */
#include "oracle_branch.c"

typedef struct { int32_t magic, n_agents, n_ages, row_len, max_days, day, agent_bytes, replica_bytes; } MigHeader;
#define MIG_MAGIC 0x4749524d   /* "MRIG" */

static MigHeader mig_header(rb_engine *e) {
    MigHeader h = {MIG_MAGIC, e->cfg.n_agents, e->cfg.n_ages, e->row_len, e->cfg.max_days, e->day, (int32_t)sizeof(Agent), (int32_t)sizeof(Replica)};
    return h;
}

int64_t ro_replica_bytes(rb_engine *e) {
    const int64_t N = e->cfg.n_agents, M = e->cfg.max_days + 1;
    return (int64_t)sizeof(MigHeader) + (int64_t)sizeof(Replica) + N * (int64_t)sizeof(Agent) + N * MAX_INFECTEES * 4
           + 2 * N * 4 + N * 4 + M * e->row_len * 4 + M * 4;
}

static int check_idx(rb_engine *e, const char *fn, int32_t n, const int32_t *idx, int slots) {
    const int R = e->cfg.n_replicas;
    if (n < 0 || (slots && n > R)) { snprintf(g_err, sizeof g_err, "%s: %d replicas", fn, n); return 1; }
    for (int j = 0; j < n; j++) {
        if (idx[j] < 0 || idx[j] >= R) { snprintf(g_err, sizeof g_err, "%s: index %d is not a replica", fn, idx[j]); return 1; }
        if (slots) for (int i = 0; i < j; i++) if (idx[i] == idx[j]) { snprintf(g_err, sizeof g_err, "%s: slot %d is written twice", fn, idx[j]); return 1; }
    }
    return 0;
}

static void put(uint8_t **o, const void *p, size_t n) { memcpy(*o, p, n); *o += n; }
static void get(const uint8_t **o, void *p, size_t n) { memcpy(p, *o, n); *o += n; }

int ro_export_replicas(rb_engine *e, int32_t n, const int32_t *idx, void *out, int64_t capacity) {
    if (check_idx(e, "ro_export_replicas", n, idx, 0)) return 1;
    if (capacity < ro_replica_bytes(e) * n) { snprintf(g_err, sizeof g_err, "ro_export_replicas: buffer too small"); return 1; }
    const int32_t N = e->cfg.n_agents, M = e->cfg.max_days + 1;
    uint32_t *hist = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)e->cfg.n_replicas * M);
    read_hist(e, hist);
    const MigHeader h = mig_header(e);
    uint8_t *o = (uint8_t *)out;
    int32_t *lists = (int32_t *)calloc((size_t)N * MAX_INFECTEES, sizeof(int32_t)), *q = (int32_t *)calloc((size_t)N, sizeof(int32_t));
    for (int j = 0; j < n; j++) {
        const Replica *r = &e->rep[idx[j]];
        if (r->n_queue > N) { snprintf(g_err, sizeof g_err, "ro_export_replicas: queue of %d entries", r->n_queue); free(hist); free(lists); free(q); return 1; }
        put(&o, &h, sizeof h);
        put(&o, r, sizeof *r);
        for (int32_t a = 0; a < N; a++) {
            Agent g = r->agents[a];
            g.infectees = (int32_t *)(uintptr_t)(g.infectees != NULL);
            put(&o, &g, sizeof g);
            if (r->agents[a].infectees) memcpy(lists + (size_t)a * MAX_INFECTEES, r->agents[a].infectees, sizeof(int32_t) * MAX_INFECTEES);
            else memset(lists + (size_t)a * MAX_INFECTEES, 0, sizeof(int32_t) * MAX_INFECTEES);
        }
        put(&o, lists, sizeof(int32_t) * (size_t)N * MAX_INFECTEES);
        put(&o, r->order, sizeof(int32_t) * (size_t)N);
        put(&o, r->perm, sizeof(int32_t) * (size_t)N);
        memset(q, 0, sizeof(int32_t) * (size_t)N);
        if (r->n_queue) memcpy(q, r->queue, sizeof(int32_t) * (size_t)r->n_queue);
        put(&o, q, sizeof(int32_t) * (size_t)N);
        put(&o, e->stats + (size_t)idx[j] * M * e->row_len, sizeof(int32_t) * (size_t)M * e->row_len);
        put(&o, hist + (size_t)idx[j] * M, sizeof(uint32_t) * (size_t)M);
    }
    free(hist); free(lists); free(q);
    return 0;
}

static SeedHist *own_hist(rb_engine *e) {
    SeedHist *h = find_hist(e);
    if (!h) {
        h = (SeedHist *)calloc(1, sizeof *h);
        h->e = e; h->seeds = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)e->cfg.n_replicas * (e->cfg.max_days + 1));
        read_hist(e, h->seeds);
        h->next = g_hist; g_hist = h;
    }
    return h;
}

int ro_import_replicas(rb_engine *e, int32_t n, const int32_t *slot, const uint32_t *seed, const void *in, int64_t n_bytes) {
    if (check_idx(e, "ro_import_replicas", n, slot, 1)) return 1;
    const int64_t rb = ro_replica_bytes(e);
    if (n_bytes != rb * n) { snprintf(g_err, sizeof g_err, "ro_import_replicas: %lld bytes for %d records", (long long)n_bytes, n); return 1; }
    const MigHeader w = mig_header(e);
    for (int j = 0; j < n; j++) {
        MigHeader h; memcpy(&h, (const uint8_t *)in + rb * j, sizeof h);
        if (h.magic == w.magic && h.day != w.day) { snprintf(g_err, sizeof g_err, "ro_import_replicas: record %d is of day %d, the engine is at day %d", j, h.day, w.day); return 1; }
        if (memcmp(&h, &w, sizeof h) != 0) { snprintf(g_err, sizeof g_err, "ro_import_replicas: record %d was made by an engine of another shape", j); return 1; }
    }
    const int32_t N = e->cfg.n_agents, M = e->cfg.max_days + 1;
    SeedHist *sh = own_hist(e);
    int32_t *lists = (int32_t *)malloc(sizeof(int32_t) * (size_t)N * MAX_INFECTEES);
    for (int j = 0; j < n; j++) {
        const uint8_t *o = (const uint8_t *)in + rb * j + sizeof(MigHeader);
        Replica *d = &e->rep[slot[j]];
        for (int32_t a = 0; a < N; a++) free(d->agents[a].infectees);
        Agent *agents = d->agents; int32_t *order = d->order, *perm = d->perm, *queue = d->queue, *newq = d->newq;
        const int32_t cap_newq = d->cap_newq;
        get(&o, d, sizeof *d);
        d->agents = agents; d->order = order; d->perm = perm; d->newq = newq; d->cap_newq = cap_newq; d->n_newq = 0;
        get(&o, d->agents, sizeof(Agent) * (size_t)N);
        get(&o, lists, sizeof(int32_t) * (size_t)N * MAX_INFECTEES);
        for (int32_t a = 0; a < N; a++) {
            Agent *g = &d->agents[a];
            if (g->infectees) {
                g->infectees = (int32_t *)malloc(sizeof(int32_t) * MAX_INFECTEES);
                memcpy(g->infectees, lists + (size_t)a * MAX_INFECTEES, sizeof(int32_t) * MAX_INFECTEES);
            }
        }
        get(&o, d->order, sizeof(int32_t) * (size_t)N);
        get(&o, d->perm, sizeof(int32_t) * (size_t)N);
        d->queue = (int32_t *)realloc(queue, sizeof(int32_t) * (size_t)(d->cap_queue > N ? d->cap_queue : (N ? N : 1)));
        d->cap_queue = d->cap_queue > N ? d->cap_queue : (N ? N : 1);
        get(&o, d->queue, sizeof(int32_t) * (size_t)N);
        get(&o, e->stats + (size_t)slot[j] * M * e->row_len, sizeof(int32_t) * (size_t)M * e->row_len);
        get(&o, sh->seeds + (size_t)slot[j] * M, sizeof(uint32_t) * (size_t)M);
        d->seed = seed[j];
        for (int dd = e->day; dd < M; dd++) sh->seeds[(size_t)slot[j] * M + dd] = seed[j];
    }
    free(lists);
    return 0;
}

int ro_copy_replicas(rb_engine *dst, rb_engine *src, int32_t n, const int32_t *src_idx, const int32_t *dst_slot, const uint32_t *seed) {
    if (dst == src) { snprintf(g_err, sizeof g_err, "ro_copy_replicas: source and destination are the same engine"); return 1; }
    if (check_idx(src, "ro_copy_replicas", n, src_idx, 0) || check_idx(dst, "ro_copy_replicas", n, dst_slot, 1)) return 1;
    const int64_t rb = ro_replica_bytes(src);
    uint8_t *buf = (uint8_t *)malloc((size_t)(rb * (n ? n : 1)));
    int rc = ro_export_replicas(src, n, src_idx, buf, rb * n);
    if (!rc) rc = ro_import_replicas(dst, n, dst_slot, seed, buf, rb * n);
    free(buf);
    return rc;
}
