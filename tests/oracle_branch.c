/*
 * oracle_branch.c -- CPU reference of branching replicas (reina_b200.h rb_branch / rb_read_seeds).  TEST INFRASTRUCTURE
 * ONLY: tests/test_branch.py compiles it, with the probes of tests/test_transmission_settings.py, into a library of its
 * own in a temporary directory.
 *
 * ro_branch deep-copies Replica src[j] into slot j -- every Agent record (with its own copy of the infectee list), the
 * sweep order and its inverse, both test queues, the counts and scalars -- and the replica's stats rows, then gives the
 * slot its new seed.  The oracle keeps no seed history, so this file keeps one in a side table per engine, created by the
 * first branch and dropped by reset and destroy (an engine without an entry has drawn with its current seeds on every
 * day).  The transmission settings after a branch need no history here: the instrumented oracle records the place of
 * every infection where it happens.
 */
#define ro_reset ro_reset_unbranched
#define ro_destroy ro_destroy_unbranched
#include "oracle_settings.c"
#undef ro_reset
#undef ro_destroy

typedef struct SeedHist { rb_engine *e; uint32_t *seeds; struct SeedHist *next; } SeedHist;   /* seeds[R][max_days + 1] */
static SeedHist *g_hist;

static SeedHist *find_hist(rb_engine *e) {
    for (SeedHist *h = g_hist; h; h = h->next) if (h->e == e) return h;
    return NULL;
}
static void forget_hist(rb_engine *e) {
    for (SeedHist **p = &g_hist; *p; p = &(*p)->next)
        if ((*p)->e == e) { SeedHist *h = *p; *p = h->next; free(h->seeds); free(h); return; }
}
static void read_hist(rb_engine *e, uint32_t *out) {
    const int32_t M = e->cfg.max_days + 1;
    const SeedHist *h = find_hist(e);
    for (int r = 0; r < e->cfg.n_replicas; r++)
        for (int d = 0; d < M; d++) out[(size_t)r * M + d] = h && d < e->day ? h->seeds[(size_t)r * M + d] : e->rep[r].seed;
}

int ro_reset(rb_engine *e, uint32_t seed) { forget_hist(e); return ro_reset_unbranched(e, seed); }
void ro_destroy(rb_engine *e) { forget_hist(e); ro_destroy_unbranched(e); }

int ro_read_seeds(rb_engine *e, uint32_t *out) { read_hist(e, out); return 0; }

static void copy_replica(rb_engine *e, Replica *d, const Replica *s) {
    const int32_t N = e->cfg.n_agents;
    for (int32_t a = 0; a < N; a++) free(d->agents[a].infectees);
    Agent *agents = d->agents; int32_t *order = d->order, *perm = d->perm, *queue = d->queue, *newq = d->newq;
    const int32_t cap_newq = d->cap_newq;
    *d = *s;
    d->agents = agents; d->order = order; d->perm = perm; d->newq = newq; d->cap_newq = cap_newq; d->n_newq = 0;
    memcpy(d->agents, s->agents, sizeof(Agent) * (size_t)N);
    for (int32_t a = 0; a < N; a++)
        if (s->agents[a].infectees) {
            d->agents[a].infectees = (int32_t *)malloc(sizeof(int32_t) * MAX_INFECTEES);
            memcpy(d->agents[a].infectees, s->agents[a].infectees, sizeof(int32_t) * MAX_INFECTEES);
        }
    memcpy(d->order, s->order, sizeof(int32_t) * (size_t)N);
    memcpy(d->perm, s->perm, sizeof(int32_t) * (size_t)N);
    d->queue = (int32_t *)realloc(queue, sizeof(int32_t) * (size_t)(s->cap_queue ? s->cap_queue : 1));
    if (s->n_queue) memcpy(d->queue, s->queue, sizeof(int32_t) * (size_t)s->n_queue);
}

int ro_branch(rb_engine *e, const int32_t *src, const uint32_t *seed) {
    const int R = e->cfg.n_replicas;
    const int32_t M = e->cfg.max_days + 1;
    for (int j = 0; j < R; j++) {
        if (src[j] < 0 || src[j] >= R) { snprintf(g_err, sizeof g_err, "ro_branch: src[%d] = %d is not a replica", j, src[j]); return 1; }
        if (src[src[j]] != src[j]) { snprintf(g_err, sizeof g_err, "ro_branch: src[%d] = %d is itself copied", j, src[j]); return 1; }
    }
    SeedHist *h = find_hist(e);
    if (!h) {
        h = (SeedHist *)calloc(1, sizeof *h);
        h->e = e; h->seeds = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)R * M);
        read_hist(e, h->seeds);
        h->next = g_hist; g_hist = h;
    }
    for (int j = 0; j < R; j++) {
        const int s = src[j];
        if (s != j) {
            copy_replica(e, &e->rep[j], &e->rep[s]);
            memcpy(e->stats + (size_t)j * M * e->row_len, e->stats + (size_t)s * M * e->row_len, sizeof(int32_t) * (size_t)M * e->row_len);
            memcpy(h->seeds + (size_t)j * M, h->seeds + (size_t)s * M, sizeof(uint32_t) * (size_t)M);
        }
        e->rep[j].seed = seed[j];
        for (int d = e->day; d < M; d++) h->seeds[(size_t)j * M + d] = seed[j];
    }
    return 0;
}
