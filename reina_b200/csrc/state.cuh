// reina_b200 / csrc / state.cuh
// Data layout of the engine in HBM (structure of arrays, agents age-sorted), the per-replica counters, the
// population-sharded message slots, and the small device helpers every kernel shares (age lookup, sweep position,
// severity thresholds, person_infect).
#ifndef REINA_B200_STATE_CUH
#define REINA_B200_STATE_CUH

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <dlfcn.h>
#include <nccl.h>      // types only: libnccl is loaded at run time by rb_shard_init, single-GPU use never needs it

#include <algorithm>
#include <vector>

#include "../../include/reina_b200.h"
#include "rng.cuh"

#define MAX_INFECTEES 64   // main.pyx:128
#define MAX_CONTACTS 128   // main.pyx:129

// ---------------------------------------------------------------- packed hot word
#define H_STATE(h) ((h) & 7u)
#define H_SEV(h) (((h) >> 3) & 7u)
#define H_DET (1u << 6)
#define H_QUEUED (1u << 7)
#define H_VAR(h) (((h) >> 8) & 3u)
#define H_FRESH (1u << 10)
#define H_INCL (1u << 11)
#define H_LIST (1u << 12)
#define H_VACC (1u << 13)
#define H_DL(h) (((h) >> 14) & 255u)
#define H_DOI(h) (((h) >> 22) & 31u)
#define H_PEND (1u << 27)    // active-list copies only: a bed / ICU claim is pending, the day boundary decides -- reload the word from `hot`
#define H_DAYS_MASK ((255u << 14) | (31u << 22))     // the two day counters: kept current in the active list, in `hot` only at state changes
#define H_SET_STATE(h, s) (((h) & ~7u) | (uint32_t)(s))
#define H_SET_DL(h, d) (((h) & ~(255u << 14)) | ((uint32_t)(d) << 14))
#define H_SET_DOI(h, d) (((h) & ~(31u << 22)) | ((uint32_t)(d) << 22))

#define KEY_IDLE 0xFFFFFFFFFFFFFFFFull
#define QKEY_SWEEP (1ull << 62)
#define CT_DEAD (1ull << 61)
#define CT_DECIDED (1ull << 60)
#define CT_KEYMASK ((1ull << 60) - 1ull)

enum { EV_HOSP_CLAIM = 0, EV_WARD_RELEASE = 1, EV_TO_ICU = 2, EV_ICU_RELEASE = 3 };

#define MAX_RANKS 16
#define WIDE_MAX_CTAS 64      // CTAs of one replica's wide day boundary
#define SORT_SMEM 2048
#ifndef PRE_THREADS
#define PRE_THREADS 512       // day-boundary CTA: two fit on an SM, so 256 replicas are one wave
#endif
#define NEG_INF (-(1 << 29))

#ifndef GUIDE_BITS
#define GUIDE_BITS 12        // 2^GUIDE_BITS cells per age in the row guide (>= 9: the boundary's low bits must fit the entry); measured 9 / 10 / 11: 721 / 645 / 607 us on the peak day
#endif
struct DevTable {
    int32_t n_rows[RB_MAX_AGES];
    float nr_contacts[RB_MAX_AGES];
    double ncdf[RB_MAX_AGES][2][RB_NCDF];
    double cum_p[RB_MAX_AGES][RB_MAX_ROWS];
    uint32_t cum24[RB_MAX_AGES][RB_MAX_ROWS];         // ceil(cum_p * 2^24): for a 24-bit uniform k / 2^24, (k / 2^24 < cum_p) == (k < cum24)
    int32_t start[RB_MAX_AGES][RB_MAX_ROWS];
    int32_t size[RB_MAX_AGES][RB_MAX_ROWS];
    float mask_p[RB_MAX_AGES][RB_MAX_ROWS];
    uint8_t place[RB_MAX_AGES][RB_MAX_ROWS];
    uint8_t lo_age[RB_MAX_AGES][RB_MAX_ROWS], hi_age[RB_MAX_AGES][RB_MAX_ROWS];
    uint8_t susc_uniform[RB_MAX_AGES][RB_MAX_ROWS];   // susceptibility identical for every age of the row's band
    uint8_t nguide[RB_MAX_AGES][2][256];              // k0 = first k with ncdf[k] > b/256: start of the contact-count search; bit 7: the cell holds a boundary, search on from k0
    // ---- everything above is filled by the host (rb_set_contact_table); the row guide below is derived from cum24 / place
    // on the device (k_build_guide), so it never crosses PCIe
    // O(1) row pick (get_one_contact, main.pyx:1290-1304): the 24-bit uniform's top GUIDE_BITS bits select a cell, and
    // ONE 4-byte entry answers for the whole cell: row0 = row of the cell's first value (7 b), its place (3 b << 7),
    // delta (4 b << 10): 0 = every value of the cell maps to row0; 1..14 = one boundary inside the cell, values whose low
    // bits are >= blow (<< 17, the boundary's low 24 - GUIDE_BITS bits) map to row0 + delta, whose place is place1
    // (3 b << 14; the rows in between have probability zero); 15 = several boundaries, the search walks on from row0 (rare).
    uint32_t guide[RB_MAX_AGES][1 << GUIDE_BITS];
};

struct Attempt { uint32_t cand, parent; unsigned long long key; };

// Everything about one agent that only infections, tracing and capacity outcomes touch, in ONE 32-byte sector:
// an infection then costs one random DRAM sector for the target and one for the infector instead of seven.
struct __align__(32) AgentRec {
    unsigned long long winner;       // atomicMin conflict slot, all-ones when idle
    int32_t infector, first_child, next_sib;   // infection tree (replaces the malloc'd infectees[64], main.pyx:227-233)
    uint32_t inf_key;                // (day << 8) | slot of this agent's infection: orders siblings; day << 8 for a root
    uint32_t cold;                   // other_people_infected 16b | ward_days 8b | icu_days 8b
    int16_t vacc_day, pad;
};

// Per-replica counters.  The scalars the grid kernels hammer with atomics each sit on their own 128-byte line, away
// from the fields every thread only READS (seed, day, sweep start ...): with one big replica all SMs share this one
// struct, and a read that lands on a line with a queue of atomics in front of it waits for all of them.
struct RepCtr {
    int32_t counts[RB_N_ATTRS][RB_MAX_AGES];
    // ---- written by the day-boundary CTA only, read by everybody
    alignas(128) int32_t beds;
    int32_t icu, avail_beds, avail_icu;
    int32_t problem, epoch, testing_mode, day;
    float p_detected_anyway, p_successful_tracing;
    uint32_t seed, start;
    uint32_t fkey[4];
    uint32_t n_queue, qsel;
    uint32_t n_queue_prev;                        // size of the queue drained yesterday (normalises tracing keys for sorting)
    uint32_t any_vacc;                            // set once the first vaccination programme starts
    uint32_t lsel;                                // active lists in force today: the sweep reads lists lsel and writes lists lsel ^ 1
    uint32_t ct_ever;                             // contact tracing has been on at some point: detections may reach agents behind the list's back
    uint32_t n_q_base;                            // entries contact tracing put into tomorrow's queue before the sweep
    uint32_t drained;                             // tomorrow's queue was already drained by k_resolve (detections parked in drain_det)
    int32_t ct_cases;
    int32_t vacc_cursor[RB_MAX_VACC];
    // ---- atomics of the grid kernels, one line per group
    alignas(128) uint32_t n_items;
    alignas(128) uint32_t n_succ;
    alignas(128) int32_t exposed_per_day;
    int32_t total_infectors, total_infections;
    alignas(128) uint32_t n_events;
    uint32_t n_newq;
    uint32_t n_upd;                               // population-sharded mode: packed-word updates logged by today's sweep
    alignas(128) int32_t daily_contacts[RB_N_PLACES];
    int32_t by_variant[RB_MAX_VARIANTS];
    alignas(128) int32_t drain_det[RB_MAX_AGES];  // detections of an early queue drain, per age, booked at the next day boundary
    alignas(128) uint32_t n_l0;
    uint32_t n_l1, n_edges;
    // wide day boundary (boundary.cuh, Team): grid barrier word on its own line, today's verdict, per-CTA scan totals
    alignas(128) unsigned int run_bar;            // k_run: barrier word of the replica's whole team
    unsigned int run_exit;                        // k_run: CTAs that have left the final barrier
    alignas(128) unsigned int wide_bar;
    alignas(128) uint32_t wide_day;
    int32_t wide_mp[WIDE_MAX_CTAS][4];
    long long dbg_t[16];                          // measurement aid: cycles spent per phase of the day-boundary kernel
    long long dbg_last;
};

struct Eng {
    int32_t dbg;                                   // measurement aid: 9 = the day-boundary kernels record cycles per phase (RepCtr::dbg_t)
    int32_t N, Npad, n_ages, n_groups, n_variants, R, max_days, row_len, n_import_classes, fhalf;
    uint32_t cap_items, cap_succ, cap_events, cap_queue;
    uint32_t *hot;
    uint32_t *perm;                                // [R][Npad] slot in the replica's sweep order, valid once the agent has been infected
    AgentRec *rec;
    uint32_t *sus;                                 // [R][sus_words] 1 bit per agent: still SUSCEPTIBLE (L2-resident gather target)
    int32_t sus_words;
    uint32_t *det;                                 // [R][sus_words] 1 bit per agent: detected by a test-queue drain (the sweep consults it once contact tracing has been on)
    // Active lists: (agent, copy of its packed word with CURRENT day counters).  Every replica has n_seg segments, agent
    // a always lives in segment a % n_seg (so a segment can never hold more than seg_cap = ceil(N / n_seg) entries), and
    // one warp of the sweep owns a whole segment while it runs.  A segment is filled from BOTH ends: the owning warp
    // writes the survivors of its pass to the front, behind a counter it keeps in a register (no atomics on the sweep's
    // hot loop); everybody else -- the sweep's own slow stage, k_resolve and the imports with their new infections --
    // appends at the back with an atomic on the segment's second counter.  The two ends cannot meet.
    uint2 *alist;                                  // [R][2][n_seg][seg_cap]
    uint2 *seg_n;                                  // [R][2][n_seg] entries at the front (.x) / at the back (.y) of each segment
    uint32_t n_seg, seg_cap;
    uint2 *items;
    Attempt *succ;
    unsigned long long *ev_key; int32_t *ev_agent;
    unsigned long long *q_key; int32_t *q_agent;   // [R][2][cap_queue]
    RepCtr *ctr;
    int32_t *stats;                                // [R][max_days+1][row_len]
    const rb_day_params *sched;
    DevTable *const *tables;
    const rb_variant *variants;
    const int32_t *age_start;                      // [n_ages+1]
    const uint8_t *age_blk;                        // age of agent (b << 10): coarse index into age_start
    const int32_t *group_of_age;
    const int32_t *import_lo, *import_hi; const float *import_cum;
    // population-sharded mode (rb_shard_init): every rank holds the whole state, sweeps and exposes only the agents
    // it owns, and publishes what the others must know in its slot of the exchange buffer (one all-gather per day)
    int32_t rank, nranks;
    int32_t wide_min;                              // a day with this many capacity events / queued tests gets the wide boundary
    int32_t r0;                                    // first replica of this launch (replica groups on concurrent streams, engine.cu)
    // exchange through NCCL: xbuf = [nranks] message slots, slot `rank` written locally, the rest filled by the daily
    // all-gather.  Exchange through peer memory (xp2p): every rank owns [256-byte flag line][slot of even days][slot of
    // odd days], xpeer[k] is rank k's buffer mapped through CUDA IPC (xpeer[rank] = xbuf = the own one), and k_merge
    // pulls exactly the bytes each message holds over NVLink once the owner's flag says the day is complete.
    uint8_t *xbuf; size_t xslot;
    uint8_t *xpeer[MAX_RANKS];
    int32_t xp2p; const uint32_t *xepoch;          // *xepoch (a device word, so that captured graphs stay valid): bumped by every reset / state load, keeps the flags monotonic
    uint32_t xcap_q, xcap_ev, xcap_upd, xcap_succ;
};

// Ownership: stripes of 4096 agents (one warp step of the sweep) dealt round-robin, so every rank holds ~1/nranks of every age.
#define XFLAG_BYTES 256
#define SH_SHIFT 12
__device__ __forceinline__ uint32_t xflag_value(const Eng &G, int day) { return *G.xepoch * 65536u + (uint32_t)day + 1u; }
__device__ __forceinline__ bool owns(const Eng &G, uint32_t a) { return G.nranks == 1 || (int)((a >> SH_SHIFT) % (uint32_t)G.nranks) == G.rank; }

// One rank's message: a RepCtr used as the header (count deltas of the sweep, list lengths) followed by the lists.
struct XSlot {
    RepCtr *hdr;
    unsigned long long *q_key; int32_t *q_agent;     // test-queue entries created by the sweep
    unsigned long long *ev_key; int32_t *ev_agent;   // capacity events
    uint2 *upd;                                      // (agent, packed word) after a state change
    struct Attempt *succ;                            // successful transmissions
};
__host__ __device__ inline size_t xalign(size_t x) { return (x + 255) & ~(size_t)255; }
__host__ __device__ inline size_t xslot_bytes(uint32_t cq, uint32_t ce, uint32_t cu, uint32_t cs) {
    return xalign(sizeof(RepCtr)) + xalign(8ull * cq) + xalign(4ull * cq) + xalign(8ull * ce) + xalign(4ull * ce) + xalign(8ull * cu) + xalign(16ull * cs);
}
__device__ __forceinline__ XSlot xslot_of(const Eng &G, int rk, int day) {
    uint8_t *p = G.xp2p ? G.xpeer[rk] + XFLAG_BYTES + (size_t)(day & 1) * G.xslot : G.xbuf + (size_t)rk * G.xslot;
    XSlot s;
    s.hdr = (RepCtr *)p; p += xalign(sizeof(RepCtr));
    s.q_key = (unsigned long long *)p; p += xalign(8ull * G.xcap_q);
    s.q_agent = (int32_t *)p; p += xalign(4ull * G.xcap_q);
    s.ev_key = (unsigned long long *)p; p += xalign(8ull * G.xcap_ev);
    s.ev_agent = (int32_t *)p; p += xalign(4ull * G.xcap_ev);
    s.upd = (uint2 *)p; p += xalign(8ull * G.xcap_upd);
    s.succ = (struct Attempt *)p;
    return s;
}

// ---------------------------------------------------------------- small device helpers
__device__ __forceinline__ int age_of(const Eng &G, int32_t a) {
    // agents are age-sorted: start from the age of the 1024-agent block and walk up (0-1 steps at HUS sizes)
    int age = __ldg(&G.age_blk[a >> 10]);
    while (a >= __ldg(&G.age_start[age + 1])) age++;
    return age;
}
__device__ __forceinline__ int age_in_band(const Eng &G, int32_t a, int lo, int hi) {   // age of agent a, known to lie in [lo, hi]
    hi += 1;
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (__ldg(&G.age_start[mid]) <= a) lo = mid; else hi = mid; }
    return lo;
}
// Position of agent a in today's sweep (main.pyx:1436, 1988): its slot in the replica's fixed random order, rotated by
// today's start.  The slot -- a keyed Feistel permutation, ~45 instructions -- does not depend on the day, so it is
// computed once, when the agent is infected (device_infect), and kept in `perm`: only infected agents ever need a sweep
// position (capacity events, test-queue entries, transmissions).
__device__ __forceinline__ uint32_t sweep_slot(const Eng &G, const RepCtr *c, uint32_t a) {
    return feistel(a, (uint32_t)G.N, G.fhalf, c->fkey[0], c->fkey[1], c->fkey[2], c->fkey[3]);
}
__device__ __forceinline__ uint32_t sweep_pos(const Eng &G, int r, const RepCtr *c, uint32_t a) {
    const uint32_t s = G.perm[(size_t)r * G.Npad + a];
    return s >= c->start ? s - c->start : s + (uint32_t)G.N - c->start;
}
// A test-queue drain detected agent a (person_detect, main.pyx:294-298).  The sweep keeps its own copies of the active
// agents' words; detections it cannot foresee (contact tracing) reach it through this bitmap.
__device__ __forceinline__ void mark_detected(const Eng &G, int r, int32_t a) {
    atomicOr(&G.det[(size_t)r * G.sus_words + (a >> 5)], 1u << (a & 31));
}
__device__ __forceinline__ void count_add(RepCtr *c, int attr, int age, int d) { atomicAdd(&c->counts[attr][age], d); }
__device__ __forceinline__ void set_problem(RepCtr *c, int p) { atomicCAS(&c->problem, 0, p); }

// Disease.get_symptom_severity, main.pyx:1042-1091 (every FATAL case dies outside hospital, SURVEY 8a note 2)
__device__ __forceinline__ int symptom_severity(const rb_variant *v, int age, float val, bool vacc_eff) {
    float vmod = 1.0f;
    if (vacc_eff) vmod = vmod * 0.1f;
    float syc = v->tab[RB_T_SYMPTOMATIC][age];
    if (val >= syc) return RB_ASYMPTOMATIC;
    syc = syc * vmod;
    float dohc = v->tab[RB_T_DEATH_OUTSIDE_HOSPITAL][age];
    if (dohc != 0.0f) {
        if (val < dohc * syc) return RB_FATAL;
        val = (val - dohc) / (1.0f - dohc);
    }
    float sc = v->tab[RB_T_SEVERE][age], cc = v->tab[RB_T_CRITICAL][age], fc = v->tab[RB_T_FATAL][age];
    if (val < ((fc * cc) * sc) * syc) return RB_FATAL;
    if (val < (cc * sc) * syc) return RB_CRITICAL;
    if (val < sc * syc) return RB_SEVERE;
    return RB_MILD;
}

// Segment s of list `which` of replica r, and its two entry counters.
__device__ __forceinline__ uint2 *seg_ptr(const Eng &G, int r, uint32_t which, uint32_t s) {
    return G.alist + (((size_t)r * 2 + which) * G.n_seg + s) * G.seg_cap;
}
__device__ __forceinline__ uint2 *seg_count(const Eng &G, int r, uint32_t which, uint32_t s) {
    return G.seg_n + ((size_t)r * 2 + which) * G.n_seg + s;
}
// One more entry at the back of agent a's segment (new infections, the sweep's slow stage, list rebuilds).
__device__ __forceinline__ void list_add(const Eng &G, int r, RepCtr *c, uint32_t which, uint32_t a, uint32_t w) {
    const uint32_t s = a % G.n_seg;
    const uint32_t k = atomicAdd(&seg_count(G, r, which, s)->y, 1u);
    if (k < G.seg_cap) seg_ptr(G, r, which, s)[G.seg_cap - 1u - k] = make_uint2(a, w); else set_problem(c, RB_OTHER_FAILURE);
}

// person_infect, main.pyx:209-235 + Population.infect :1576-1582.  `src_h` = packed word of the infector
// (ignored when src < 0).  Severity and incubation use wild-type parameters (variant_idx is still 0 there).
// `list`: the active list the new entry goes to (0 / 1), or -1 for none (the caller rebuilds the lists afterwards).
__device__ void device_infect(const Eng &G, int r, RepCtr *c, int32_t t, int32_t src, uint32_t src_h, int variant,
                              int slot, bool fresh, int list, bool has_list) {
    const size_t base = (size_t)r * G.Npad;
    const int day = c->day;
    // the two atomics whose results are needed go first; the draws below hide their round trip
    uint32_t old = 0; int32_t prev_child = -1;
    if (src >= 0) {
        old = atomicAdd(&G.rec[base + src].cold, 1u);
        prev_child = atomicExch(&G.rec[base + src].first_child, t);
    }
    const int vd = c->any_vacc ? (int)G.rec[base + t].vacc_day : -1;     // nobody is vaccinated in most configurations
    const int age = age_of(G, t);
    const rb_variant *v0 = &G.variants[0];
    const bool vacc_eff = vd >= 0 && (day - vd) > 14;
    int sev = 0, dl = 0;
    if (owns(G, (uint32_t)t)) {     // severity and day counters are only ever read by the owner's sweep (sharded mode)
        u32x4 x = philox(c->seed, (uint32_t)t, (uint32_t)day, PU_SEVERITY, 0);
        sev = symptom_severity(v0, age, u01f(x.x), vacc_eff);
        dl = clamp255(round_to_int(gamma_f(c->seed, (uint32_t)t, (uint32_t)day, PU_INCUB, v0->incubation_kappa, v0->incubation_theta)));
    }
    if (src >= 0) {
        variant = (int)H_VAR(src_h);
        G.rec[base + t].infector = src;
        if ((src_h & H_LIST) && (old & 0xffffu) >= MAX_INFECTEES) set_problem(c, RB_TOO_MANY_INFECTEES);
        G.rec[base + t].inf_key = ((uint32_t)day << 8) | (uint32_t)slot;
        G.rec[base + t].next_sib = prev_child;
    } else {
        G.rec[base + t].inf_key = (uint32_t)day << 8;   // roots (imports, initial state) keep their infection day too: k_transmission
    }
    // a SUSCEPTIBLE agent's word carries nothing but the vaccinated flag, which vacc_day implies
    uint32_t nh = (vd >= 0 ? H_VACC : 0u) | RB_INCUBATION | ((uint32_t)sev << 3) | ((uint32_t)variant << 8) | ((uint32_t)dl << 14);
    if (fresh) nh |= H_FRESH;
    if (has_list) nh |= H_LIST;      // person_infect, main.pyx:227-233: an infectee list only under contact tracing
    G.hot[base + t] = nh;
    G.perm[base + t] = sweep_slot(G, c, (uint32_t)t);
    atomicAnd(&G.sus[(size_t)r * G.sus_words + (t >> 5)], ~(1u << (t & 31)));
    if (list >= 0 && owns(G, (uint32_t)t)) list_add(G, r, c, (uint32_t)list, (uint32_t)t, nh);      // from now on the sweep visits this agent
    count_add(c, RB_A_SUSCEPTIBLE, age, -1);
    count_add(c, RB_A_INFECTED, age, 1);
    count_add(c, RB_A_ALL_INFECTED, age, 1);
    count_add(c, RB_A_NEW_INFECTIONS, age, 1);
    {   // infected_by_variant: one atomic per group of converged lanes with the same variant
        const unsigned act = __activemask();
        const unsigned grp = __match_any_sync(act, variant);
        if ((int)(threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(&c->by_variant[variant], __popc(grp));
    }
}

#endif
