// reina_b200 / csrc / transmission.cuh
// Transmission statistics of the current state, read from the infection tree the engine keeps anyway (AgentRec: infector,
// inf_key = infection day << 8 | slot, other_people_infected in the low 16 bits of `cold`).  One pass per replica over
// the agents that have left SUSCEPTIBLE; nothing on the per-day path reads or writes anything here.
//
// Row of one replica (int32, rb_transmission_len entries), M = max_days + 1, B = RB_TX_BINS:
//   cohort_infected[M]   infected agents by infection day d
//   cohort_offspring[M]  sum of their other_people_infected
//   cohort_open[M]       of those, still INCUBATION / ILLNESS (the states that expose others): offspring not final yet
//   offspring_hist[B]    closed cases by min(other_people_infected, 64)
//   gi_hist[B]           agents with an infector, by min(d - d(infector), 64): the generation interval in days
//   group_closed[n_groups], group_offspring[n_groups]              closed cases and their offspring by age group
//   variant_closed[RB_MAX_VARIANTS], variant_offspring[...]        the same by variant
#ifndef REINA_B200_TRANSMISSION_CUH
#define REINA_B200_TRANSMISSION_CUH

#include "state.cuh"

#define TX_THREADS 256

struct TxLayout {
    int M, n_groups;
    int infected, offspring, open, ohist, gi, gclosed, goff, vclosed, voff, len;
};
__host__ __device__ inline TxLayout tx_layout(int max_days, int n_groups) {
    TxLayout L;
    L.M = max_days + 1; L.n_groups = n_groups;
    L.infected = 0; L.offspring = L.M; L.open = 2 * L.M;
    L.ohist = 3 * L.M; L.gi = L.ohist + RB_TX_BINS;
    L.gclosed = L.gi + RB_TX_BINS; L.goff = L.gclosed + n_groups;
    L.vclosed = L.goff + n_groups; L.voff = L.vclosed + RB_MAX_VARIANTS;
    L.len = L.voff + RB_MAX_VARIANTS;
    return L;
}

// blockIdx.y = replica, grid-stride over the agents.  A warp covers 32 consecutive agents = one word of the
// susceptibility bitmap, so the never-infected majority costs 4 bytes per 32 agents; an infected agent costs its packed
// word, its 32-byte record and, with an infector, one gathered record of the infector.  The CTA counts in shared memory
// and adds its counts to out[replica] with integer atomics: the result does not depend on the launch geometry.
__global__ void __launch_bounds__(TX_THREADS) k_transmission(Eng G, TxLayout L, int32_t *out) {
    extern __shared__ int32_t s_tx[];
    const int r = blockIdx.y;
    const size_t base = (size_t)r * G.Npad;
    const uint32_t *sus = G.sus + (size_t)r * G.sus_words;
    for (int i = threadIdx.x; i < L.len; i += blockDim.x) s_tx[i] = 0;
    __syncthreads();
    const int stride = gridDim.x * blockDim.x;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < G.N; a += stride) {
        if ((__ldg(&sus[a >> 5]) >> (a & 31)) & 1u) continue;
        const uint32_t h = G.hot[base + a];
        const uint32_t st = H_STATE(h);
        if (st == RB_SUSCEPTIBLE) continue;
        const AgentRec &rec = G.rec[base + a];
        const int32_t inf = rec.infector;
        const int d = (int)(rec.inf_key >> 8);
        const int o = (int)(rec.cold & 0xffffu);
        if (d < L.M) {
            atomicAdd(&s_tx[L.infected + d], 1);
            atomicAdd(&s_tx[L.offspring + d], o);
        }
        if (inf >= 0) {
            const int gi = d - (int)(G.rec[base + inf].inf_key >> 8);
            atomicAdd(&s_tx[L.gi + min(max(gi, 0), RB_TX_BINS - 1)], 1);
        }
        if (st == RB_INCUBATION || st == RB_ILLNESS) {
            if (d < L.M) atomicAdd(&s_tx[L.open + d], 1);
        } else {
            atomicAdd(&s_tx[L.ohist + min(o, RB_TX_BINS - 1)], 1);
            const int g = __ldg(&G.group_of_age[age_of(G, a)]);
            atomicAdd(&s_tx[L.gclosed + g], 1);
            atomicAdd(&s_tx[L.goff + g], o);
            const int v = (int)H_VAR(h);
            atomicAdd(&s_tx[L.vclosed + v], 1);
            atomicAdd(&s_tx[L.voff + v], o);
        }
    }
    __syncthreads();
    int32_t *row = out + (size_t)r * L.len;
    for (int i = threadIdx.x; i < L.len; i += blockDim.x)
        if (s_tx[i]) atomicAdd(&row[i], s_tx[i]);
}

// Infection day of every agent of one replica, -1 for the never infected (rb_read_infection_days).
__global__ void k_infection_days(Eng G, int r, int32_t *out) {
    const size_t base = (size_t)r * G.Npad;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < G.N; a += gridDim.x * blockDim.x)
        out[a] = H_STATE(G.hot[base + a]) == RB_SUSCEPTIBLE ? -1 : (int32_t)(G.rec[base + a].inf_key >> 8);
}

// ---------------------------------------------------------------- transmission by setting and age
// The place of a child's infection is not stored anywhere, but it is a pure function of what is: every draw is keyed on
// (replica seed in force that day, agent, day, purpose | slot), and the child's record holds its infector and
// inf_key = day << 8 | slot of the contact slot that won.  The seed comes from the seed history seed_of_day[R][max_days + 1]
// (branch.cuh), not from RepCtr::seed: rb_branch gives a replica a new seed, and a child infected before that was drawn
// with the old one.  Recomputing that slot's 24-bit uniform and picking the row against the contact table of that day's
// epoch gives the row k_expose picked, hence the place.  The row is found by an upper-bound binary search
// over cum24 (non-decreasing, so the search returns the linear scan's first row with k24 < cum24[row]), independent of
// the 4096-cell guide k_expose decodes.
//
// Row of one replica (int32, rb_transmission_settings_len entries), M = max_days + 1, P = RB_N_PLACES, G = n_groups:
//   by_day_place[M][P + 1]   infected agents by infection day and place of infection (column P = RB_PLACE_ROOT:
//                            imports and the initial state)
//   pair_all[P][G][G]        children by place, infector's age group, child's age group
//   pair_closed[P][G][G]     the same, counting only children of closed infectors (neither INCUBATION nor ILLNESS)
//   closed_by_group[G]       closed cases by age group
struct SxLayout {
    int M, n_groups;
    int by_day, pair_all, pair_closed, closed, len;
};
__host__ __device__ inline SxLayout sx_layout(int max_days, int n_groups) {
    SxLayout L;
    L.M = max_days + 1; L.n_groups = n_groups;
    const int pgg = RB_N_PLACES * n_groups * n_groups;
    L.by_day = 0; L.pair_all = L.M * (RB_N_PLACES + 1);
    L.pair_closed = L.pair_all + pgg; L.closed = L.pair_closed + pgg;
    L.len = L.closed + n_groups;
    return L;
}

// Place (0 .. RB_N_PLACES - 1) of the contact in slot `slot` that `infector` (of age `iage`) made on `day` under table tb.
__device__ __forceinline__ int contact_place(const DevTable *tb, uint32_t seed, int32_t infector, int iage, uint32_t day, uint32_t slot) {
    const u32x4 x = philox(seed, (uint32_t)infector, day, PU_CONTACT | ((slot >> 2) << 8), 0);
    const uint32_t q = slot & 3u;
    const uint32_t k24 = (q == 0 ? x.x : q == 1 ? x.y : q == 2 ? x.z : x.w) >> 8;
    const uint32_t *cum24 = tb->cum24[iage];
    const int n = __ldg(&tb->n_rows[iage]);
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (k24 < __ldg(&cum24[mid])) hi = mid; else lo = mid + 1;
    }
    return (int)__ldg(&tb->place[iage][max(min(lo, n - 1), 0)]);     // last row on overrun, as k_expose
}

// The infection place of an agent that has left SUSCEPTIBLE: RB_PLACE_ROOT for a root.
__device__ __forceinline__ int infection_place(const Eng &G, int r, const AgentRec &rec, const int32_t *epoch_of_day, const uint32_t *seed_of_day) {
    if (rec.infector < 0) return RB_PLACE_ROOT;
    const uint32_t d = rec.inf_key >> 8;
    return contact_place(G.tables[__ldg(&epoch_of_day[d])], seed_of_day[(size_t)r * (G.max_days + 1) + d], rec.infector, age_of(G, rec.infector), d, rec.inf_key & 255u);
}

// Same skeleton as k_transmission: blockIdx.y = replica, grid-stride over the agents, the never infected skipped through
// the susceptibility bitmap, counts in shared memory added to out[replica] with integer atomics (geometry-independent).
// Per child one gathered packed word of the infector (its state) and one Philox block; the contact tables are read
// through L1 / L2.
__global__ void __launch_bounds__(TX_THREADS) k_transmission_settings(Eng G, SxLayout L, const int32_t *epoch_of_day, const uint32_t *seed_of_day, int32_t *out) {
    extern __shared__ int32_t s_sx[];
    const int r = blockIdx.y;
    const size_t base = (size_t)r * G.Npad;
    const uint32_t *sus = G.sus + (size_t)r * G.sus_words;
    const int NG = L.n_groups;
    for (int i = threadIdx.x; i < L.len; i += blockDim.x) s_sx[i] = 0;
    __syncthreads();
    const int stride = gridDim.x * blockDim.x;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < G.N; a += stride) {
        if ((__ldg(&sus[a >> 5]) >> (a & 31)) & 1u) continue;
        const uint32_t st = H_STATE(G.hot[base + a]);
        if (st == RB_SUSCEPTIBLE) continue;
        const AgentRec &rec = G.rec[base + a];
        const int32_t inf = rec.infector;
        const uint32_t key = rec.inf_key;
        const int d = (int)(key >> 8);
        const int cg = __ldg(&G.group_of_age[age_of(G, a)]);
        int place = RB_PLACE_ROOT;
        if (inf >= 0) {
            const uint32_t ist = H_STATE(G.hot[base + inf]);
            const int iage = age_of(G, inf);
            place = contact_place(G.tables[__ldg(&epoch_of_day[d])], seed_of_day[(size_t)r * (G.max_days + 1) + d], inf, iage, (uint32_t)d, key & 255u);
            const int cell = (place * NG + __ldg(&G.group_of_age[iage])) * NG + cg;
            atomicAdd(&s_sx[L.pair_all + cell], 1);
            if (ist != RB_INCUBATION && ist != RB_ILLNESS) atomicAdd(&s_sx[L.pair_closed + cell], 1);
        }
        if (d < L.M) atomicAdd(&s_sx[L.by_day + d * (RB_N_PLACES + 1) + place], 1);
        if (st != RB_INCUBATION && st != RB_ILLNESS) atomicAdd(&s_sx[L.closed + cg], 1);
    }
    __syncthreads();
    int32_t *row = out + (size_t)r * L.len;
    for (int i = threadIdx.x; i < L.len; i += blockDim.x)
        if (s_sx[i]) atomicAdd(&row[i], s_sx[i]);
}

// Infection place of every agent of one replica (rb_read_infection_places): -1 never infected, 0 .. RB_N_PLACES - 1 the
// place of the contact, RB_PLACE_ROOT an import or the initial state.
__global__ void k_infection_places(Eng G, int r, const int32_t *epoch_of_day, const uint32_t *seed_of_day, int32_t *out) {
    const size_t base = (size_t)r * G.Npad;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < G.N; a += gridDim.x * blockDim.x)
        out[a] = H_STATE(G.hot[base + a]) == RB_SUSCEPTIBLE ? -1 : infection_place(G, r, G.rec[base + a], epoch_of_day, seed_of_day);
}

#endif
