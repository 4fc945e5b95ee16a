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

#endif
