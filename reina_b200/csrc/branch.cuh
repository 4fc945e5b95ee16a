// reina_b200 / csrc / branch.cuh
// Branching replicas (rb_branch): replica j continues from the current state of replica src[j] with a seed of its own.
// Two keys make this exact without touching any per-day kernel: RepCtr::seed keys every draw, RepCtr::fkey keys the
// replica's fixed sweep-order permutation.  The copy takes the source's fkey along with its state, so every sweep position
// already stored (test queue, capacity events, perm) stays valid, and the new seed changes only the draws of the days to
// come.  The state copied is what rb_save_state saves (state_parts in engine.cu); the active lists and perm are rebuilt
// from the copied packed words, as rb_load_state does.  Precondition (checked by the host): src[src[j]] == src[j], so no
// replica is both read and written.
//
// The seed history seed_of_day[R][max_days + 1] (the seed of every replica on every day) is a kernel argument, not a
// member of Eng: a larger Eng would move the parameters k_run takes after it, and the per-day kernels stay as built.
#ifndef REINA_B200_BRANCH_CUH
#define REINA_B200_BRANCH_CUH

#include "state.cuh"

// 16-byte loads and stores where both ends and the length allow it (every section but the stats rows), else 4-byte words.
__device__ __forceinline__ void branch_copy_bytes(void *dst, const void *src, size_t bytes, size_t tid, size_t nt) {
    if ((((uintptr_t)dst | (uintptr_t)src | bytes) & 15u) == 0) {
        uint4 *d = (uint4 *)dst; const uint4 *s = (const uint4 *)src;
        for (size_t i = tid; i < bytes / 16; i += nt) d[i] = s[i];
    } else {
        uint32_t *d = (uint32_t *)dst; const uint32_t *s = (const uint32_t *)src;
        for (size_t i = tid; i < bytes / 4; i += nt) d[i] = s[i];
    }
}

// blockIdx.y = destination replica j, grid-stride over its sections.  A replica with src[j] == j keeps its state and
// only takes the new seed.  Block 0 of a column copies the counters (with the new seed in place of the source's) and
// writes the seed history: the source's seeds before `today`, the new seed from today on.  The destination's list
// counters are zeroed for k_branch_rebuild.
__global__ void k_branch_copy(Eng G, uint32_t *seed_of_day, const int32_t *src, const uint32_t *seed, int today) {
    const int j = blockIdx.y, s = src[j];
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    const size_t M = (size_t)G.max_days + 1;
    if (s != j) {
        const size_t N = G.Npad, W = G.sus_words, Q = 2 * (size_t)G.cap_queue, S = M * G.row_len;
        branch_copy_bytes(G.hot + j * N, G.hot + s * N, N * sizeof(uint32_t), tid, nt);
        branch_copy_bytes(G.rec + j * N, G.rec + s * N, N * sizeof(AgentRec), tid, nt);
        branch_copy_bytes(G.sus + j * W, G.sus + s * W, W * sizeof(uint32_t), tid, nt);
        branch_copy_bytes(G.det + j * W, G.det + s * W, W * sizeof(uint32_t), tid, nt);
        branch_copy_bytes(G.q_key + j * Q, G.q_key + s * Q, Q * sizeof(unsigned long long), tid, nt);
        branch_copy_bytes(G.q_agent + j * Q, G.q_agent + s * Q, Q * sizeof(int32_t), tid, nt);
        branch_copy_bytes(G.stats + j * S, G.stats + s * S, S * sizeof(int32_t), tid, nt);
        for (size_t i = tid; i < 2 * (size_t)G.n_seg; i += nt) G.seg_n[2 * (size_t)G.n_seg * j + i] = make_uint2(0u, 0u);
    }
    if (blockIdx.x != 0) return;
    const uint32_t *cs = reinterpret_cast<const uint32_t *>(&G.ctr[s]);
    uint32_t *cd = reinterpret_cast<uint32_t *>(&G.ctr[j]);
    const uint32_t seed_word = (uint32_t)(offsetof(RepCtr, seed) / 4);
    if (s != j)
        for (uint32_t w = threadIdx.x; w < (uint32_t)(sizeof(RepCtr) / 4); w += blockDim.x) cd[w] = w == seed_word ? seed[j] : cs[w];
    else if (threadIdx.x == 0) cd[seed_word] = seed[j];
    const uint32_t *hs = seed_of_day + (size_t)s * M;
    uint32_t *hd = seed_of_day + (size_t)j * M;
    for (size_t d = threadIdx.x; d < M; d += blockDim.x)
        if ((int)d >= today) hd[d] = seed[j]; else if (s != j) hd[d] = hs[d];
}

// The active list `lsel` of every destination replica from its copied packed words (k_rebuild_lists for the replicas
// that were written), and perm -- the sweep slot under the copied fkey -- for every agent that has left SUSCEPTIBLE,
// i.e. the source's perm of every agent whose slot can still be read.
__global__ void k_branch_rebuild(Eng G, const int32_t *src) {
    const int r = blockIdx.y;
    if (src[r] == r) return;
    RepCtr *c = &G.ctr[r];
    const size_t base = (size_t)r * G.Npad;
    const uint32_t cur = c->lsel;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < G.N; a += gridDim.x * blockDim.x) {
        uint32_t h = G.hot[base + a];
        const uint32_t st = H_STATE(h);
        if (st == RB_SUSCEPTIBLE) continue;
        G.perm[base + a] = sweep_slot(G, c, (uint32_t)a);
        if (!((st >= RB_INCUBATION && st <= RB_IN_ICU) || (st >= RB_RECOVERED && !(h & H_INCL)))) continue;
        if (h & H_QUEUED) h |= H_DET;
        list_add(G, r, c, cur, (uint32_t)a, h);
    }
}

// Seed history of a fresh population (rb_create, rb_reset: seed + r on every day) or of a version-2 checkpoint (the
// loaded counters' seed on every day): from_ctr selects the latter.
__global__ void k_init_seeds(Eng G, uint32_t *seed_of_day, uint32_t seed, int from_ctr) {
    const int r = blockIdx.x;
    const uint32_t v = from_ctr ? G.ctr[r].seed : seed + (uint32_t)r;
    for (int d = threadIdx.x; d <= G.max_days; d += blockDim.x) seed_of_day[(size_t)r * (G.max_days + 1) + d] = v;
}

#endif
