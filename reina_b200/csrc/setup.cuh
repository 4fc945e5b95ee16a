// reina_b200 / csrc / setup.cuh
// One-time and auxiliary kernels: Population.set_initial_state, state initialisation, stats snapshot, ensemble moments, samplers.
#ifndef REINA_B200_SETUP_CUH
#define REINA_B200_SETUP_CUH
#include "state.cuh"

// ---------------------------------------------------------------- initial population condition
// Population.set_initial_state, main.pyx:1452-1516 (Context.__init__ :1780-1781: day 0, testing still NO_TESTING).
// One-time, order-dependent setup of a few thousand people drawn WITH replacement: lane 0 of one CTA per replica replays
// the reference's loop literally (see apply_initial_state in the oracle for the quirks that are kept).
struct Ipc { int32_t dead, in_icu, in_ward, confirmed, incubating, ill, recovered; };

__device__ void init_remove(const Eng &G, RepCtr *c, size_t base, int32_t a, int age, bool dies) {   // person_recover / person_die
    uint32_t h = G.hot[base + a];
    count_add(c, RB_A_INFECTED, age, -1);
    if (dies) { count_add(c, RB_A_DEAD, age, 1); if (H_SEV(h) == RB_FATAL) count_add(c, RB_A_NON_HOSPITAL_DEATHS, age, 1); }
    else count_add(c, RB_A_RECOVERED, age, 1);
    G.hot[base + a] = H_SET_STATE(h, dies ? RB_DEAD : RB_RECOVERED) & ~(H_LIST | H_FRESH);
}
__device__ bool init_dies_without_care(const Eng &G, RepCtr *c, int32_t a, uint32_t h) {   // dies_in_hospital(care_available=False)
    const uint32_t sev = H_SEV(h);
    if (sev == RB_FATAL) return true;
    const rb_variant *v = &G.variants[H_VAR(h)];
    const float ch = sev == RB_CRITICAL ? v->p_icu_death_no_beds : (sev == RB_SEVERE ? v->p_hospital_death_no_beds : 0.0f);
    u32x4 x = philox(c->seed, (uint32_t)a, (uint32_t)c->day, PU_NOBED, 0);
    return chance(u01d(x.x, x.y), ch);
}
__device__ void init_hospitalize(const Eng &G, RepCtr *c, size_t base, int32_t a, int age) {   // person_hospitalize, main.pyx:321-338
    uint32_t h = G.hot[base + a];
    if (!(h & H_DET)) { h |= H_DET; count_add(c, RB_A_DETECTED, age, 1); count_add(c, RB_A_ALL_DETECTED, age, 1); G.hot[base + a] = h; }
    if (c->avail_beds == 0) { init_remove(G, c, base, a, age, init_dies_without_care(G, c, a, h)); return; }
    c->avail_beds -= 1;
    G.hot[base + a] = H_SET_DL(H_SET_STATE(h, RB_HOSPITALIZED), (G.rec[base + a].cold >> 16) & 255u) & ~H_FRESH;
    count_add(c, RB_A_IN_WARD, age, 1);
}
__device__ void init_to_icu(const Eng &G, RepCtr *c, size_t base, int32_t a, int age) {   // person_transfer_to_icu, main.pyx:341-351
    uint32_t h = G.hot[base + a];
    c->avail_beds += 1;
    if (c->avail_icu == 0) {
        if (init_dies_without_care(G, c, a, h)) { count_add(c, RB_A_IN_WARD, age, -1); init_remove(G, c, base, a, age, true); return; }
    } else c->avail_icu -= 1;
    G.hot[base + a] = H_SET_DL(H_SET_STATE(h, RB_IN_ICU), (G.rec[base + a].cold >> 24) & 255u) & ~H_FRESH;
    count_add(c, RB_A_IN_WARD, age, -1); count_add(c, RB_A_IN_ICU, age, 1); count_add(c, RB_A_CUM_ICU, age, 1);
}
__device__ void init_become_ill(const Eng &G, RepCtr *c, size_t base, int32_t a) {   // person_become_ill, main.pyx:284-291 (nobody seeks testing yet)
    uint32_t h = G.hot[base + a];
    const uint32_t sev = H_SEV(h);
    const rb_variant *v = &G.variants[H_VAR(h)];
    const int day = c->day;
    float T = (sev == RB_FATAL)
        ? gamma_f(c->seed, (uint32_t)a, (uint32_t)day, PU_ONSET, v->onset_death_kappa, v->onset_death_theta)
        : gamma_f(c->seed, (uint32_t)a, (uint32_t)day, PU_ONSET, v->onset_recovery_kappa, v->onset_recovery_theta);
    float f = T;
    if (sev != RB_ASYMPTOMATIC && sev != RB_MILD) f = f * v->ratio_before_hospitalisation;
    const uint32_t dl = (uint32_t)clamp255(round_to_int(f));
    float w = 0.0f, u = 0.0f;
    if (sev == RB_SEVERE) w = T * (1.0f - v->ratio_before_hospitalisation);
    else if (sev == RB_CRITICAL || sev == RB_FATAL) {
        w = T * v->ratio_in_ward;
        u = ((1.0f - v->ratio_in_ward) - v->ratio_before_hospitalisation) * T;
    }
    const uint32_t wd = (uint32_t)clamp255(round_to_int(w)), ud = (uint32_t)clamp255(round_to_int(u));
    G.rec[base + a].cold = (G.rec[base + a].cold & 0xffffu) | (wd << 16) | (ud << 24);     // assigned, not OR-ed: the person may have been drawn before
    G.hot[base + a] = H_SET_DL(H_SET_STATE(h, RB_ILLNESS), dl) & ~H_FRESH;
}

__global__ void k_initial_state(Eng G, Ipc P) {
    if (threadIdx.x != 0) return;
    const int r = blockIdx.x;
    RepCtr *c = &G.ctr[r];
    const size_t base = (size_t)r * G.Npad;
    const int32_t were_ill = P.dead + P.recovered + P.in_icu + P.in_ward + P.ill, were_incubating = were_ill + P.incubating;
    const int32_t i_incubating = P.incubating, i_rws = i_incubating + (were_incubating - were_ill);
    const int32_t i_ill_at_home = i_rws + P.ill, i_dead = i_ill_at_home + P.dead, i_in_icu = i_dead + P.in_icu, i_in_ward = i_in_icu + P.in_ward;
    for (int32_t i = 0; i < were_incubating; i++) {
        u32x4 x = philox(c->seed, (uint32_t)i, 0u, PU_INIT, 0);
        const int32_t a = (int32_t)(x.x % (uint32_t)G.N);           // get_random_person, main.pyx:1518-1523
        const int age = age_of(G, a);
        // a person drawn before is infected again, exactly as the reference does; person_infect (main.pyx:209-235) resets
        // state, severity and the day counter but leaves was_detected alone
        const uint32_t was_detected = G.hot[base + a] & H_DET;
        device_infect(G, r, c, a, -1, 0u, 0, 0, true, -1, false);     // no list entry: a person drawn twice must not be listed twice, k_rebuild_lists follows
        if (was_detected) G.hot[base + a] |= H_DET;
        if (i < i_incubating) continue;                              // still incubating: waits one day like any same-day infection
        if (i < i_rws) { init_remove(G, c, base, a, age, false); continue; }
        init_become_ill(G, c, base, a);
        if (i < i_ill_at_home) continue;
        if (i < i_dead) { init_remove(G, c, base, a, age, true); continue; }
        if (i < i_in_icu) { init_hospitalize(G, c, base, a, age); init_to_icu(G, c, base, a, age); continue; }
        if (i < i_in_ward) { init_hospitalize(G, c, base, a, age); continue; }
        init_remove(G, c, base, a, age, false);
    }
    for (int age = 0; age < 100 && age < G.n_ages; age++) c->counts[RB_A_ALL_DETECTED][age] = 0;
    for (int32_t i = 0; i < P.confirmed; i++) c->counts[RB_A_ALL_DETECTED][(100 + i) % 100] += 1;
}

// ---------------------------------------------------------------- row guide of a contact table
// DevTable::guide from cum24 / place, one CTA per age.  rowfn(k) = first row r < nrows - 1 with k < cum24[r], else nrows - 1.
__device__ __forceinline__ int guide_rowfn(const uint32_t *cum, int nrows, uint32_t k) {
    int lo = 0, hi = nrows - 1;                       // cum24 is non-decreasing: binary search for the first row with k < cum[r]
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (k < cum[mid]) hi = mid; else lo = mid + 1; }
    return lo;
}
__global__ void k_build_guide(DevTable *tb, int n_ages) {
    const int age = blockIdx.x;
    if (age >= n_ages) return;
    const int nrows = tb->n_rows[age];
    if (nrows <= 0) return;
    const uint32_t *cum = tb->cum24[age];
    const int shift = 24 - GUIDE_BITS;
    for (uint32_t cell = threadIdx.x; cell < (1u << GUIDE_BITS); cell += blockDim.x) {
        const uint32_t lo = cell << shift, hi = lo + (1u << shift) - 1u;
        const int r0 = guide_rowfn(cum, nrows, lo), r1 = guide_rowfn(cum, nrows, hi);
        uint32_t delta = 0, blow = 0, place1 = 0;
        if (r1 != r0) {
            // lo < cum[r0] <= hi: the first boundary inside the cell.  One boundary only <=> its own value already maps to r1.
            if (guide_rowfn(cum, nrows, cum[r0]) == r1 && r1 - r0 <= 14) { delta = (uint32_t)(r1 - r0); blow = cum[r0] - lo; place1 = tb->place[age][r1]; }
            else delta = 15;
        }
        tb->guide[age][cell] = (uint32_t)r0 | ((uint32_t)tb->place[age][r0] << 7) | (delta << 10) | (place1 << 14) | (blow << 17);
    }
}

// ---------------------------------------------------------------- misc kernels
// The per-replica counters of a fresh Context (Context.__init__, main.pyx:1759-1781): everything zero, every age
// susceptible, full capacity, the replica's seed and the keys of its sweep-order permutation.  One CTA per replica.
__global__ void k_init_counters(Eng G, uint32_t seed, int32_t beds, int32_t icu) {
    RepCtr *c = &G.ctr[blockIdx.x];
    uint32_t *w = reinterpret_cast<uint32_t *>(c);
    for (uint32_t i = threadIdx.x; i < (uint32_t)(sizeof(RepCtr) / 4); i += blockDim.x) w[i] = 0u;
    __syncthreads();
    for (int age = threadIdx.x; age < G.n_ages; age += blockDim.x) c->counts[RB_A_SUSCEPTIBLE][age] = G.age_start[age + 1] - G.age_start[age];
    if (threadIdx.x == 0) {
        c->beds = c->avail_beds = beds; c->icu = c->avail_icu = icu;
        c->p_successful_tracing = 1.0f;
        c->seed = seed + blockIdx.x;
        const u32x4 k = philox(c->seed, 0, 0, PU_PERM, 0);
        c->fkey[0] = k.x; c->fkey[1] = k.y; c->fkey[2] = k.z; c->fkey[3] = k.w;
        for (int i = 0; i < RB_MAX_VACC; i++) c->vacc_cursor[i] = -2;
    }
}

// Every agent SUSCEPTIBLE and untouched.  SPARSE (rb_reset): the arrays hold the end of a previous run, in which an agent
// was only ever written if it stopped being susceptible or its packed word became non-zero (vaccinated, queued,
// detected) -- conflict slots are always handed back idle -- so only those agents are rewritten: the reset reads 4 bytes
// per agent and writes 36 for the ~20 % a HUS run has touched, instead of writing 36 for everybody.
template <bool SPARSE>
__global__ void k_init(Eng G) {
    const int r = blockIdx.y;
    const size_t base = (size_t)r * G.Npad;
    const uint32_t *sus = G.sus + (size_t)r * G.sus_words;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < G.Npad; i += gridDim.x * blockDim.x) {
        // padding words beyond N are marked RECOVERED+included (nobody ever lists them)
        const uint32_t fresh = i < G.N ? 0u : (RB_RECOVERED | H_INCL);
        if (SPARSE && i < G.N && G.hot[base + i] == 0u && ((sus[i >> 5] >> (i & 31)) & 1u)) continue;
        G.hot[base + i] = fresh;
        AgentRec z; z.winner = KEY_IDLE; z.infector = -1; z.first_child = -1; z.next_sib = -1; z.inf_key = 0; z.cold = 0; z.vacc_day = -1; z.pad = 0;
        G.rec[base + i] = z;
    }
}
// the two bitmaps of a fresh population; after k_init<true>, which still reads the old susceptibility bits
__global__ void k_init_bitmaps(Eng G) {
    const int r = blockIdx.y;
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < G.sus_words; w += gridDim.x * blockDim.x) {
        int first = w * 32;
        uint32_t m = first + 32 <= G.N ? 0xffffffffu : (first >= G.N ? 0u : ((1u << (G.N - first)) - 1u));
        G.sus[(size_t)r * G.sus_words + w] = m;
        G.det[(size_t)r * G.sus_words + w] = 0u;
    }
}

__global__ void k_snapshot(Eng G) {
    __shared__ int32_t srow[RB_N_ATTRS * 16 + RB_N_SCALARS];
    write_stats_row(G, blockIdx.x, &G.ctr[blockIdx.x], srow);
}

// Per-day metric aggregation across the ensemble: sum and sum of squares over replicas of every stats column.
__global__ void k_moments(Eng G, int day0, double *out_sum, double *out_sq) {
    const int d = blockIdx.x;
    for (int col = threadIdx.x; col < G.row_len; col += blockDim.x) {
        double s1 = 0.0, s2 = 0.0;
        for (int r = 0; r < G.R; r++) {
            const double v = (double)G.stats[((size_t)r * (G.max_days + 1) + day0 + d) * G.row_len + col];
            s1 += v; s2 += v * v;
        }
        out_sum[(size_t)d * G.row_len + col] = s1; out_sq[(size_t)d * G.row_len + col] = s2;
    }
}

// Context.sample, main.pyx:2047-2101
// keyed on the engine's seed, not on replica 0's counters: rb_branch may re-seed replica 0
__global__ void k_sample(Eng G, uint32_t seed, int what, int age, int severity, int n, int epoch, int32_t *out) {
    const rb_variant *v = &G.variants[0];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t pu = PU_SAMPLE | ((uint32_t)what << 8);
        int res;
        if (what == 0) {
            u32x4 x = philox(seed, (uint32_t)i, (uint32_t)age, pu, 0);
            double u = u01d(x.x, x.y);
            const double *cdf = G.tables[epoch]->ncdf[age][0];
            int lo = 0, hi = 100;
            while (lo < hi) { int mid = (lo + hi) >> 1; if (u < cdf[mid]) hi = mid; else lo = mid + 1; }
            res = lo;
        } else if (what == 1) {
            u32x4 x = philox(seed, (uint32_t)i, (uint32_t)age, pu, 0);
            res = symptom_severity(v, age, u01f(x.x), false, 0.0f, 0.0f, 0.0f);      // no replica: unscaled
        } else if (what == 2) {
            res = round_to_int(gamma_f(seed, (uint32_t)i, (uint32_t)age, pu, v->incubation_kappa, v->incubation_theta));
        } else {
            float T = severity == RB_FATAL ? gamma_f(seed, (uint32_t)i, (uint32_t)age, pu, v->onset_death_kappa, v->onset_death_theta)
                                           : gamma_f(seed, (uint32_t)i, (uint32_t)age, pu, v->onset_recovery_kappa, v->onset_recovery_theta);
            float f = 0.0f;
            if (what == 3) { f = T; if (severity != RB_ASYMPTOMATIC && severity != RB_MILD) f = f * v->ratio_before_hospitalisation; }
            else if (what == 4) { if (severity == RB_SEVERE) f = T * (1.0f - v->ratio_before_hospitalisation); else if (severity >= RB_CRITICAL) f = T * v->ratio_in_ward; }
            else if (what == 5) { if (severity >= RB_CRITICAL) f = ((1.0f - v->ratio_in_ward) - v->ratio_before_hospitalisation) * T; }
            else f = T;
            res = round_to_int(f);
        }
        out[i] = res;
    }
}

#endif
