// reina_b200 / csrc / contacts.cuh
// k_expose (contact sampling + transmission) and k_resolve (first infector wins; person_infect).
#ifndef REINA_B200_CONTACTS_CUH
#define REINA_B200_CONTACTS_CUH
#include "state.cuh"

// ---------------------------------------------------------------- k_expose
// Contacts.  One thread per group of four contact slots of one infector (they share one Philox block):
// get_one_contact (main.pyx:1290-1304) picks the row, daily_contacts[place] is counted, and a coarse 8-bit filter
// (thinning, see the oracle) decides whether the contact can transmit at all.  The few survivors go through a
// warp-private shared-memory ring and are finished on dense warps: get_person_from_age_range (:1525-1535),
// person_expose / did_infect (:238-244, 908-934), atomicMin on the target's conflict slot.
#ifndef EX_THREADS
#define EX_THREADS 128
#endif
#ifndef EX_CTAS_PER_SM
#define EX_CTAS_PER_SM 24        // CTAs per SM the grid is sized for: two waves of the 12 resident ones.  A replica's CTAs share its
                                 // work items by grid stride, so a finer grid evens out the tail: measured on the peak day 8 / 10 /
                                 // 12 / 16 / 24 per SM: 553 / 519 / 588 (1.04 waves: the worst case) / 504 / 482 us
#endif
#define EX_RESIDENT_PER_SM 12    // 42 registers
#define EX_WARPS (EX_THREADS / 32)
#define EX_RCAP 256

__device__ __forceinline__ void expose_survivors(const Eng &G, int r, RepCtr *c, RepCtr *cd, const DevTable *tb, const uint2 *items, const uint32_t *sus,
                                                 Attempt *succ, uint32_t cap_succ, const uint32_t *ri, const uint32_t *rx, uint32_t head, uint32_t m, int lane) {
    const size_t base = (size_t)r * G.Npad;
    bool ok = false;
    uint32_t a = 0, t = 0, slot = 0;
    if ((uint32_t)lane < m) {
        const uint2 it = items[ri[(head + lane) & (EX_RCAP - 1)]];
        const uint32_t info = rx[(head + lane) & (EX_RCAP - 1)];
        const uint32_t row = (info >> 7) & 127u, kq = info >> 14;
        slot = info & 127u;
        a = it.x;
        const uint32_t age = (it.y >> 7) & 127u, dayidx = (it.y >> 14) & 31u, var = (it.y >> 20) & 3u;
        const rb_variant *v = &G.variants[var];
        float si = v->iot[dayidx];
        if ((it.y >> 19) & 1u) si = si * v->p_asymptomatic_infection;
        const u32x4 y = philox(c->seed, a, (uint32_t)c->day, PU_CONTACT2 | (slot << 8), 0);
        t = (uint32_t)tb->start[age][row] + y.x % (uint32_t)tb->size[age][row];
        // person_expose (main.pyx:238-244): only a SUSCEPTIBLE target can be infected; the 1-bit-per-agent map keeps
        // this random gather inside L2 instead of pulling a 32-byte DRAM sector per contact
        if ((__ldg(&sus[t >> 5]) >> (t & 31)) & 1u) {
            const int tage = tb->susc_uniform[age][row] ? (int)tb->lo_age[age][row]
                                                        : age_in_band(G, (int32_t)t, tb->lo_age[age][row], tb->hi_age[age][row]);
            const float pr = ((si * v->tab[RB_T_SUSCEPTIBILITY][tage]) * v->infectiousness_multiplier) * (1.0f + c->tscale_m1);
            if (((double)y.y * (1.0 / 4294967296.0)) * (double)kq < (double)pr * 256.0) {
                ok = true;
                const float mp = tb->mask_p[age][row];
                if (mp != 0.0f) {
                    const float ma = mp * v->p_mask_protects_others, mb = mp * v->p_mask_protects_wearer;
                    const float pm = (ma + mb) - ma * mb;
                    if (chance((double)y.z * (1.0 / 4294967296.0), pm)) ok = false;
                }
            }
        }
    }
    const uint32_t okm = __ballot_sync(0xffffffffu, ok);
    if (!okm) return;
    uint32_t b = 0;
    if (lane == 0) b = atomicAdd(&cd->n_succ, (uint32_t)__popc(okm));     // one atomic per warp batch
    b = __shfl_sync(0xffffffffu, b, 0);
    if (!ok) return;
    const uint32_t idx = b + __popc(okm & ((1u << lane) - 1u));
    const unsigned long long key = ((unsigned long long)sweep_pos(G, r, c, a) << 7) | slot;
    if (idx < cap_succ) {
        succ[idx].cand = t; succ[idx].parent = a; succ[idx].key = key;
        if (!G.xbuf) atomicMin(&G.rec[base + t].winner, key);     // sharded: k_merge does it over every rank's list
    } else set_problem(cd, RB_OTHER_FAILURE);
}

// The contacts of replica r as seen by ONE CTA: CTA `cta` of the `ncta` that share the replica's work items by grid
// stride.  s_place: RB_N_PLACES counters of the CTA; ri / rx: this warp's survivor ring.  Called by every thread of the CTA.
__device__ __forceinline__ void expose_cta(const Eng &G, const int r, const uint32_t cta, const uint32_t ncta, int *s_place, uint32_t *ri, uint32_t *rx) {
    RepCtr *c = &G.ctr[r];
    const DevTable *tb = G.tables[c->epoch];
    const uint32_t n = min(c->n_items, G.cap_items);
    if (cta * blockDim.x >= n) return;              // CTA-uniform: nothing for this CTA today
    if (threadIdx.x < RB_N_PLACES) s_place[threadIdx.x] = 0;
    __syncthreads();
    const uint2 *items = G.items + (size_t)r * G.cap_items;
    Attempt *succ = G.succ + (size_t)r * G.cap_succ;
    uint32_t cap_succ = G.cap_succ;
    RepCtr *cd = c;
    if (G.xbuf) { const XSlot x = xslot_of(G, G.rank, c->day); succ = x.succ; cap_succ = G.xcap_succ; cd = x.hdr; }
    const uint32_t *sus = G.sus + (size_t)r * G.sus_words;
    const uint32_t day = (uint32_t)c->day;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t head = 0, tail = 0;
    uint32_t places = 0;                 // this thread's per-place counters, 5 bits each, flushed every 7 iterations
    int since_flush = 0;
    const uint32_t stride = ncta * blockDim.x;
    uint2 nxt = make_uint2(0u, 0u);
    if (cta * blockDim.x + warp * 32 + lane < n) nxt = __ldcs(&items[cta * blockDim.x + warp * 32 + lane]);
    for (uint32_t i0 = cta * blockDim.x + warp * 32; i0 < n; i0 += stride) {
        const uint32_t i = i0 + lane;
        const bool valid = i < n;
        const uint2 it = nxt;
        if (i + stride < n) nxt = __ldcs(&items[i + stride]);       // the next step's work item: in flight while this one is processed
        uint32_t words[4] = {0, 0, 0, 0}, ncnt = 0, age = 0, grp = 0;
        int kq = 0;
        if (valid) {
            grp = it.y & 31u; ncnt = ((it.y >> 5) & 3u) + 1u; age = (it.y >> 7) & 127u;
            const rb_variant *v = &G.variants[(it.y >> 20) & 3u];
            float si = v->iot[(it.y >> 14) & 31u];
            if ((it.y >> 19) & 1u) si = si * v->p_asymptomatic_infection;
            // the replica's transmission scale f (RepCtr::tscale_m1) multiplies p and p_upper alike: float products are
            // monotone, so pr <= p_upper still holds, and with kq = 256 a pr >= 1 always passes, which is min(1, f p)
            const float p_upper = ((si * v->reserved[0]) * v->infectiousness_multiplier) * (1.0f + c->tscale_m1);
            kq = (int)(p_upper * 256.0f) + 1;
            if (kq > 256) kq = 256;
            const u32x4 x = philox(c->seed, it.x, day, PU_CONTACT | (grp << 8), 0);
            words[0] = x.x; words[1] = x.y; words[2] = x.z; words[3] = x.w;
        }
        const int nrows = tb->n_rows[age];
        const uint32_t *cum24 = tb->cum24[age];
        const uint32_t *guide = tb->guide[age];
        // get_one_contact (main.pyx:1290-1304): u = (word >> 8) / 2^24, the row is the first one with u < cum_p (an integer
        // compare against ceil(cum_p 2^24)).  ONE guide entry, fetched from u's top bits, answers for its whole cell unless
        // the cell holds several row boundaries (see DevTable::guide); the four gathers of a thread are issued together.
        uint32_t gd[4];
#pragma unroll
        for (uint32_t w = 0; w < 4; w++) gd[w] = w < ncnt ? __ldg(&guide[words[w] >> (32 - GUIDE_BITS)]) : 0u;
#pragma unroll
        for (uint32_t w = 0; w < 4; w++) {
            bool pass = false;
            uint32_t row = 0;
            if (w < ncnt) {
                const uint32_t word = words[w];
                const uint32_t k24 = word >> 8, g = gd[w], delta = (g >> 10) & 15u;
                row = g & 127u;
                uint32_t place = (g >> 7) & 7u;
                if (delta) {
                    if (delta < 15u) {
                        if ((k24 & ((1u << (24 - GUIDE_BITS)) - 1u)) >= (g >> 17)) { row += delta; place = (g >> 14) & 7u; }
                    } else {
                        while ((int)row < nrows - 1 && !(k24 < __ldg(&cum24[row]))) row++;   // last row on overrun: the reference fails there (p ~ 1e-15)
                        place = tb->place[age][row];
                    }
                }
                places += 1u << (5 * place);                              // daily_contacts[place]++ (main.pyx:1571)
                pass = (int)(word & 255u) < kq;
            }
            const unsigned m = __ballot_sync(0xffffffffu, pass);
            if (pass) {
                const uint32_t p = (tail + __popc(m & ((1u << lane) - 1u))) & (EX_RCAP - 1);
                ri[p] = i; rx[p] = (grp * 4u + w) | (row << 7) | ((uint32_t)kq << 14);
            }
            tail += __popc(m);
        }
        __syncwarp();
        while (tail - head >= 32) { expose_survivors(G, r, c, cd, tb, items, sus, succ, cap_succ, ri, rx, head, 32, lane); head += 32; }
        __syncwarp();
        if (++since_flush == 7) {        // 7 iterations x 4 contacts = 28 < 32 fits the 5-bit fields
#pragma unroll
            for (int pl = 0; pl < RB_N_PLACES; pl++) { const uint32_t k = (places >> (5 * pl)) & 31u; if (k) atomicAdd(&s_place[pl], (int)k); }
            places = 0; since_flush = 0;
        }
    }
    if (tail != head) expose_survivors(G, r, c, cd, tb, items, sus, succ, cap_succ, ri, rx, head, tail - head, lane);
#pragma unroll
    for (int pl = 0; pl < RB_N_PLACES; pl++) { const uint32_t k = (places >> (5 * pl)) & 31u; if (k) atomicAdd(&s_place[pl], (int)k); }
    __syncthreads();
    if (threadIdx.x < RB_N_PLACES && s_place[threadIdx.x]) atomicAdd(&cd->daily_contacts[threadIdx.x], s_place[threadIdx.x]);
}
__global__ void __launch_bounds__(EX_THREADS, EX_RESIDENT_PER_SM) k_expose(Eng G) {
    __shared__ int s_place[RB_N_PLACES];
    __shared__ uint32_t s_ri[EX_WARPS][EX_RCAP], s_rx[EX_WARPS][EX_RCAP];
    const int warp = threadIdx.x >> 5;
    expose_cta(G, blockIdx.y + G.r0, blockIdx.x, gridDim.x, s_place, s_ri[warp], s_rx[warp]);
}

// ---------------------------------------------------------------- k_resolve
// DRAIN: this day is followed by the fused day boundary, so tomorrow's test queue -- complete once today's sweep is
// over -- is drained here by the whole grid instead of by tomorrow's single boundary CTA (HealthcareSystem.iterate,
// main.pyx:514-545: every queued agent is detected).  The per-age detection counts are parked in drain_det and booked
// by the boundary at the point where the reference drains, so every stats row is unchanged.
// Thread `tid` of the `nth` that share replica r's list of successful transmissions.
template <bool DRAIN>
__device__ __forceinline__ void resolve_part(const Eng &G, const int r, const uint32_t tid, const uint32_t nth) {
    RepCtr *c = &G.ctr[r];
    const size_t base = (size_t)r * G.Npad;
    const uint32_t n = min(c->n_succ, G.cap_succ);
    const Attempt *succ = G.succ + (size_t)r * G.cap_succ;
    // two attempts per thread and pass: their gathers (conflict slot of the target, packed word of the infector) are in
    // flight together.  Two attempts on one target cannot both hold the winning key, so their order does not matter.
    const uint32_t stride = nth;
    const int list = (int)(c->lsel ^ 1u);      // infected during today's sweep: first visited tomorrow, so the entry goes to the lists today's sweep has written
    const bool has_list = c->testing_mode == RB_ALL_WITH_SYMPTOMS_CT;
    for (uint32_t i = tid; i < n; i += 2 * stride) {
        const uint32_t j = i + stride;
        const bool two = j < n;
        const Attempt a0 = succ[i];
        Attempt a1 = a0;
        if (two) a1 = succ[j];
        const unsigned long long w0 = G.rec[base + a0.cand].winner;
        const uint32_t h0 = G.hot[base + a0.parent];
        unsigned long long w1 = KEY_IDLE; uint32_t h1 = 0;
        if (two) { w1 = G.rec[base + a1.cand].winner; h1 = G.hot[base + a1.parent]; }
#pragma unroll 1
        for (int k = 0; k < 2; k++) {
            const Attempt at = k ? a1 : a0;
            if ((k && !two) || (k ? w1 : w0) != at.key) continue;      // first infector in sweep order wins
            device_infect(G, r, c, (int32_t)at.cand, (int32_t)at.parent, k ? h1 : h0, 0, (int)(at.key & 127ull), false, list, has_list);
            G.rec[base + at.cand].winner = KEY_IDLE;
        }
    }
    // verdict for the day boundary that follows: enough capacity events or queued tests to be worth a team of CTAs
    if (tid == 0)
        c->wide_day = (c->n_events >= (uint32_t)G.wide_min || c->n_newq >= (uint32_t)G.wide_min) ? 1u : 0u;
    if (DRAIN) {
        const uint32_t nq = min(c->n_newq, G.cap_queue);
        const int32_t *qa = G.q_agent + ((size_t)r * 2 + (c->qsel ^ 1u)) * G.cap_queue;
        for (uint32_t i = tid; i < nq; i += nth) {
            const int32_t a = qa[i];
            const uint32_t h = G.hot[base + a];
            if (h & H_DET) set_problem(c, RB_WRONG_STATE);   // person_detect, main.pyx:294-298
            G.hot[base + a] = (h & ~H_QUEUED) | H_DET;
            mark_detected(G, r, a);
            atomicAdd(&c->drain_det[age_of(G, a)], 1);
        }
        if (tid == 0) c->drained = 1u;
    }
}
template <bool DRAIN>
__global__ void __launch_bounds__(256, 4) k_resolve(Eng G) {
    resolve_part<DRAIN>(G, blockIdx.y + G.r0, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

#endif
