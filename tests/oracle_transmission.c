/*
 * oracle_transmission.c -- CPU reference of the transmission statistics (reina_b200.h rb_transmission_len /
 * rb_transmission_stats / rb_read_infection_days).  TEST INFRASTRUCTURE ONLY: tests/test_transmission.py compiles it
 * into a library of its own in a temporary directory.
 *
 * It includes the sequential oracle unchanged and adds the three entry points with the `ro_` prefix, as straight loops
 * over the oracle's Agent records (day_of_infection, n_infected, infector, state, variant, age): the resulting library is
 * the oracle plus these exports, bound through the same ctypes wrapper as the CUDA library.
 */
#include "../oracle/reina_oracle.c"

int32_t ro_transmission_len(rb_engine *e) {
    return 3 * (e->cfg.max_days + 1) + 2 * RB_TX_BINS + 2 * e->cfg.n_groups + 2 * RB_MAX_VARIANTS;
}

int ro_transmission_stats(rb_engine *e, int32_t *out) {
    const int32_t M = e->cfg.max_days + 1, G = e->cfg.n_groups, len = ro_transmission_len(e);
    for (int ri = 0; ri < e->cfg.n_replicas; ri++) {
        const Replica *r = &e->rep[ri];
        int32_t *row = out + (size_t)ri * len;
        int32_t *infected = row, *offspring = row + M, *open = row + 2 * M, *ohist = row + 3 * M, *gi = ohist + RB_TX_BINS;
        int32_t *gclosed = gi + RB_TX_BINS, *goff = gclosed + G, *vclosed = goff + G, *voff = vclosed + RB_MAX_VARIANTS;
        memset(row, 0, sizeof(int32_t) * (size_t)len);
        for (int32_t a = 0; a < e->cfg.n_agents; a++) {
            const Agent *p = &r->agents[a];
            if (p->state == RB_SUSCEPTIBLE) continue;
            const int d = p->day_of_infection, o = p->n_infected;
            if (d < M) { infected[d] += 1; offspring[d] += o; }
            if (p->infector >= 0) {
                int g = d - r->agents[p->infector].day_of_infection;
                gi[g < 0 ? 0 : (g > RB_TX_BINS - 1 ? RB_TX_BINS - 1 : g)] += 1;
            }
            if (p->state == RB_INCUBATION || p->state == RB_ILLNESS) {
                if (d < M) open[d] += 1;
            } else {
                ohist[o > RB_TX_BINS - 1 ? RB_TX_BINS - 1 : o] += 1;
                const int grp = e->group_of_age[p->age];
                gclosed[grp] += 1; goff[grp] += o;
                vclosed[p->variant] += 1; voff[p->variant] += o;
            }
        }
    }
    return 0;
}

int ro_read_infection_days(rb_engine *e, int32_t replica, int32_t *out) {
    const Replica *r = &e->rep[replica];
    for (int32_t a = 0; a < e->cfg.n_agents; a++)
        out[a] = r->agents[a].state == RB_SUSCEPTIBLE ? -1 : r->agents[a].day_of_infection;
    return 0;
}
