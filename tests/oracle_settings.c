/*
 * oracle_settings.c -- CPU reference of the transmission tables by setting and age (reina_b200.h
 * rb_transmission_settings_len / rb_transmission_settings / rb_read_infection_places).  TEST INFRASTRUCTURE ONLY:
 * tests/test_transmission_settings.py compiles it into a library of its own in a temporary directory.
 *
 * The place of an infection is what the oracle observed where it infected: the test build adds one write-only field to
 * the oracle's Agent, `infection_place`, set to RB_PLACE_ROOT by person_infect and to the place of the contact row
 * (found by the oracle's own linear scan over cum_p) right after person_expose_others' person_infect call.  Nothing the
 * oracle computes or reports changes.  The CUDA engine instead recomputes the place afterwards from the infection tree,
 * so the two derivations share no code.  The entry points below are plain loops over the Agent records; the epochs
 * passed in are checked against the schedule the oracle ran.
 */
#include "oracle_transmission.c"

int32_t ro_transmission_settings_len(rb_engine *e) {
    const int32_t G = e->cfg.n_groups;
    return (e->cfg.max_days + 1) * (RB_N_PLACES + 1) + 2 * RB_N_PLACES * G * G + G;
}

static int check_epochs(rb_engine *e, const int32_t *epoch_of_day, int32_t n_days) {
    if (n_days != e->day) { snprintf(g_err, sizeof g_err, "transmission settings: %d epochs given, %d days completed", n_days, e->day); return 1; }
    for (int d = 0; d < n_days; d++)
        if (epoch_of_day[d] != e->sched[d].table_epoch) {
            snprintf(g_err, sizeof g_err, "transmission settings: day %d ran epoch %d, %d given", d, e->sched[d].table_epoch, epoch_of_day[d]);
            return 1;
        }
    return 0;
}

static int is_closed(const Agent *p) { return p->state != RB_INCUBATION && p->state != RB_ILLNESS; }

int ro_transmission_settings(rb_engine *e, const int32_t *epoch_of_day, int32_t n_days, int32_t *out) {
    if (check_epochs(e, epoch_of_day, n_days)) return 1;
    const int32_t M = e->cfg.max_days + 1, G = e->cfg.n_groups, P = RB_N_PLACES, len = ro_transmission_settings_len(e);
    for (int ri = 0; ri < e->cfg.n_replicas; ri++) {
        const Replica *r = &e->rep[ri];
        int32_t *row = out + (size_t)ri * len;
        int32_t *by_day = row, *pair_all = row + M * (P + 1), *pair_closed = pair_all + P * G * G, *closed = pair_closed + P * G * G;
        memset(row, 0, sizeof(int32_t) * (size_t)len);
        for (int32_t a = 0; a < e->cfg.n_agents; a++) {
            const Agent *p = &r->agents[a];
            if (p->state == RB_SUSCEPTIBLE) continue;
            const int d = p->day_of_infection, pl = p->infection_place, cg = e->group_of_age[p->age];
            if (d < M) by_day[d * (P + 1) + pl] += 1;
            if (p->infector >= 0) {
                const Agent *q = &r->agents[p->infector];
                const int cell = (pl * G + e->group_of_age[q->age]) * G + cg;
                pair_all[cell] += 1;
                if (is_closed(q)) pair_closed[cell] += 1;
            }
            if (is_closed(p)) closed[cg] += 1;
        }
    }
    return 0;
}

int ro_read_infection_places(rb_engine *e, int32_t replica, const int32_t *epoch_of_day, int32_t n_days, int32_t *out) {
    if (check_epochs(e, epoch_of_day, n_days)) return 1;
    const Replica *r = &e->rep[replica];
    for (int32_t a = 0; a < e->cfg.n_agents; a++)
        out[a] = r->agents[a].state == RB_SUSCEPTIBLE ? -1 : r->agents[a].infection_place;
    return 0;
}
