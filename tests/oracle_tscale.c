/*
 * oracle_tscale.c -- CPU reference of the per-replica transmission scale (reina_b200.h rb_set_transmission_scale /
 * rb_read_transmission_scale).  TEST INFRASTRUCTURE ONLY: tests/test_transmission_scale.py compiles it, with the probes of
 * tests/test_transmission_settings.py and its own, into a library of its own in a temporary directory.
 *
 * The probes add `float tscale_m1` (f - 1, zero from init_replica's memset) to the copy's Replica and multiply p_upper
 * and did_infect's p by 1 + tscale_m1 right after the oracle computes them -- the CUDA engine's products, in the same
 * order.  ro_branch copies the Replica whole and oracle_migrate.c serialises it raw, so branches, records and copies carry
 * the scale with no code here.
 */
#include "oracle_migrate.c"

int ro_set_transmission_scale(rb_engine *e, const float *scale) {
    for (int r = 0; r < e->cfg.n_replicas; r++)
        if (!(scale[r] > 0.0f && scale[r] <= 16.0f)) {
            snprintf(g_err, sizeof g_err, "ro_set_transmission_scale: scale[%d] = %g is not in (0, 16]", r, (double)scale[r]);
            return 1;
        }
    for (int r = 0; r < e->cfg.n_replicas; r++) e->rep[r].tscale_m1 = scale[r] - 1.0f;
    return 0;
}

int ro_read_transmission_scale(rb_engine *e, float *out) {
    for (int r = 0; r < e->cfg.n_replicas; r++) out[r] = 1.0f + e->rep[r].tscale_m1;
    return 0;
}
