/*
 * oracle_sscale.c -- CPU reference of the per-replica severity scales (reina_b200.h rb_set_severity_scale /
 * rb_read_severity_scale).  TEST INFRASTRUCTURE ONLY: tests/test_severity_scale.py compiles it, with the probes of
 * tests/test_transmission_settings.py, tests/test_transmission_scale.py and its own, into a library of its own in a
 * temporary directory.
 *
 * The probes add `float sscale_m1[3]` (severe, critical, fatal minus 1, zero from init_replica's memset) to the copy's
 * Replica, point a file-scope pointer at the infected agent's replica's scales right before person_infect draws the
 * severity (and clear it right after, so the sampler's draws stay unscaled), and apply the CUDA engine's four clamped
 * products where symptom_severity reads dohc and sc / cc / fc.  ro_branch copies the Replica whole and oracle_migrate.c
 * serialises it raw, so branches, records and copies carry the scales with no code here.
 */
#include "oracle_tscale.c"

int ro_set_severity_scale(rb_engine *e, const float *scale) {
    for (int i = 0; i < 3 * e->cfg.n_replicas; i++)
        if (!(scale[i] > 0.0f && scale[i] <= 16.0f)) {
            snprintf(g_err, sizeof g_err, "ro_set_severity_scale: scale[%d][%d] = %g is not in (0, 16]", i / 3, i % 3, (double)scale[i]);
            return 1;
        }
    for (int r = 0; r < e->cfg.n_replicas; r++)
        for (int j = 0; j < 3; j++) e->rep[r].sscale_m1[j] = scale[3 * r + j] - 1.0f;
    return 0;
}

int ro_read_severity_scale(rb_engine *e, float *out) {
    for (int r = 0; r < e->cfg.n_replicas; r++)
        for (int j = 0; j < 3; j++) out[3 * r + j] = 1.0f + e->rep[r].sscale_m1[j];
    return 0;
}
