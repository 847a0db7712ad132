/* CPU restatement of the DYNAMIC policy of SPEC §4.6 — TEST INFRASTRUCTURE.
 *
 * The rate rule (§4.2) while the buffer is low, BOLA (§4.3) once it is high, with the per-session mode that carries the
 * hysteresis from one decision to the next.  Both halves are tests/policy_oracle.c's, included here, so that the two
 * oracles cannot drift apart.  Built by tests/dynamic_oracle.py with gcc -O2 -ffp-contract=off -fno-fast-math (no FMA
 * contraction), like the environment oracle.
 */
#include "policy_oracle.c"

/* 0 when the thresholds are what abr_env_set_dynamic_params accepts, 1 otherwise */
int dyn_params_invalid(double switch_on_buffer, double switch_off_buffer) {
    if (!isfinite(switch_on_buffer) || !isfinite(switch_off_buffer)) return 1;
    if (!(switch_off_buffer >= 0.0) || !(switch_off_buffer < switch_on_buffer)) return 1;
    return 0;
}

/* The DYNAMIC action of N sessions; mode[N] (0 = rate rule, 1 = BOLA) is read and written in place.  bw_hist: the
 * per-session rings [N][K]; done nullable (a done session answers 0 and keeps its mode). */
void dyn_decide(const double* sizes, int V, int A, int default_quality, double chunk_length, double rb_safety,
                double bola_min_buffer, double bola_target_buffer, double switch_on_buffer, double switch_off_buffer,
                int N, const int32_t* chunk, const double* buffer, const uint8_t* done, const double* bw_hist,
                const int32_t* hist_len, int K, uint8_t* mode, int32_t* action) {
    double* v = (double*)malloc(sizeof(double) * (size_t)V * A);
    double vmax = pol_bola_table(sizes, V, A, v);
    double gp = vmax / (bola_target_buffer / bola_min_buffer - 1.0);
    double Vp = bola_min_buffer / gp;
    for (int s = 0; s < N; ++s) {
        if (done && done[s]) { action[s] = 0; continue; }
        int prev = chunk[s] == 0 ? 0 : mode[s];                 /* every episode starts on the rate rule */
        double threshold = prev ? switch_off_buffer : switch_on_buffer;
        int m = buffer[s] > threshold ? 1 : 0;
        mode[s] = (uint8_t)m;
        const double* row = sizes + (size_t)chunk[s] * A;
        action[s] = m ? bola_rule(row, v + (size_t)chunk[s] * A, A, Vp, gp, vmax, buffer[s])
                      : rb_rule(row, A, default_quality, chunk_length, rb_safety, bw_hist + (size_t)s * K, hist_len[s], K);
    }
    free(v);
}
