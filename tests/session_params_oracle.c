/* CPU restatement of per-session policy parameters (SPEC §4.7) — TEST INFRASTRUCTURE.
 *
 * The decisions of BBA, RATE, BOLA (SPEC §4, §4.2, §4.3) and DYNAMIC (§4.6) with every session's own knobs: the rules
 * are tests/policy_oracle.c's (included through tests/dynamic_oracle.c, unchanged), called once per session with that
 * session's values, and BOLA's (Vp, gp) are derived per session exactly as pol_decide derives the environment-wide
 * pair.  Built by tests/session_params_oracle.py with gcc -O2 -ffp-contract=off -fno-fast-math (no FMA contraction).
 */
#include "dynamic_oracle.c"

/* The first field of session s that fails the environment-wide setters' checks, in the order bba_reservoir,
 * bba_cushion, rb_safety, bola_min_buffer, bola_target_buffer, switch_on_buffer, switch_off_buffer (0..6); -1 if
 * none.  x: [7][N] field-major. */
int sp_first_invalid(const double* x, int N, int s) {
    double r = x[0 * N + s], c = x[1 * N + s], rb = x[2 * N + s], mn = x[3 * N + s], tg = x[4 * N + s];
    double on = x[5 * N + s], off = x[6 * N + s];
    if (!isfinite(r)) return 0;
    if (!isfinite(c) || !(c > 0.0)) return 1;
    if (!isfinite(rb) || !(rb > 0.0)) return 2;
    if (!isfinite(mn) || !(mn > 0.0)) return 3;
    if (!isfinite(tg) || !(mn < tg)) return 4;
    if (!isfinite(on)) return 5;
    if (!isfinite(off) || !(off >= 0.0) || !(off < on)) return 6;
    return -1;
}

/* BOLA's (Vp, gp) of session parameters (min, target) for the table maximum vmax: install_policy_params' operations */
void sp_bola_derive(double vmax, double mn, double tg, double* Vp, double* gp) {
    *gp = vmax / (tg / mn - 1.0);
    *Vp = mn / *gp;
}

/* The action of `policy` (BBA, RATE, BOLA or DYNAMIC) for N sessions, session s with knobs x[f * N + s] (field order
 * as sp_first_invalid).  mode[N]: DYNAMIC's per-session rule, read and written; done nullable. */
void sp_decide(const double* sizes, int V, int A, int default_quality, double chunk_length, const double* x, int N,
               int policy, const int32_t* chunk, const double* buffer, const uint8_t* done, const double* bw_hist,
               const int32_t* hist_len, int K, uint8_t* mode, int32_t* action) {
    double* v = (double*)malloc(sizeof(double) * (size_t)V * A);
    double vmax = pol_bola_table(sizes, V, A, v);
    for (int s = 0; s < N; ++s) {
        double rb = x[2 * N + s], Vp, gp;
        sp_bola_derive(vmax, x[3 * N + s], x[4 * N + s], &Vp, &gp);
        if (policy == POL_BBA) { action[s] = bba_rule(x[0 * N + s], x[1 * N + s], A, buffer[s]); continue; }
        if (done && done[s]) { action[s] = 0; continue; }
        const double* row = sizes + (size_t)chunk[s] * A;
        const double* vrow = v + (size_t)chunk[s] * A;
        const double* ring = bw_hist + (size_t)s * K;
        int use_bola = policy == POL_BOLA;
        if (policy == 5) {   /* ABR_POLICY_DYNAMIC */
            int prev = chunk[s] == 0 ? 0 : mode[s];
            use_bola = buffer[s] > (prev ? x[6 * N + s] : x[5 * N + s]) ? 1 : 0;
            mode[s] = (uint8_t)use_bola;
        }
        action[s] = use_bola ? bola_rule(row, vrow, A, Vp, gp, vmax, buffer[s])
                             : rb_rule(row, A, default_quality, chunk_length, rb, ring, hist_len[s], K);
    }
    free(v);
}
