/* CPU restatement of the RATE and BOLA policies of SPEC §4.2 / §4.3 (and BBA, §4) — TEST INFRASTRUCTURE.
 *
 * Scalar C, every operation in the order SPEC writes it; built by tests/policy_oracle.py with
 * gcc -O2 -ffp-contract=off -fno-fast-math (no FMA contraction), like the environment oracle.  The kernels must agree
 * with it bit for bit; tests/policy_oracle.py also holds a pure-Python restatement that it is checked against.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

enum { POL_BBA = 2, POL_RATE = 3, POL_BOLA = 4 };

/* 0 when the parameters are what abr_env_set_policy_params accepts, 1 otherwise */
int pol_params_invalid(double rb_safety, double bola_min_buffer, double bola_target_buffer) {
    if (!(rb_safety > 0.0) || !isfinite(rb_safety)) return 1;
    if (!(bola_min_buffer > 0.0) || !isfinite(bola_min_buffer) || !isfinite(bola_target_buffer) ||
        !(bola_min_buffer < bola_target_buffer))
        return 1;
    return 0;
}

/* v[k][a] = log(sizes[k][a] / sizes[k][0]); returns v_max */
double pol_bola_table(const double* sizes, int V, int A, double* v) {
    double vmax = -INFINITY;
    for (int k = 0; k < V; ++k)
        for (int a = 0; a < A; ++a) {
            double x = log(sizes[k * A + a] / sizes[k * A]);
            v[k * A + a] = x;
            if (x > vmax) vmax = x;
        }
    return vmax;
}

/* rate-based: ring = the session's K slots, newest at (len - 1) mod K; row = sizes of the current chunk */
static int rb_rule(const double* row, int A, int default_quality, double L, double rb_safety, const double* ring,
                   int len, int K) {
    int n = len < K ? len : K;
    if (n == 0) {
        int d = default_quality < 0 ? 0 : default_quality;
        return d > A - 1 ? A - 1 : d;
    }
    double S = 0.0;
    for (int j = 0; j < n; ++j) S = S + 1.0 / ring[(len - n + j) % K];   /* oldest first */
    double hm = (double)n / S;
    double budget = (rb_safety * hm) * L;
    int q = 0;
    for (int a = 0; a < A; ++a)
        if (row[a] <= budget) q = a;
    return q;
}

static int bola_rule(const double* row, const double* vrow, int A, double Vp, double gp, double vmax, double b) {
    if (vmax <= 0.0) return 0;
    int q = 0;
    double best = 0.0;
    for (int a = 0; a < A; ++a) {
        double sc = (Vp * (vrow[a] + gp) - b) / row[a];
        if (a == 0 || sc > best) { best = sc; q = a; }
    }
    return q;
}

static int bba_rule(double reservoir, double cushion, int A, double b) {
    if (b < reservoir) return 0;
    if (b >= reservoir + cushion) return A - 1;
    int q = (int)floor(((double)(A - 1) * (b - reservoir)) / cushion);
    return q > A - 1 ? A - 1 : q;
}

/* The action of `policy` for N sessions.  bw_hist: per-session rings [N][K]; done nullable (a done session,
 * chunk == V, answers 0 under RATE and BOLA). */
void pol_decide(const double* sizes, int V, int A, int default_quality, double chunk_length, double bba_reservoir,
                double bba_cushion, double rb_safety, double bola_min_buffer, double bola_target_buffer, int N,
                int policy, const int32_t* chunk, const double* buffer, const uint8_t* done, const double* bw_hist,
                const int32_t* hist_len, int K, int32_t* action) {
    double* v = (double*)malloc(sizeof(double) * (size_t)V * A);
    double vmax = pol_bola_table(sizes, V, A, v);
    double gp = vmax / (bola_target_buffer / bola_min_buffer - 1.0);
    double Vp = bola_min_buffer / gp;
    for (int s = 0; s < N; ++s) {
        if (policy == POL_BBA) { action[s] = bba_rule(bba_reservoir, bba_cushion, A, buffer[s]); continue; }
        if (done && done[s]) { action[s] = 0; continue; }
        const double* row = sizes + (size_t)chunk[s] * A;
        action[s] = policy == POL_RATE
                        ? rb_rule(row, A, default_quality, chunk_length, rb_safety, bw_hist + (size_t)s * K,
                                  hist_len[s], K)
                        : bola_rule(row, v + (size_t)chunk[s] * A, A, Vp, gp, vmax, buffer[s]);
    }
    free(v);
}
