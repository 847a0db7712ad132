/* CPU restatement of MPC over caller-supplied throughput scenarios (SPEC §5.7) — TEST INFRASTRUCTURE.
 *
 * Scalar C, every operation in the order SPEC §5.7 writes it; built by tests/mpc_scen_oracle.py with
 * gcc -O2 -ffp-contract=off -fno-fast-math (no FMA contraction).  The kernels must agree with it bit for bit;
 * tests/mpc_scen_oracle.py also holds a pure-Python restatement that it is checked against.
 */
#include <math.h>
#include <stdint.h>

#define MAXH 8
#define MAXA 16
#define MAXK 16

static double max0(double x) { return x > 0.0 ? x : 0.0; } /* Python max(0, x) */

/* q_k = (vq - vw qv) - rw rt_k of SPEC §5.2 for the sequence R over h steps, scenario table RB [h][A] */
static double rollout_q(const double* U, const double* RB, int A, int h, const int* R, int prev_q, double buffer,
                        double L, double B, double vw, double rw) {
    double vq = 0.0, qv = 0.0, rt = 0.0, b = buffer;
    int ap = prev_q;
    for (int i = 0; i < h; ++i) {
        int a = R[i];
        vq = vq + U[i * A + a];
        if (ap >= 0) qv = qv + fabs(U[i * A + a] - U[i * A + ap]);
        rt = rt + max0(RB[i * A + a] - b);
        if (i != h - 1) {
            double t = max0(b - RB[i * A + a]);
            double w = max0((t + L) - B);
            b = max0((t + L) - w);
        }
        ap = a;
    }
    return (vq - vw * qv) - rw * rt;
}

/* SPEC §5.7 for N sessions: pred [N][K][H] row-major, weight [N][K] (nullable), objective 0 mean / 1 worst, done
 * nullable.  action [N], best_j [N] and best_seq [N][H] as abr_env_mpc_decide_scen writes them.  Returns the number
 * of sessions with an input error. */
int orc_mpc_decide_scen(const double* sizes, const double* util, int V, int A, double L, double B, double vw,
                        double rw, int N, const int32_t* chunk, const int32_t* prev_q, const double* buffer,
                        const uint8_t* done, const double* pred, const double* weight, int K, int H, int objective,
                        int32_t* action, double* best_j, int32_t* best_seq) {
    static double U[MAXH * MAXA], RB[MAXK][MAXH * MAXA];
    double w[MAXK];
    int errors = 0;
    for (int s = 0; s < N; ++s) {
        const int k = chunk[s], q = prev_q[s];
        action[s] = 0;
        best_j[s] = NAN;
        for (int i = 0; i < H; ++i) best_seq[(long)s * H + i] = -1;
        if (done && done[s]) continue;
        if (k < 0 || q >= A || H < 1 || H > MAXH || A > MAXA || K < 1 || K > MAXK) { action[s] = -1; ++errors; continue; }
        const int h = H < V - k ? H : V - k;
        if (h <= 0) continue;
        int bad = 0;
        for (int c = 0; c < K; ++c)
            for (int i = 0; i < h; ++i) {
                const double p = pred[((long)s * K + c) * H + i];
                if (!(p > 0.0) || isinf(p)) bad = 1;
            }
        if (objective == 0) {
            int any = 0;
            for (int c = 0; c < K; ++c) {
                w[c] = weight ? weight[(long)s * K + c] : 1.0 / K;
                if (!(w[c] >= 0.0) || isinf(w[c])) bad = 1;
                if (w[c] != 0.0) any = 1;
            }
            if (!any) bad = 1;
        }
        if (bad) { action[s] = -1; ++errors; continue; }
        for (int i = 0; i < h; ++i)
            for (int a = 0; a < A; ++a) {
                U[i * A + a] = util[(k + i) * A + a];
                for (int c = 0; c < K; ++c) RB[c][i * A + a] = sizes[(k + i) * A + a] / pred[((long)s * K + c) * H + i];
            }
        /* the first maximum of Q in C order, a NaN Q never chosen; none above -inf: sequence 0, best_j = +inf */
        int R[MAXH] = {0}, best[MAXH] = {0};
        double bq = -INFINITY;
        for (;;) {
            double Q = 0.0;
            for (int c = 0; c < K; ++c) {
                const double qk = rollout_q(U, RB[c], A, h, R, q, buffer[s], L, B, vw, rw);
                if (objective == 0) Q = c == 0 ? w[0] * qk : Q + w[c] * qk;
                else if (c == 0 || qk < Q) Q = qk;
            }
            if (Q > bq) {                                                /* first minimum of J = -Q, C order */
                bq = Q;
                for (int i = 0; i < h; ++i) best[i] = R[i];
            }
            int d = h - 1;
            while (d >= 0 && ++R[d] == A) { R[d] = 0; --d; }
            if (d < 0) break;
        }
        action[s] = best[0];
        best_j[s] = -bq;
        for (int i = 0; i < h; ++i) best_seq[(long)s * H + i] = best[i];
    }
    return errors;
}
