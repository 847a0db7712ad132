/* CPU restatement of MPC over caller-supplied predictions (SPEC §5.6) — TEST INFRASTRUCTURE.
 *
 * Scalar C, every operation in the order SPEC §5.2 writes it; built by tests/mpc_pred_oracle.py with
 * gcc -O2 -ffp-contract=off -fno-fast-math (no FMA contraction), like the environment oracle.  The kernels must agree
 * with it bit for bit; tests/mpc_pred_oracle.py also holds a pure-Python restatement that it is checked against.
 */
#include <math.h>
#include <stdint.h>

#define MAXH 8
#define MAXA 16

static double max0(double x) { return x > 0.0 ? x : 0.0; } /* Python max(0, x) */

/* -J of SPEC §5.2 for the sequence R over h steps of per-step tables [h][A] (the oracle's rollout_j, clamped) */
static double rollout_j(const double* U, const double* RB, const double* DL, int A, int h, const int* R, int prev_q,
                        double buffer, double L, double B, double vw, double rw) {
    double vq = 0.0, qv = 0.0, rt = 0.0, b = buffer;
    int ap = prev_q;
    for (int i = 0; i < h; ++i) {
        int a = R[i];
        vq = vq + U[i * A + a];
        if (ap >= 0) qv = qv + fabs(U[i * A + a] - U[i * A + ap]);
        double d = RB[i * A + a] - b;
        rt = rt + max0(d);
        if (i != h - 1) {
            double t = max0(b - DL[i * A + a]);
            double w = max0((t + L) - B);
            b = max0((t + L) - w);
        }
        ap = a;
    }
    return -((vq - vw * qv) - rw * rt);
}

/* SPEC §5.6 for N sessions: pred [N][H] row-major, done nullable.  action [N], best_j [N] and best_seq [N][H]
 * (nullable) as abr_env_mpc_decide_pred writes them.  Returns the number of sessions with an input error. */
int orc_mpc_decide_pred(const double* sizes, const double* util, int V, int A, double L, double B, double vw,
                        double rw, int N, const int32_t* chunk, const int32_t* prev_q, const double* buffer,
                        const uint8_t* done, const double* pred, int H, int32_t* action, double* best_j,
                        int32_t* best_seq) {
    double U[MAXH * MAXA], RB[MAXH * MAXA], DL[MAXH * MAXA];
    int errors = 0;
    for (int s = 0; s < N; ++s) {
        const int k = chunk[s], q = prev_q[s];
        action[s] = 0;
        if (best_j) best_j[s] = NAN;
        if (best_seq) for (int i = 0; i < H; ++i) best_seq[(long)s * H + i] = -1;
        if (done && done[s]) continue;
        if (k < 0 || q >= A || H < 1 || H > MAXH || A > MAXA) { action[s] = -1; ++errors; continue; }
        const int h = H < V - k ? H : V - k;
        if (h <= 0) continue;
        int bad = 0;
        for (int i = 0; i < h; ++i) {
            const double p = pred[(long)s * H + i];
            if (!(p > 0.0) || isinf(p)) bad = 1;
        }
        if (bad) { action[s] = -1; ++errors; continue; }
        for (int i = 0; i < h; ++i)
            for (int a = 0; a < A; ++a) {
                RB[i * A + a] = DL[i * A + a] = sizes[(k + i) * A + a] / pred[(long)s * H + i];
                U[i * A + a] = util[(k + i) * A + a];
            }
        int R[MAXH] = {0}, best[MAXH] = {0}, have = 0;
        double bj = 0.0;
        for (;;) {
            const double j = rollout_j(U, RB, DL, A, h, R, q, buffer[s], L, B, vw, rw);
            if (!have || j < bj) {                                       /* first minimum, C order */
                have = 1; bj = j;
                for (int i = 0; i < h; ++i) best[i] = R[i];
            }
            int d = h - 1;
            while (d >= 0 && ++R[d] == A) { R[d] = 0; --d; }
            if (d < 0) break;
        }
        action[s] = best[0];
        if (best_j) best_j[s] = bj;
        if (best_seq) for (int i = 0; i < h; ++i) best_seq[(long)s * H + i] = best[i];
    }
    return errors;
}
